"""Which sensor kernel serves a frame (aom_comp_wfs_image): every wfs path, in every per-environment state, for every
kind of frame, either runs or is refused with the message include/aomarl.h documents."""
import numpy as np
import pytest

PATHS = ("umma_ws", "umma", "umma_fast", "simt", "tensor", "tensor_fast", "tensor_reg")
ROUND1 = ("tensor", "tensor_fast", "tensor_reg")
KERNELS = {"umma_ws": "wfs_frame_ws_kernel", "umma": "wfs_frame_umma_kernel", "umma_fast": "wfs_frame_umma_kernel",
           "simt": "wfs_frame_kernel", "tensor": "wfs_frame_tma_kernel", "tensor_fast": "wfs_frame_tma_kernel",
           "tensor_reg": "wfs_frame_mma_kernel"}
FRAMES = {"noise-free": dict(noise=-1.0), "noisy": dict(noise=3.0), "kept image": dict(noise=-1.0, keep_image=True),
          "no atmosphere": dict(noise=-1.0, atmos=False)}
# state -> (message of the round-1 kernels' refusal, frames they refuse)
STATES = {"uniform": (None, ()),
          "per-environment wind": ("per-environment wind", ("noise-free", "noisy", "kept image")),
          "per-environment noise": ("per-environment sensor", ("noisy",)),
          "per-environment photon counts": ("per-environment sensor", tuple(FRAMES)),
          "staggered": ("staggered", tuple(FRAMES))}
SEEDS = np.array([11, 12, 13], dtype=np.int64)


def _enter(sim, state):
    sim.reset(SEEDS)
    if state == "per-environment wind":
        dx, dy = float(sim.cfg.deltax[0]), float(sim.cfg.deltay[0])
        sim.set_layer_wind(0, np.array([1.0, 0.5, -0.5], np.float32) * dx, np.array([1.0, -0.5, 0.5], np.float32) * dy)
        sim.move_atmos()
    elif state == "per-environment noise":
        sim.set_wfs_noise_env(noise=[3.0, 0.0, -1.0])
    elif state == "per-environment photon counts":
        sim.set_wfs_noise_env(nphotons=sim.wfs_nphotons * np.array([0.5, 1.0, 2.0], np.float32))
    elif state == "staggered":
        sim.move_atmos()
        sim.reset_envs([1], np.array([99], np.int64))


def _leave(sim, state):
    if state == "per-environment wind":
        sim.set_layer_wind(0, None, None)
    elif state.startswith("per-environment"):
        sim.set_wfs_noise_env(None, None)


@pytest.mark.gpu
def test_routing_matrix(static10):
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from ao_marl_b200.lib import Simulator
    sim = Simulator(static10, len(SEEDS), rl=None)
    try:
        for path in PATHS:
            sim.set_wfs_path(path)
            assert sim.wfs_kernel() == KERNELS[path], path
            for state, (message, refused) in STATES.items():
                _enter(sim, state)
                for frame, kw in FRAMES.items():
                    if path in ROUND1 and frame in refused:
                        with pytest.raises(RuntimeError, match=message):
                            sim.comp_wfs_image(**kw)
                    else:
                        sim.comp_wfs_image(**kw)
                        sim.check_device()
                _leave(sim, state)
    finally:
        sim.close()
