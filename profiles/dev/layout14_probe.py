"""Development probe: the literal BASELINE config-3 agent layout (14 x 90 modes + tip-tilt) through the fused step."""
import sys, time
sys.path.insert(0, ".")
import numpy as np
import torch
from ao_marl_b200.system import build_system

E = int(sys.argv[1]) if len(sys.argv) > 1 else 1024
sim, t, rl = build_system("production_sh_40x40_8m_3layers.py", E,
                          env_rl=dict(n_zernike_start_end=[0, 1260], window_n_zernike=20, include_tip_tilt_windowed=True,
                                      n_reverse_filtered_from_cmat=5, delayed_assignment=2), world_size=16, seed=0)
print("agents", rl.n_agents, "actor_in", rl.actor_in, "actor_out", rl.actor_out, "state_dim", rl.state_dim)
sim.reset(1234 + np.arange(E, dtype=np.int64))
sim.state_begin(); sim.move_atmos(); sim.comp_wfs_image(); sim.do_centroids(); sim.do_control(); sim.state_end()
for _ in range(3):
    sim.step(mode=0)
torch.cuda.synchronize()
ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
ev[0].record()
for _ in range(5):
    sim.step(mode=0)
ev[1].record()
torch.cuda.synchronize()
ms = ev[0].elapsed_time(ev[1]) / 5
st = sim.rows("STATE", rl.state_dim)
act = sim.rows("ACTION", rl.action_dim)
rw = sim.buffer("REWARD").view(E, rl.n_agents)
assert torch.isfinite(st).all() and torch.isfinite(act).all() and torch.isfinite(rw).all()
assert float(act.abs().max()) <= 1.0 + 1e-6 and float(rw.max()) <= 0.0
sim.check_device()
print("E=%d: %.2f ms per step, %.0f env-steps/s" % (E, ms, E / ms * 1e3))
sim.close()
