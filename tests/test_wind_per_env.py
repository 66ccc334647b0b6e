"""Per-environment wind (aom_set_layer_wind, AtmosB200.set_wind with [E] arrays): every environment of a batch with its
own wind computes exactly what it computes in a batch where every environment has that wind."""
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "..", "ao_marl_b200", "csrc")

# the directions of test_extrusion_directions, a step above one pixel per frame and no wind at all
WINDS10 = [(1.3, 0.0), (-1.3, 0.0), (0.0, 0.7), (0.0, -0.7), (0.8, 0.8), (-0.6, 0.45), (2.26, -1.7), (0.0, 0.0)]

SHIM = r"""
#include "wind_host.h"
extern "C" void wind_run(int E, int T, const float* dx, const float* dy, float xoff, float yoff,
                         int* n, double* acc, int* ij, float* w) {
  for (int e = 0; e < E; ++e) {
    double ax = 0.0, ay = 0.0;
    for (int t = 0; t < T; ++t) {
      const size_t i = (size_t)t * E + e;
      n[2 * i] = wind_advance(ax, dx[i]);
      n[2 * i + 1] = wind_advance(ay, dy[i]);
      acc[2 * i] = ax; acc[2 * i + 1] = ay;
      const WindRec r = wind_record(xoff, yoff, ax, ay);
      ij[2 * i] = r.ix; ij[2 * i + 1] = r.iy;
      w[6 * i] = r.fx; w[6 * i + 1] = r.fy;
      w[6 * i + 2] = r.w00; w[6 * i + 3] = r.w01; w[6 * i + 4] = r.w10; w[6 * i + 5] = r.w11;
    }
  }
}
"""


def test_wind_accumulator_matches_oracle(tmp_path):
    """The accumulator / offset header shared by the host mirror and wind_state_kernel, built by a host compiler: whole
    pixels and accumulators equal OracleAtmos.move exactly, offsets and weights equal fill_wfs_params' formula (the
    oracle's raytrace_layer)."""
    import ctypes
    from oracle import aoframe
    src = tmp_path / "wind_shim.cpp"
    src.write_text(SHIM)
    lib = tmp_path / "libwind_shim.so"
    subprocess.run(["g++", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-I", CSRC, "-o", str(lib), str(src)], check=True)
    L = ctypes.CDLL(str(lib))
    E, T = 6, 2000
    r = np.random.default_rng(11)
    dx = (r.standard_normal((T, E)) * 1.5).astype(np.float32)      # negative, above one pixel, both signs per env
    dy = (r.uniform(-2.5, 2.5, (T, E))).astype(np.float32)
    dx[:, 5] = 0.0
    xoff, yoff = np.float32(2.0), np.float32(1.75)
    n = np.zeros((T, E, 2), np.int32)
    acc = np.zeros((T, E, 2), np.float64)
    ij = np.zeros((T, E, 2), np.int32)
    w = np.zeros((T, E, 6), np.float32)
    P = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    L.wind_run.argtypes = [ctypes.c_int, ctypes.c_int] + [ctypes.c_void_p] * 2 + [ctypes.c_float] * 2 + [ctypes.c_void_p] * 4
    L.wind_run(E, T, P(dx), P(dy), float(xoff), float(yoff), P(n), P(acc), P(ij), P(w))
    F32 = np.float32
    for e in range(E):
        tab = {"nscreens": 1, "dim_screens": [8], "deltax": np.zeros(1, F32), "deltay": np.zeros(1, F32)}
        o = aoframe.OracleAtmos(tab, 0)
        moves = []
        o._one = lambda l, axis, sign: moves.append((axis, sign))     # the extrusions themselves are not at stake
        for t in range(T):
            tab["deltax"][0], tab["deltay"][0] = dx[t, e], dy[t, e]
            moves.clear()
            o.move()
            nx = sum(s for a, s in moves if a == 0)
            ny = sum(s for a, s in moves if a == 1)
            assert (n[t, e, 0], n[t, e, 1]) == (nx, ny), (t, e)
            assert acc[t, e, 0] == o.accx[0] and acc[t, e, 1] == o.accy[0], (t, e)
            px, py = float(xoff) + o.accx[0], float(yoff) + o.accy[0]
            ix, iy = int(np.floor(px)), int(np.floor(py))
            fx, fy = F32(px - ix), F32(py - iy)
            ref = [fx, fy, (F32(1) - fx) * (F32(1) - fy), fx * (F32(1) - fy), (F32(1) - fx) * fy, fx * fy]
            assert (ij[t, e, 0], ij[t, e, 1]) == (ix, iy), (t, e)
            assert np.array_equal(w[t, e], np.array(ref, F32)), (t, e)


# ------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _logical(sim, layer, env):
    n = int(sim.cfg.screen_dim[layer])
    scr = sim.buffer("SCREEN", layer).view(sim.n_env, n, n)[env]
    ox, oy = int(sim.buffer("RING_OX", layer)[env]), int(sim.buffer("RING_OY", layer)[env])
    return np.roll(scr.cpu().numpy(), (-oy, -ox), axis=(0, 1))


@pytest.mark.gpu
def test_screens_per_environment(static10, oracle_tab10, torch):
    """One layer, eight environments, eight winds (+x, -x, +y, -y, diagonal, mixed signs, > 1 px / frame, none):
    reset + 10 move_atmos.  Each logical screen == the same environment of a uniform batch with its wind (same seeds),
    and within 3e-5 of the oracle run with that wind."""
    from ao_marl_b200.lib import Simulator
    from oracle import aoframe
    E = len(WINDS10)
    dx = np.array([w[0] for w in WINDS10], np.float32)
    dy = np.array([w[1] for w in WINDS10], np.float32)
    seeds = np.arange(E, dtype=np.int64) * 7 + 300
    sim = Simulator(static10, E, rl=None)
    try:
        amp = float(sim.cfg.amp[0])
        sim.set_layer_wind(0, dx, dy)
        sim.reset(seeds)
        for _ in range(10):
            sim.move_atmos()
        got = [_logical(sim, 0, e) for e in range(E)]
        sim.check_device()
        sim.set_layer_wind(0, None, None)
        for e in range(E):
            sim.set_layer(0, float(dx[e]), float(dy[e]), amp)
            sim.reset(seeds)
            for _ in range(10):
                sim.move_atmos()
            assert np.array_equal(got[e], _logical(sim, 0, e)), WINDS10[e]
            tab = dict(oracle_tab10)
            tab["deltax"] = dx[e:e + 1].copy()
            tab["deltay"] = dy[e:e + 1].copy()
            o = aoframe.OracleAtmos(tab, int(seeds[e]))
            o.reset(int(seeds[e]))
            for _ in range(10):
                o.move()
            err = np.abs(got[e] - o.screens[0]).max() / np.abs(o.screens[0]).max()
            assert err < 3e-5, (WINDS10[e], err)
        sim.check_device()
    finally:
        sim.close()


def _sample_everything(sim, t, torch):
    """Every consumer of the screens, after one more frame of wind."""
    out = {}
    sim.move_atmos()
    for path, noise, keep in (("umma_ws", -1.0, False), ("umma", -1.0, False), ("umma", 3.0, True), ("simt", -1.0, False)):
        sim.set_wfs_path(path)
        sim.comp_wfs_image(noise=noise, keep_image=keep)
        sim.do_centroids()
        out["slopes_%s_%g" % (path, noise)] = sim.rows("SLOPES", t.nslopes).cpu().numpy().copy()
        if keep:
            out["image"] = sim.buffer("BINCUBE").cpu().numpy().copy()
    sim.set_wfs_path(sim.DEFAULT_WFS_PATH)
    out["phase"] = sim.raytrace_wfs().cpu().numpy().copy()
    sim.do_centroids_geom()
    out["slopes_geom"] = sim.rows("SLOPES", t.nslopes).cpu().numpy().copy()
    for pupil in ("sweep", "pixel"):
        sim.set_pupil_path(pupil)
        out["strehl_%s" % pupil] = sim.comp_strehl(1.65, accumulate=False).cpu().numpy().copy()
        out["strehl_peak_%s" % pupil] = sim.comp_strehl(1.65, accumulate=False, peak=True).cpu().numpy().copy()
        out["geo_com_%s" % pupil] = sim.do_control_geo().cpu().numpy().copy()
    sim.set_pupil_path("sweep")
    return out


@pytest.mark.gpu
def test_every_sampler_per_environment(torch):
    """production_sh_40x40_8m_3layers, three layers with a wind per environment each: sensor slopes of umma_ws, umma
    (noise-free, and with photon + read noise and a kept image), simt; the phase getter; geometric slopes; Strehl on
    axis and from the PSF core (sweep and pixel paths); geometric controller commands -- each environment equal to the
    uniform batch of its winds, over several frames."""
    from ao_marl_b200 import tables
    from ao_marl_b200.config import load_config_from_file
    from ao_marl_b200.init import geo
    from ao_marl_b200.lib import Simulator
    t = tables.build_static(load_config_from_file("production_sh_40x40_8m_3layers.py"))
    geo.build_geo(t)
    E, NL = 3, 3
    r = np.random.default_rng(5)
    speed = np.abs(np.asarray(t.config.p_atmos._deltax) + 1j * np.asarray(t.config.p_atmos._deltay))
    ang = r.uniform(0, 2 * np.pi, (NL, E))
    dx = (speed[:, None] * r.uniform(0.6, 1.4, (NL, E)) * np.cos(ang)).astype(np.float32)
    dy = (speed[:, None] * r.uniform(0.6, 1.4, (NL, E)) * np.sin(ang)).astype(np.float32)
    seeds = np.array([41, 42, 43], dtype=np.int64)
    sim = Simulator(t, E, rl=None)
    try:
        amps = [float(sim.cfg.amp[l]) for l in range(NL)]
        for l in range(NL):
            sim.set_layer_wind(l, dx[l], dy[l])
        sim.reset(seeds)
        frames = [_sample_everything(sim, t, torch) for _ in range(3)]
        sim.check_device()
        for f in frames:
            assert np.array_equal(f["slopes_umma_ws_-1"], f["slopes_umma_-1"])
            assert np.abs(f["slopes_simt_-1"]).max() > 1e-3
        for l in range(NL):
            sim.set_layer_wind(l, None, None)
        for e in range(E):
            for l in range(NL):
                sim.set_layer(l, float(dx[l, e]), float(dy[l, e]), amps[l])
            sim.reset(seeds)
            for i in range(3):
                ref = _sample_everything(sim, t, torch)
                for k, v in ref.items():
                    if k == "image":
                        nv = t.p_wfs._nvalid
                        a, b = frames[i][k].reshape(E, nv, 256)[e], v.reshape(E, nv, 256)[e]
                    else:
                        a, b = frames[i][k][e], v[e]
                    assert np.array_equal(a, b), (k, e, i)
        sim.check_device()
    finally:
        sim.close()


@pytest.mark.gpu
def test_closed_loop_through_set_wind(torch):
    """AoEnv (10x10, two agents): winds set per environment through env.supervisor.atmos.set_wind with [E] speeds and
    directions; over a few aom_step calls state, rewards and commands of each environment equal the uniform run."""
    from ao_marl_b200.env.ao_env import AoEnv
    from ao_marl_b200.env.config_rl import Config
    cfg = Config(parameters_telescope="production_sh_10x10_2m.py", n_zernike_start_end=[0, 80],
                 n_reverse_filtered_from_cmat=5, delayed_assignment=2)
    E = 4
    env = AoEnv(cfg, n_env=E, world_size=3, initial_seed=1234)
    sim, rl, atm = env.sim, env.supervisor.rl, env.supervisor.atmos
    ws, wd = np.array([20.0, 8.0, 35.0, 0.0]), np.array([45.0, 200.0, 300.0, 90.0])
    seeds = np.array([71, 72, 73, 74], dtype=np.int64)
    nactu = sim.cfg.nactu

    def run():
        sim.reset(seeds)
        out = []
        for _ in range(4):
            sim.step(mode=0)
            out.append((sim.rows("STATE", rl.state_dim).cpu().numpy().copy(),
                        sim.buffer("REWARD").view(E, rl.n_agents).cpu().numpy().copy(),
                        sim.rows("COM", nactu).cpu().numpy().copy()))
        return out

    try:
        atm.set_wind(0, windspeed=ws, winddir=wd)
        got = run()
        assert np.abs(got[-1][2]).max() > 0
        for e in range(E):
            atm.set_wind(0, windspeed=float(ws[e]), winddir=float(wd[e]))
            ref = run()
            for (a1, a2, a3), (b1, b2, b3) in zip(got, ref):
                assert np.array_equal(a1[e], b1[e]) and np.array_equal(a2[e], b2[e]) and np.array_equal(a3[e], b3[e]), e
        sim.check_device()
    finally:
        sim.close()


@pytest.mark.gpu
def test_handover(static10, torch):
    """Switching to per-environment winds mid-episode (everyone on the current common wind) == never switching, and
    back; a scalar set_wind + reset == a context that never had per-environment winds; set_r0(scalar) keeps them; a
    wrong length raises ValueError; the round-1 sensor kernel refuses to run with them."""
    from ao_marl_b200.lib import Simulator
    from ao_marl_b200.supervisor.components import AtmosB200
    E = 3
    seeds = np.array([5, 6, 7], dtype=np.int64)
    a, b = Simulator(static10, E, rl=None), Simulator(static10, E, rl=None)
    try:
        dx0, dy0 = float(a.cfg.deltax[0]), float(a.cfg.deltay[0])

        def frame(sim):
            sim.comp_wfs_image(noise=-1.0)
            sim.do_centroids()
            return _logical(sim, 0, 0), _logical(sim, 0, 2), sim.rows("SLOPES", static10.nslopes).cpu().numpy().copy()

        def same(x, y):
            return all(np.array_equal(u, v) for u, v in zip(x, y))

        a.reset(seeds); b.reset(seeds)
        for _ in range(3):
            a.move_atmos(); b.move_atmos()
        a.set_layer_wind(0, np.full(E, dx0, np.float32), np.full(E, dy0, np.float32))
        for _ in range(5):
            a.move_atmos(); b.move_atmos()
            assert same(frame(a), frame(b))
        a.set_layer_wind(0, None, None)
        for _ in range(3):
            a.move_atmos(); b.move_atmos()
            assert same(frame(a), frame(b))

        atm_a, atm_b = AtmosB200(a, static10.config), AtmosB200(b, static10.config)
        p = static10.config.p_atmos
        ws0, wd0 = float(p.windspeed[0]), float(p.winddir[0])
        with pytest.raises(ValueError):
            atm_a.set_wind(0, windspeed=np.ones(E + 1))
        atm_a.set_wind(0, windspeed=np.array([5.0, 15.0, 25.0]), winddir=np.array([10.0, 130.0, 250.0]))
        a.reset(seeds)
        for _ in range(4):
            a.move_atmos()
        pe = frame(a)
        atm_a.set_r0(float(p.r0))                        # scalar r0: per-environment winds stay in force
        a.reset(seeds)
        for _ in range(4):
            a.move_atmos()
        assert same(frame(a), pe)
        a.set_wfs_path("tensor")
        with pytest.raises(RuntimeError, match="per-environment wind"):
            a.comp_wfs_image(noise=-1.0)
        a.set_wfs_path(a.DEFAULT_WFS_PATH)
        atm_a.set_wind(0, windspeed=ws0 * 1.5, winddir=wd0 + 20.0)   # scalar: common wind again
        atm_b.set_wind(0, windspeed=ws0 * 1.5, winddir=wd0 + 20.0)
        a.reset(seeds); b.reset(seeds)
        for _ in range(4):
            a.move_atmos(); b.move_atmos()
            assert same(frame(a), frame(b))
        atm_a.set_wind(0, windspeed=ws0, winddir=wd0); atm_b.set_wind(0, windspeed=ws0, winddir=wd0)
        a.check_device(); b.check_device()
    finally:
        a.close(); b.close()
