"""Per-environment reset (aom_reset_envs, Simulator / RlSupervisor / AoEnv / StepLearner.reset_envs): a restarted
environment computes exactly what the same environment computes in a batch that was reset with its new seed and given
one linear step, and every other environment computes exactly what it would have computed without the call."""
import copy
import ctypes

import numpy as np
import pytest

# the directions of test_wind_per_env: both signs on both axes, a diagonal, more than one pixel per frame, no wind
WINDS10 = [(1.3, 0.0), (-1.3, 0.0), (0.0, 0.7), (0.0, -0.7), (0.8, 0.8), (-0.6, 0.45), (2.26, -1.7), (0.0, 0.0)]
RESET = [1, 4]


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


@pytest.fixture(scope="module")
def static40():
    from ao_marl_b200 import tables
    from ao_marl_b200.config import load_config_from_file
    return tables.build_static(load_config_from_file("production_sh_40x40_8m_3layers.py"))


@pytest.fixture(scope="module")
def system(static10, torch):
    """10x10 system with two agents (as test_gpu_parity's system10), photon + read noise on the sensor, the Strehl of the
    target every step (long exposure accumulated) and the geometric controller every step."""
    from ao_marl_b200 import calibration
    from ao_marl_b200.init import geo
    from ao_marl_b200.init import rtc as rtc_b
    from ao_marl_b200.lib import Simulator
    from ao_marl_b200.rl.layout import RLLayout
    t = copy.copy(static10)
    t.imat = calibration.measure_imat(static10)
    t.cmat = rtc_b.cmat_with_btt(t.imat, t.Btt, 5)
    geo.build_geo(t)
    t.p_wfs = copy.copy(static10.p_wfs)
    t.p_wfs.noise = 3.0
    rl = RLLayout(t.Btt.shape[1], dict(parameters_telescope="production_sh_10x10_2m.py", n_zernike_start_end=[0, 80],
                                       n_reverse_filtered_from_cmat=5), None, world_size=3, seed=3)
    torch.manual_seed(20240607)
    with torch.no_grad():
        for p in rl.policies:
            p.mean_linear.weight.normal_(0, 0.05)
            p.log_std_linear.weight.normal_(0, 0.05)
            p.log_std_linear.bias.fill_(-1.0)
    sim = Simulator(t, 3, rl)
    sim.step_with_strehl(True)
    sim.step_with_geo(True)
    yield sim, t, rl
    sim.close()


def _logical(sim, layer, env):
    n = int(sim.cfg.screen_dim[layer])
    scr = sim.buffer("SCREEN", layer).view(sim.n_env, n, n)[env]
    ox, oy = int(sim.buffer("RING_OX", layer)[env]), int(sim.buffer("RING_OY", layer)[env])
    return np.roll(scr.cpu().numpy(), (-oy, -ox), axis=(0, 1))


def _atmosphere(sim):
    """Per (layer, environment): logical screen, ring origins, extrusion count."""
    out = {}
    for l in range(sim.cfg.n_layers):
        ox, oy = sim.buffer("RING_OX", l).cpu().numpy(), sim.buffer("RING_OY", l).cpu().numpy()
        cnt = sim.buffer("EXT_COUNT", l).cpu().numpy()
        for e in range(sim.n_env):
            out[l, e] = (_logical(sim, l, e), int(ox[e]), int(oy[e]), int(cnt[e]))
    return out


def _same_atmosphere(a, b, e, n_layers):
    return all(np.array_equal(a[l, e][0], b[l, e][0]) and a[l, e][1:] == b[l, e][1:] for l in range(n_layers))


SCREEN_CASES = [("10x10", "common", "i8"), ("10x10", "winds", "i8"), ("10x10", "common", "ffma"),
                ("40x40", "common", "i8"), ("40x40", "winds", "i8")]


@pytest.mark.gpu
@pytest.mark.parametrize("system_name,wind,path", SCREEN_CASES)
def test_screens(system_name, wind, path, static10, static40, torch):
    """A: reset, 7 moves, reset_envs([1, 4], new), 9 moves.  B: the same 16 moves without the partial reset.  C: reset
    with the new seeds at slots 1 and 4, then 9 moves.  Environments 1 and 4 of A equal C, the others equal B: logical
    screens, ring origins and extrusion counts."""
    from ao_marl_b200.lib import Simulator
    t = static10 if system_name == "10x10" else static40
    E = 8
    seeds = np.arange(E, dtype=np.int64) * 7 + 300
    new = np.array([9001, 9002], dtype=np.int64)
    seeds_c = seeds.copy()
    seeds_c[RESET] = new
    sim = Simulator(t, E, rl=None)
    try:
        sim.set_extrude_path(path)
        NL = sim.cfg.n_layers
        if wind == "winds":
            r = np.random.default_rng(3)
            for l in range(NL):
                if system_name == "10x10":
                    dx, dy = np.array(WINDS10, np.float32).T
                else:
                    speed = float(np.hypot(sim.cfg.deltax[l], sim.cfg.deltay[l]))
                    ang = r.uniform(0, 2 * np.pi, E)
                    dx = (speed * r.uniform(0.6, 1.4, E) * np.cos(ang)).astype(np.float32)
                    dy = (speed * r.uniform(0.6, 1.4, E) * np.sin(ang)).astype(np.float32)
                sim.set_layer_wind(l, dx, dy)

        def run(s, first, then, partial=False):
            sim.reset(s)
            for _ in range(first):
                sim.move_atmos()
            if partial:
                sim.reset_envs(RESET, new)
            for _ in range(then):
                sim.move_atmos()
            return _atmosphere(sim)

        a = run(seeds, 7, 9, partial=True)
        b = run(seeds, 7, 9)
        c = run(seeds_c, 0, 9)
        sim.check_device()
        for e in range(E):
            assert _same_atmosphere(a, c if e in RESET else b, e, NL), e
        assert not np.array_equal(a[0, 1][0], b[0, 1][0])       # the restarted screens are new ones
    finally:
        sim.close()


# ------------------------------------------------------------------------------------------------------------------
def _linear_step(sim):
    """The linear half-step of aom_step with the geometric controller: what follows an aom_reset."""
    sim.state_begin()
    sim.move_atmos()
    sim.do_control_geo()
    sim.apply_control_geo()
    sim.comp_wfs_image()
    sim.do_centroids()
    sim.do_control()
    sim.state_end()


def _snap(sim, t, rl):
    E = sim.n_env
    geo = sim.comp_strehl(1.65, geo=True).cpu().numpy().copy()          # long exposure behind the geometric mirrors
    return {"state": sim.rows("STATE", rl.state_dim).cpu().numpy().copy(),
            "action": sim.rows("ACTION", rl.action_dim).cpu().numpy().copy(),
            "reward": sim.buffer("REWARD").view(E, rl.n_agents).cpu().numpy().copy(),
            "com": sim.rows("COM", t.nactu).cpu().numpy().copy(),
            "slopes": sim.rows("SLOPES", t.nslopes).cpu().numpy().copy(),
            "strehl": sim.buffer("STREHL").view(E, 4).cpu().numpy().copy(),
            "strehl_geo": geo}


def _episode(sim, t, rl, seeds, steps, partial_at=None, envs=(1,), new=(777,)):
    """reset + linear step, then `steps` aom_step calls; reset_envs(envs, new) before step `partial_at` (1-based).
    Snapshots after the linear step and after every step."""
    sim.reset(seeds)
    _linear_step(sim)
    out = [_snap(sim, t, rl)]
    for i in range(1, steps + 1):
        if i == partial_at:
            sim.reset_envs(list(envs), np.asarray(new, np.int64))
        sim.step(mode=0)
        out.append(_snap(sim, t, rl))
    return out


@pytest.mark.gpu
def test_closed_loop(system, torch):
    """Agents drawing exploration noise, noisy sensor, LE Strehl of the main and geometric targets: environment 1 restarted
    before step 6 of 15.  Its fresh step gives reward 0 and the s0 of the fresh-reset run, every later step equals that run
    (state, action, reward, com, slopes, LE Strehl, geometric LE Strehl); the other environments equal the run without
    the partial reset at every step."""
    sim, t, rl = system
    seeds = np.array([1234, 4321, 999], dtype=np.int64)
    seeds_c = seeds.copy()
    seeds_c[1] = 777
    a = _episode(sim, t, rl, seeds, 15, partial_at=6)
    b = _episode(sim, t, rl, seeds, 15)
    c = _episode(sim, t, rl, seeds_c, 9)
    sim.check_device()
    assert np.abs(a[-1]["com"]).max() > 0 and np.abs(a[-1]["action"]).max() > 0
    assert a[-1]["strehl"][1, 1] > 0 and a[-1]["strehl_geo"][1, 1] > 0
    for i in range(16):
        for k in a[i]:
            if i == 0 and k == "reward":
                continue                                   # no reward is computed in the linear step after a reset
            assert np.array_equal(a[i][k][[0, 2]], b[i][k][[0, 2]]), (i, k)
    assert np.array_equal(a[6]["reward"][1], np.zeros(rl.n_agents, np.float32))
    for k in ("state", "com", "slopes", "strehl", "strehl_geo"):
        assert np.array_equal(a[6][k][1], c[0][k][1]), k
    for j in range(1, 10):
        for k in a[6 + j]:
            assert np.array_equal(a[6 + j][k][1], c[j][k][1]), (j, k)


@pytest.mark.gpu
def test_reset_all_equals_reset(system, torch):
    """reset_envs(every environment) + one step == reset + linear step; n = 0 changes nothing."""
    sim, t, rl = system
    seeds = np.array([5, 6, 7], dtype=np.int64)
    seeds2 = np.array([50, 60, 70], dtype=np.int64)
    a = _episode(sim, t, rl, seeds, 4, partial_at=4, envs=(2, 0, 1), new=seeds2[[2, 0, 1]])
    c = _episode(sim, t, rl, seeds2, 0)
    assert np.array_equal(a[4]["reward"], np.zeros_like(a[4]["reward"]))
    for k in ("state", "com", "slopes", "strehl", "strehl_geo"):
        assert np.array_equal(a[4][k], c[0][k]), k
    a = _episode(sim, t, rl, seeds, 5, partial_at=3, envs=(), new=())
    b = _episode(sim, t, rl, seeds, 5)
    for i, (x, y) in enumerate(zip(a, b)):
        for k in x:
            if i or k != "reward":                         # no reward is computed in the linear step after a reset
                assert np.array_equal(x[k], y[k]), (i, k)
    sim.check_device()


@pytest.mark.gpu
def test_errors_and_round1_kernel(static10, torch):
    """Duplicates, out-of-range indices, n < 0 and a call before any reset fail with the right error (Python and C); the
    round-1 sensor kernel refuses while environments are staggered; after the next full reset the outputs equal those of
    a context that never had a partial reset, on the uniform kernels (the round-1 kernel runs again)."""
    from ao_marl_b200.lib import Simulator
    E = 4
    seeds = np.array([11, 12, 13, 14], dtype=np.int64)
    a, b = Simulator(static10, E, rl=None), Simulator(static10, E, rl=None)
    try:
        with pytest.raises(RuntimeError, match="aom_reset must be called"):
            a.reset_envs([0], [1])

        def c_call(n, envs, sds):
            envs = np.ascontiguousarray(envs, np.int32)
            sds = np.ascontiguousarray(sds, np.int64)
            return a.lib.aom_reset_envs(a._ctx, n, envs.ctypes.data_as(ctypes.c_void_p),
                                        sds.ctypes.data_as(ctypes.c_void_p), a.stream)

        assert c_call(1, [0], [1]) == -4                      # AOM_ERR_STATE
        a.reset(seeds)
        assert c_call(2, [1, 1], [1, 2]) == -1                # AOM_ERR_INVALID
        assert c_call(1, [E], [1]) == -1
        assert c_call(1, [-1], [1]) == -1
        assert c_call(-1, [0], [1]) == -1
        assert c_call(0, [0], [1]) == 0
        with pytest.raises(ValueError, match="duplicate"):
            a.reset_envs([2, 2], [1, 2])
        with pytest.raises(ValueError, match="out of range"):
            a.reset_envs([E], [1])
        with pytest.raises(ValueError):
            a.reset_envs([0, 1], [1])
        with pytest.raises(TypeError):
            a.reset_envs([0.0], [1])
        a.set_wfs_path("tensor")
        a.comp_wfs_image(noise=-1.0)                          # in lockstep: the round-1 kernel runs
        a.move_atmos()
        a.reset_envs([1], [99])
        with pytest.raises(RuntimeError, match="staggered"):
            a.comp_wfs_image(noise=-1.0)
        a.set_wfs_path(a.DEFAULT_WFS_PATH)
        for _ in range(3):
            a.move_atmos()
        a.reset(seeds)
        b.reset(seeds)
        for path in ("tensor", a.DEFAULT_WFS_PATH):
            a.set_wfs_path(path)
            b.set_wfs_path(path)
            for _ in range(3):
                a.move_atmos(); b.move_atmos()
                a.comp_wfs_image(noise=2.0); b.comp_wfs_image(noise=2.0)
                a.do_centroids(); b.do_centroids()
                assert np.array_equal(a.rows("SLOPES", static10.nslopes).cpu().numpy(),
                                      b.rows("SLOPES", static10.nslopes).cpu().numpy()), path
                assert all(np.array_equal(_logical(a, 0, e), _logical(b, 0, e)) for e in range(E))
        a.check_device(); b.check_device()
    finally:
        a.close(); b.close()


@pytest.mark.gpu
def test_step_learner(system, torch):
    """StepLearner (learn=False): the replay rows of the restarted environment equal those of a StepLearner started
    after a full reset with its seed; rows whose window spans the reset never appear."""
    from ao_marl_b200.env.trainer import StepLearner
    from ao_marl_b200.rl.sac import BatchedSAC
    sim, t, rl = system
    seeds = np.array([21, 22, 23], dtype=np.int64)
    seeds_c = seeds.copy()
    seeds_c[1] = 555
    f, n_after = 5, 8                                      # environment 1 restarted before step f; its fresh step is f

    def run(s, steps, partial):
        L = BatchedSAC.from_layout(rl, device="cuda", seed=3, memory_size=4096)
        sim.reset(s)
        _linear_step(sim)
        sl = StepLearner(sim, rl, L)
        depth = sl.mdp.depth
        rows = {}                                          # step -> {env: replay slot}
        for g in range(1, steps + 1):
            if partial and g == f:
                sl.reset_envs([1], [555])
            pos = L.memory.position
            sl.step(learn=False)
            first = [f if (partial and e == 1 and g >= f) else 0 for e in range(3)]
            ok = [e for e in range(3) if g - depth - 1 >= first[e]]
            assert L.memory.position - pos == len(ok), g     # no transition spans the reset
            rows[g] = {e: pos + i for i, e in enumerate(ok)}
        return L.memory, rows

    ma, ra = run(seeds, f + n_after, True)
    mc, rc = run(seeds_c, n_after, False)
    sim.check_device()
    pushed = 0
    for j in range(1, n_after + 1):
        assert (1 in ra[f + j]) == (1 in rc[j]), j
        if 1 in rc[j]:
            i, k = ra[f + j][1], rc[j][1]
            for name in ("s", "a", "r", "s2", "m"):
                assert torch.equal(getattr(ma, name)[:, i], getattr(mc, name)[:, k]), (j, name)
            pushed += 1
    assert pushed > 0
