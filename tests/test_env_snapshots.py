"""Per-environment snapshots (aom_save_envs / aom_load_envs, Simulator / RlSupervisor / AoEnv / StepLearner.save_envs /
load_envs / copy_envs): a loaded environment computes bit for bit what the saved one would have computed, in the same
context or another one with the same configuration; every other environment computes what it would have computed
without the call.  Every comparison is exact."""
import ctypes

import numpy as np
import pytest

E = 130                                 # straddles the 128-row M tile of the integer contractions
ENV_RL_43 = dict(n_zernike_start_end=[0, 1260], window_n_zernike=20, include_tip_tilt_windowed=True,
                 n_reverse_filtered_from_cmat=5, delayed_assignment=2)


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


@pytest.fixture(scope="module")
def tables40(torch):
    from ao_marl_b200.system import build_tables
    from ao_marl_b200.rl.layout import RLLayout
    t = build_tables("production_sh_40x40_8m_3layers.py", nfilt=5)
    rl = RLLayout(t.Btt.shape[1], dict(ENV_RL_43, parameters_telescope="production_sh_40x40_8m_3layers.py"), None, 44,
                  seed=0)
    return t, rl


def _conditions(sim, n):
    """Stochastic actions, per-frame Strehl (pending sums carried), photon + read noise on every third environment,
    per-environment winds on layer 1."""
    sim.step_with_strehl(True)
    noise = np.where(np.arange(n) % 3 == 0, 3.0, -1.0).astype(np.float32)
    sim.set_wfs_noise_env(noise=noise)
    r = np.random.default_rng(5)
    speed = float(np.hypot(sim.cfg.deltax[1], sim.cfg.deltay[1]))
    ang = r.uniform(0, 2 * np.pi, n)
    sim.set_layer_wind(1, (speed * np.cos(ang)).astype(np.float32), (speed * np.sin(ang)).astype(np.float32))


@pytest.fixture(scope="module")
def sims(tables40):
    from ao_marl_b200.lib import Simulator
    t, rl = tables40
    a, b = Simulator(t, E, rl), Simulator(t, 8, rl)
    _conditions(a, E)
    _conditions(b, 8)
    yield a, b
    a.close()
    b.close()


def _logical(sim, layer, env):
    n = int(sim.cfg.screen_dim[layer])
    scr = sim.buffer("SCREEN", layer).view(sim.n_env, n, n)[env]
    ox, oy = int(sim.buffer("RING_OX", layer)[env]), int(sim.buffer("RING_OY", layer)[env])
    return np.roll(scr.cpu().numpy(), (-oy, -ox), axis=(0, 1))


def _outputs(sim, t, rl, envs=None):
    """Rows of every environment (or of `envs`): slopes, com, volts, state, reward, action, Strehl."""
    n = sim.n_env
    idx = slice(None) if envs is None else list(envs)
    out = {"slopes": sim.rows("SLOPES", t.nslopes), "com": sim.rows("COM", t.nactu), "volts": sim.rows("VOLTS", t.nactu),
           "state": sim.rows("STATE", rl.state_dim), "reward": sim.buffer("REWARD").view(n, rl.n_agents),
           "action": sim.rows("ACTION", rl.action_dim), "strehl": sim.buffer("STREHL").view(n, 4)}
    return {k: v[idx].cpu().numpy().copy() for k, v in out.items()}


def _screens(sim, envs):
    return {(l, e): _logical(sim, l, e) for l in range(sim.cfg.n_layers) for e in envs}


def _run(sim, seeds, steps, at=None, action=None):
    """reset, then `steps` aom_step calls; action() before step `at` (1-based).  Outputs after every step."""
    sim.reset(seeds)
    out = []
    for i in range(1, steps + 1):
        if i == at:
            action()
        sim.step(mode=0)
        out.append(_outputs(sim, sim.tables, sim.rl))
    return out


@pytest.mark.gpu
def test_copy(sims, tables40, torch):
    """After 7 steps three environments are copied onto three others (one across the 128 boundary): for 9 steps every
    destination equals its source (logical screens, slopes, com, volts, state, reward, action, Strehl); every other
    environment equals the run without the copy."""
    a, _ = sims
    t, rl = tables40
    seeds = 1000 + 13 * np.arange(E, dtype=np.int64)
    src, dst = np.array([3, 127, 64]), np.array([20, 128, 129])
    x, y = [], []
    a.reset(seeds)
    for i in range(16):
        if i == 7:
            assert a.env_state_bytes() % 16 == 0
            a.copy_envs(src, dst)
        a.step(mode=0)
        x.append(_outputs(a, t, rl))
        if i >= 7:
            scr = _screens(a, np.concatenate([src, dst]))
            for s, d in zip(src, dst):
                for l in range(a.cfg.n_layers):
                    assert np.array_equal(scr[l, s], scr[l, d]), (i, l, s, d)
    end_a = {l: (a.buffer("SCREEN", l).view(E, -1)[np.setdiff1d(np.arange(E), dst)].cpu().numpy(),
                 a.buffer("RING_OX", l).cpu().numpy(), a.buffer("RING_OY", l).cpu().numpy()) for l in range(a.cfg.n_layers)}
    y = _run(a, seeds, 16)
    a.check_device()
    keep = np.setdiff1d(np.arange(E), dst)
    for i in range(16):
        for k in x[i]:
            assert np.array_equal(x[i][k][keep], y[i][k][keep]), (i, k)
            if i >= 7:
                assert np.array_equal(x[i][k][src], x[i][k][dst]), (i, k)
    for l in range(a.cfg.n_layers):
        assert np.array_equal(end_a[l][0], a.buffer("SCREEN", l).view(E, -1)[keep].cpu().numpy()), l
        assert np.array_equal(end_a[l][1][keep], a.buffer("RING_OX", l).cpu().numpy()[keep])
        assert np.array_equal(end_a[l][2][keep], a.buffer("RING_OY", l).cpu().numpy()[keep])
    assert np.abs(x[-1]["action"]).max() > 0 and x[-1]["strehl"][:, 1].min() > 0
    assert not np.array_equal(x[6]["com"][dst], x[6]["com"][src])          # the destinations were other environments


@pytest.mark.gpu
def test_rewind_and_resume(sims, tables40, torch):
    """Save two environments at step 5, step 6 more; load the records into the same slots and replay: the same outputs.
    Load them into a context of 8 environments whose history head, noise frame and decision counters differ (stepped
    once more since its reset): the same outputs there too."""
    a, b = sims
    t, rl = tables40
    envs = np.array([5, 77])
    a.reset(2000 + np.arange(E, dtype=np.int64))
    for _ in range(5):
        a.step(mode=0)
    snap = a.save_envs(envs)
    ref = []
    for _ in range(6):
        a.step(mode=0)
        ref.append(_outputs(a, t, rl, envs) | {"screens": _screens(a, envs)})
    a.load_envs(envs, snap)
    for j in range(6):
        a.step(mode=0)
        o = _outputs(a, t, rl, envs)
        for k in o:
            assert np.array_equal(o[k], ref[j][k]), ("rewind", j, k)
        s = _screens(a, envs)
        assert all(np.array_equal(s[key], ref[j]["screens"][key]) for key in s), ("rewind", j)
    b.reset(77 + np.arange(8, dtype=np.int64))
    for _ in range(6):
        b.step(mode=0)
    slots = np.array([6, 1])
    b.load_envs(slots, snap.cpu())                    # a CPU copy (torch.save) loads as well
    for j in range(6):
        b.step(mode=0)
        o = _outputs(b, t, rl, slots)
        for k in o:
            assert np.array_equal(o[k], ref[j][k]), ("resume", j, k)
        s = _screens(b, slots)
        assert all(np.array_equal(s[l, d], ref[j]["screens"][l, e]) for l in range(b.cfg.n_layers)
                   for d, e in zip(slots, envs)), ("resume", j)
    a.check_device()
    b.check_device()


@pytest.mark.gpu
def test_fast_autoreset(sims, tables40, torch):
    """Context B: reset_envs([j], [s]), save j.  Context A mid-run: loading that record into slot e equals reset_envs([e],
    [s]) on A -- every environment's outputs in the following steps, and the transitions StepLearner pushes."""
    from ao_marl_b200.env.trainer import StepLearner
    from ao_marl_b200.rl.sac import BatchedSAC
    a, b = sims
    t, rl = tables40
    seeds = 3000 + np.arange(E, dtype=np.int64)
    e, s = 128, 4242
    for sim in (a, b):                                # the new episode's conditions: the common ones in both contexts
        sim.set_wfs_noise_env(None, None)
        sim.set_layer_wind(1, None, None)
    b.reset(11 + np.arange(8, dtype=np.int64))
    b.step(mode=0)
    b.reset_envs([3], [s])
    rec = b.save_envs([3])

    def run(restart):
        L = BatchedSAC.from_layout(rl, device="cuda", seed=3, memory_size=4096)
        a.reset(seeds)
        a.step(mode=0)
        sl = StepLearner(a, rl, L)
        out = []
        for g in range(1, 9):
            if g == 3:
                restart(sl)
            sl.step(learn=False)
            out.append(_outputs(a, t, rl))
        return out, L.memory

    x, mx = run(lambda sl: sl.load_envs([e], rec))
    y, my = run(lambda sl: sl.reset_envs([e], [s]))
    a.check_device()
    for i in range(len(x)):
        for k in x[i]:
            assert np.array_equal(x[i][k], y[i][k]), (i, k)
    assert mx.position == my.position > 0
    for name in ("s", "a", "r", "s2", "m"):
        assert torch.equal(getattr(mx, name)[:, :mx.position], getattr(my, name)[:, :my.position]), name


@pytest.mark.gpu
def test_conditions_travel(tables40, torch):
    """A record of an environment with its own amplitude, wind, noise, photon count and gain, loaded into a batch with
    common values: that environment runs with its saved conditions; the others are unchanged."""
    from ao_marl_b200.lib import Simulator
    t, rl = tables40
    n = 6
    b, a = Simulator(t, n, rl), Simulator(t, n, rl)
    try:
        for sim in (a, b):
            sim.step_with_strehl(True)
        amp = np.full(n, b.cfg.amp[0], np.float32)
        amp[2] *= 1.7
        b.set_layer_amp(0, amp)
        dx = np.full(n, b.cfg.deltax[2], np.float32)
        dy = np.full(n, b.cfg.deltay[2], np.float32)
        dx[2], dy[2] = -0.9, 0.55
        b.set_layer_wind(2, dx, dy)
        b.set_wfs_noise_env(noise=np.where(np.arange(n) == 2, 2.0, -1.0), nphotons=np.where(np.arange(n) == 2, 50.0, b.wfs_nphotons))
        b.set_gain(np.where(np.arange(n) == 2, 0.35, b.cfg.gain).astype(np.float32))
        b.reset(500 + np.arange(n, dtype=np.int64))
        for _ in range(3):
            b.step(mode=0)
        rec = b.save_envs([2])
        ref = []
        for _ in range(5):
            b.step(mode=0)
            ref.append(_outputs(b, t, rl, [2]) | {"screens": _screens(b, [2])})
        seeds = 900 + np.arange(n, dtype=np.int64)
        y = _run(a, seeds, 8)
        a.reset(seeds)
        for _ in range(3):
            a.step(mode=0)
        a.load_envs([4], rec)
        assert a.wfs_noise_env is not None and a.gain_env is not None and a.gain_env[4] == np.float32(0.35)
        for j in range(5):
            a.step(mode=0)
            o = _outputs(a, t, rl)
            for k in o:
                assert np.array_equal(o[k][4], ref[j][k][0]), (j, k)
                assert np.array_equal(o[k][[0, 1, 2, 3, 5]], y[3 + j][k][[0, 1, 2, 3, 5]]), (j, k)
            s = _screens(a, [4])
            assert all(np.array_equal(s[l, 4], ref[j]["screens"][l, 2]) for l in range(a.cfg.n_layers)), j
        a.check_device()
        b.check_device()
    finally:
        a.close()
        b.close()


@pytest.mark.gpu
def test_refusals(tables40, static10, torch):
    """A wrong buffer size, a 10x10 record loaded into a 40x40 context, a repeated or out-of-range slot and a load before
    aom_reset: each fails with its documented error and changes nothing."""
    from ao_marl_b200.lib import Simulator
    t, _ = tables40
    a, c = Simulator(t, 4, rl=None), Simulator(static10, 2, rl=None)
    try:
        nb = a.env_state_bytes()
        rec = torch.zeros((1, nb), dtype=torch.uint8, device="cuda")

        def c_load(n, envs, buf):
            envs = np.ascontiguousarray(envs, np.int32)
            return a.lib.aom_load_envs(a._ctx, n, envs.ctypes.data_as(ctypes.c_void_p), ctypes.c_void_p(buf.data_ptr()),
                                       a.stream)

        assert c_load(1, [0], rec) == -4                      # AOM_ERR_STATE: no aom_reset yet
        with pytest.raises(RuntimeError, match="aom_reset must be called"):
            a.load_envs([0], rec)
        with pytest.raises(RuntimeError, match="aom_reset must be called"):
            a.save_envs([0])
        a.reset(np.arange(4, dtype=np.int64) + 40)
        a.move_atmos()
        torch.cuda.synchronize()

        def state():
            return [a.buffer(k, l).cpu().numpy().copy() for l in range(a.cfg.n_layers)
                    for k in ("SCREEN", "RING_OX", "RING_OY", "EXT_COUNT")] + [a.buffer("COM").cpu().numpy().copy()]

        before = state()
        good = a.save_envs([1])
        with pytest.raises(ValueError, match="shape"):
            a.load_envs([0], good[:, :-16])
        with pytest.raises(ValueError, match="shape"):
            a.load_envs([0, 1], good)
        c.reset(np.array([1, 2], np.int64))
        small = c.save_envs([0])
        assert small.shape[1] != nb
        rec[:, :small.shape[1]] = small
        assert c_load(1, [0], rec) == -1                      # AOM_ERR_INVALID: another configuration
        with pytest.raises(ValueError, match="another configuration"):
            a.load_envs([0], rec)
        assert c_load(1, [0], torch.zeros_like(rec)) == -1   # not a record
        two = a.save_envs([1, 2])
        assert c_load(2, [3, 3], two) == -1
        assert c_load(1, [4], good) == -1
        assert c_load(1, [-1], good) == -1
        assert c_load(-1, [0], good) == -1
        with pytest.raises(ValueError, match="duplicate"):
            a.load_envs([3, 3], two)
        with pytest.raises(ValueError, match="out of range"):
            a.load_envs([4], good)
        torch.cuda.synchronize()
        after = state()
        assert all(np.array_equal(x, y) for x, y in zip(before, after))
        assert c_load(0, [0], good) == 0
        a.check_device()
    finally:
        a.close()
        c.close()
