"""Per-environment controller delay (aom_set_delay / aom_set_delay_env; Simulator.set_delay / set_delay_env,
rtc.d_control[0].set_delay): any real delay in [0, 2] frames, one per environment of the batch, through the three-row
delay line of aom_apply_control.  Each environment of a mixed batch computes exactly what a uniform batch with its delay
computes, a fractional delay matches the oracle's blend, and the delay travels with records and survives resets."""
import copy

import numpy as np
import pytest

from delay_line_ref import DelayOracleEnv

pytestmark = pytest.mark.gpu

RTOL = 1e-4
DELAYS = [0.0, 0.5, 1.0, 1.5, 2.0]
F32 = np.float32


def relerr(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


@pytest.fixture(scope="module")
def system10(static10, torch):
    """10x10 tables with a command matrix and two agents whose actors draw exploration."""
    from ao_marl_b200 import calibration
    from ao_marl_b200.init import rtc as rtc_b
    from ao_marl_b200.rl.layout import RLLayout
    t = copy.copy(static10)
    t.imat = calibration.measure_imat(static10)
    t.cmat = rtc_b.cmat_with_btt(t.imat, t.Btt, 5)
    rl = RLLayout(t.Btt.shape[1], dict(parameters_telescope="production_sh_10x10_2m.py", n_zernike_start_end=[0, 80],
                                       n_reverse_filtered_from_cmat=5), None, world_size=3, seed=3)
    torch.manual_seed(20240607)
    with torch.no_grad():
        for p in rl.policies:
            p.mean_linear.weight.normal_(0, 0.05)
            p.log_std_linear.weight.normal_(0, 0.05)
            p.log_std_linear.bias.fill_(-1.0)
    return t, rl


@pytest.fixture(scope="module")
def system40(torch):
    """production_sh_40x40_8m_3layers with the 43 agents of the benchmark."""
    from ao_marl_b200.rl.layout import RLLayout
    from ao_marl_b200.system import build_tables
    t = build_tables("production_sh_40x40_8m_3layers.py", nfilt=5)
    env_rl = dict(parameters_telescope="production_sh_40x40_8m_3layers.py", n_zernike_start_end=[0, 1260],
                  window_n_zernike=20, include_tip_tilt_windowed=True, n_reverse_filtered_from_cmat=5,
                  delayed_assignment=2)
    rl = RLLayout(t.Btt.shape[1], env_rl, None, world_size=44, seed=0)
    return t, rl


def _with_delay(t, d):
    """Tables whose parameter file has controller delay d (Simulator: aom_config.delay = floor(d), then aom_set_delay)."""
    u = copy.copy(t)
    u.delay = float(d)
    return u


def _snap(sim, t, rl):
    E = sim.n_env
    out = {"slopes": sim.rows("SLOPES", t.nslopes), "err": sim.rows("ERR", t.nactu), "com": sim.rows("COM", t.nactu),
           "volts": sim.rows("VOLTS", t.nactu), "state": sim.rows("STATE", rl.state_dim),
           "reward": sim.buffer("REWARD").view(E, rl.n_agents), "action": sim.rows("ACTION", rl.action_dim)}
    return {k: v.cpu().numpy().copy() for k, v in out.items()}


def _actions(rl, E, i):
    """Deterministic actions of step i for aom_step mode 1 (the same in every context)."""
    r = np.random.default_rng(1000 + i)
    return (r.standard_normal((E, rl.action_dim)) * 0.3).astype(F32)


def _steps(sim, t, rl, modes, torch, switch=None):
    """One aom_step per entry of `modes` (0: actors, 1: given actions, 2: integrator); switch(i, sim) runs before step i."""
    out = []
    for i, m in enumerate(modes):
        if switch is not None:
            switch(i, sim)
        if m == 1:
            sim.rows("ACTION", rl.action_dim).copy_(torch.as_tensor(_actions(rl, sim.n_env, i), device="cuda"))
        sim.step(mode=m)
        out.append(_snap(sim, t, rl))
    return out


def _linear_step(sim):
    """The linear half-step of aom_step: what follows an aom_reset (AoEnv.reset)."""
    sim.state_begin()
    sim.move_atmos()
    sim.comp_wfs_image()
    sim.do_centroids()
    sim.do_control()
    sim.state_end()


def _seeds(E):
    return (np.arange(E, dtype=np.int64) * 7919 + 1234)


MODES = [0, 0, 0, 0, 1, 1, 1, 2, 2, 0, 0, 0]


# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("d", DELAYS)
def test_against_oracle_10x10(d, system10, oracle_tab10, torch):
    """Uniform delay d: 12 closed-loop steps with exploring agents match the oracle with the three-row delay line (slopes,
    commands, voltages, rewards, state, actions at rel 1e-4)."""
    from ao_marl_b200.lib import Simulator
    t, rl = system10
    sim = Simulator(_with_delay(t, d), 3, rl)
    try:
        assert sim.delay == F32(d) and sim.delay_env is None and sim.cfg.delay == int(d)
        seeds = np.array([1234, 4321, 999], dtype=np.int64)
        sim.reset(seeds)
        envs = [DelayOracleEnv(oracle_tab10, t.cmat, t.Btt, t.P, rl, seed=int(s), delay=d) for s in seeds[:2]]
        for o, s in zip(envs, seeds):
            o.reset(int(s))
        _linear_step(sim)
        states = [o.linear_step() for o in envs]
        worst = {}
        for it in range(12):
            sim.step(mode=0)
            got = _snap(sim, t, rl)
            for e, o in enumerate(envs):
                a, _ = o.actors(states[e])
                worst["actions"] = max(worst.get("actions", 0), relerr(got["action"][e], a))
                states[e], r = o.env_step(got["action"][e])
                for k, (x, y) in dict(slopes=(got["slopes"][e], o.slopes), commands=(got["com"][e], o.com),
                                      volts=(got["volts"][e], o.volts), rewards=(got["reward"][e], r),
                                      state=(got["state"][e], states[e])).items():
                    worst[k] = max(worst.get(k, 0), relerr(x, y))
        sim.check_device()
    finally:
        sim.close()
    print("delay", d, "worst rel errors over 12 steps:", worst)
    for k, v in worst.items():
        assert v < RTOL, (d, k, worst)


def _impulse(sim, t, rl, torch, n):
    """Open loop, an action impulse in environment 1 at step 1: max |err[1] - err[0]| after each step."""
    E = sim.n_env
    sim.reset(np.full(E, 5, dtype=np.int64))
    sim.set_loop(False)
    errs = []
    try:
        for it in range(n):
            a = torch.zeros((E, rl.action_dim), device="cuda")
            if it == 1:
                a[1, 0] = 5.0
            sim.rows("ACTION", rl.action_dim).copy_(a)
            sim.step(mode=1)
            e = sim.rows("ERR", t.nactu)
            errs.append(float((e[1] - e[0]).abs().max()))
    finally:
        sim.set_loop(True)
    return errs


def test_impulse_delay_two(system10, torch):
    """The impulse of test_delay_impulse shows in err one frame later for delay 2 than for delay 1, and a fractional delay
    of 1.5 shows it in both frames.  The delays are changed on one context with set_delay."""
    from ao_marl_b200.lib import Simulator
    t, rl = system10
    sim = Simulator(t, 3, rl)
    try:
        first = {}
        for d in (0.0, 1.0, 2.0, 1.5):
            sim.set_delay(d)
            errs = _impulse(sim, t, rl, torch, 5)
            first[d] = next(i for i, x in enumerate(errs) if x > 0)
            assert all(x == 0.0 for x in errs[:first[d]]), (d, errs)
        assert first == {0.0: 1, 1.0: 2, 2.0: 3, 1.5: 2}, first
        sim.check_device()
    finally:
        sim.close()


# ------------------------------------------------------------------------------------------------------------------
def _mixed_conditions(sim, t, E):
    """Per-environment delays cycling through DELAYS, with per-environment gains and noise (the d0 / d1 files differ in
    all three)."""
    delay = np.array([DELAYS[e % len(DELAYS)] for e in range(E)], F32)
    gain = np.array([(0.3, 0.5, 0.7)[e % 3] for e in range(E)], F32)
    noise = np.array([(-1.0, 3.0, 0.0, 3.0)[e % 4] for e in range(E)], F32)
    return delay, gain, noise


@pytest.mark.parametrize("name,E", [("10x10", 10), ("40x40", 200)])
def test_mixed_batch_bit_identical(name, E, request, torch):
    """A batch with per-environment delays {0, 0.5, 1, 1.5, 2, ...}, gains and noise: over aom_step modes 0, 1 and 2, every
    environment's slopes, err, com, volts, state, rewards and actions equal those of the same environment in a batch whose
    common delay is its delay (same seeds, same per-environment gains and noise)."""
    from ao_marl_b200.lib import Simulator
    t, rl = request.getfixturevalue("system10" if name == "10x10" else "system40")
    seeds = _seeds(E)

    def run(sim, delay_env, common):
        delay, gain, noise = _mixed_conditions(sim, t, E)
        sim.set_gain(gain)
        sim.set_wfs_noise_env(noise=noise)
        if delay_env:
            sim.set_delay(delay)
            assert np.array_equal(sim.delay_env, delay)
        else:
            assert sim.delay == F32(common) and sim.delay_env is None
        sim.reset(seeds)
        out = _steps(sim, t, rl, MODES, torch)
        sim.check_device()
        return out, delay

    sim = Simulator(t, E, rl)
    try:
        got, delay = run(sim, True, None)
    finally:
        sim.close()
    assert np.abs(got[-1]["volts"]).max() > 0 and np.abs(got[3]["action"]).max() > 0
    for d in DELAYS:
        ref = Simulator(_with_delay(t, d), E, rl)
        try:
            want, _ = run(ref, False, d)
        finally:
            ref.close()
        envs = np.flatnonzero(delay == F32(d))
        for i in range(len(MODES)):
            for k in want[i]:
                assert np.array_equal(got[i][k][envs], want[i][k][envs]), (d, i, k)


def test_delay_changed_mid_episode(system10, torch):
    """Per-environment delays changed at step 6 (and a common delay set while they are in force) equal, environment by
    environment, a uniform batch whose delay was switched at the same step."""
    from ao_marl_b200.lib import Simulator
    t, rl = system10
    E = 5
    d1 = np.array(DELAYS, F32)
    d2 = d1[::-1].copy()
    seeds = _seeds(E)

    def switch_env(i, sim):
        if i == 6:
            sim.set_delay_env(d2)
        if i == 9:
            sim.set_delay(0.0)                       # the common value: per-environment delays stay in force
            assert np.array_equal(sim.delay_env, d2)

    sim = Simulator(t, E, rl)
    try:
        sim.set_delay_env(d1)
        sim.reset(seeds)
        got = _steps(sim, t, rl, MODES, torch, switch_env)
        sim.check_device()
    finally:
        sim.close()
    for e in range(E):
        ref = Simulator(_with_delay(t, d1[e]), E, rl)
        try:
            ref.reset(seeds)
            want = _steps(ref, t, rl, MODES, torch, lambda i, s: s.set_delay(d2[e]) if i == 6 else None)
            ref.check_device()
        finally:
            ref.close()
        for i in range(len(MODES)):
            for k in want[i]:
                assert np.array_equal(got[i][k][e], want[i][k][e]), (e, i, k)


def test_reset_envs_clears_the_delay_line(system10, torch):
    """Delay 2: after aom_reset_envs an environment's next voltages are zeros (com1 and com2 cleared), and from then on it
    computes what a batch reset with its new seed and given one linear step computes."""
    from ao_marl_b200.lib import Simulator
    t, rl = system10
    E = 4
    seeds = _seeds(E)
    new = np.array([99991], dtype=np.int64)
    sim = Simulator(_with_delay(t, 2.0), E, rl)
    try:
        sim.set_delay_env([2.0, 2.0, 1.5, 2.0])
        sim.reset(seeds)
        _steps(sim, t, rl, [0] * 6, torch)
        assert np.abs(sim.rows("VOLTS", t.nactu).cpu().numpy()[1]).max() > 0
        sim.reset_envs(np.array([1], np.int32), new)
        got = _steps(sim, t, rl, [0] * 6, torch)
        assert np.abs(got[0]["volts"][1]).max() == 0.0
        sim.check_device()
    finally:
        sim.close()
    ref = Simulator(_with_delay(t, 2.0), E, rl)
    try:
        s2 = seeds.copy()
        s2[1] = new[0]
        ref.reset(s2)
        _linear_step(ref)
        want = _steps(ref, t, rl, [0] * 5, torch)
        ref.check_device()
    finally:
        ref.close()
    for i in range(5):
        for k in want[i]:
            assert np.array_equal(got[i + 1][k][1], want[i][k][1]), (i, k)


def test_save_load_copy_carry_the_delay(system10, torch):
    """copy_envs across environments with different delays and a load into another context: the destination takes the
    record's delay (aom_get_condition, Simulator.delay_env, rtc.d_control[0].delay), every other environment keeps its
    own, and the copies continue bit for bit as their sources."""
    import ctypes
    from ao_marl_b200.lib import COND, Simulator
    from ao_marl_b200.supervisor.components import RtcB200
    t, rl = system10
    E = 4
    a, b = Simulator(t, E, rl), Simulator(_with_delay(t, 1.0), E, rl)
    try:
        rtc = RtcB200(a, copy.deepcopy(t.config), t)
        a.set_delay_env([0.0, 2.0, 0.5, 1.5])
        a.reset(_seeds(E))
        b.reset(_seeds(E) + 3)
        _steps(a, t, rl, [0] * 5, torch)
        _steps(b, t, rl, [0] * 2, torch)
        b.load_envs([3], a.save_envs([1]))
        a.copy_envs([1], [0])
        assert np.array_equal(a.delay_env, np.array([2.0, 2.0, 0.5, 1.5], F32))
        assert np.array_equal(rtc.d_control[0].delay, a.delay_env)
        assert np.array_equal(b.delay_env, np.array([1.0, 1.0, 1.0, 2.0], F32)) and b.delay == F32(1.0)
        common, per_env, values = ctypes.c_float(), ctypes.c_int(), np.zeros(E, F32)
        assert b.lib.aom_get_condition(b._ctx, COND["DELAY"], 0, ctypes.byref(common),
                                       values.ctypes.data_as(ctypes.c_void_p), ctypes.byref(per_env)) == 0
        assert common.value == 1.0 and per_env.value == 1 and np.array_equal(values, b.delay_env)
        ga = _steps(a, t, rl, [0, 0, 2, 0, 0, 0], torch)
        gb = _steps(b, t, rl, [0, 0, 2, 0, 0, 0], torch)
        for i in range(6):
            for k in ga[i]:
                assert np.array_equal(ga[i][k][0], ga[i][k][1]), (i, k)
                assert np.array_equal(gb[i][k][3], ga[i][k][1]), (i, k)
        rtc.d_control[0].set_delay(1.0)
        assert a.delay_env is None and a.delay == F32(1.0) and rtc.d_control[0].delay == F32(1.0)
        a.check_device()
        b.check_device()
    finally:
        a.close()
        b.close()


def _conditions(sim):
    import ctypes
    from ao_marl_b200.lib import COND
    out = {}
    for name, k in COND.items():
        for l in range(sim.cfg.n_layers if name in ("AMP", "WIND_X", "WIND_Y") else 1):
            c, p, v = ctypes.c_float(), ctypes.c_int(), np.zeros(sim.n_env, F32)
            assert sim.lib.aom_get_condition(sim._ctx, k, l, ctypes.byref(c), v.ctypes.data_as(ctypes.c_void_p),
                                             ctypes.byref(p)) == 0
            out[name, l] = (c.value, p.value, v.tobytes())
    return out


def test_invalid_delays_change_nothing(system10, torch):
    """Non-finite delays, delays outside [0, 2] and arrays of the wrong length are refused and leave every condition as
    it was; 6 (AOM_COND_COUNT of builds without the delay) is still not a condition."""
    from ao_marl_b200.lib import Simulator
    t, rl = system10
    E = 4
    sim = Simulator(t, E, rl)
    try:
        sim.set_delay_env([0.0, 0.5, 2.0, 1.0])
        sim.set_gain_env([0.1, 0.2, 0.3, 0.4])
        before = _conditions(sim)
        bad = [(lambda: sim.set_delay(np.nan), "not finite"), (lambda: sim.set_delay(np.inf), "not finite"),
               (lambda: sim.set_delay(2.5), r"\[0, 2\]"), (lambda: sim.set_delay(-0.25), r"\[0, 2\]"),
               (lambda: sim.set_delay_env([0.0, np.nan, 1.0, 1.0]), "environment 1 is not finite"),
               (lambda: sim.set_delay_env([0.0, 1.0, 1.0, 2.0001]), r"environment 3 must be in \[0, 2\]"),
               (lambda: sim.set_delay_env([0.0, 1.0, 1.0]), "expected a scalar or 4 values"),
               (lambda: sim.set_delay_env(np.ones(5)), "expected a scalar or 4 values")]
        for i, (call, msg) in enumerate(bad):
            with pytest.raises(ValueError, match=msg):
                call()
            assert _conditions(sim) == before, i
        assert sim.lib.aom_get_condition(sim._ctx, 6, 0, None, None, None) == -1
        with pytest.raises(NotImplementedError, match=r"\[0, 2\]"):
            Simulator(_with_delay(t, 2.5), E, rl)
        sim.check_device()
    finally:
        sim.close()


def test_nan_reaches_volts_when_its_delay_says(system10, torch):
    """A NaN written into one environment's com at call 0 of aom_apply_control reaches that environment's volts at the
    calls its delay reads it (0: call 0; 0.5: 0, 1; 1: 1; 1.5: 1, 2; 2: 2), in that column only, and never another
    environment's row."""
    from ao_marl_b200.lib import Simulator
    t, rl = system10
    E = len(DELAYS)
    when = {0.0: {0}, 0.5: {0, 1}, 1.0: {1}, 1.5: {1, 2}, 2.0: {2}}
    sim = Simulator(t, E, rl)
    try:
        sim.set_delay_env(DELAYS)
        for e, d in enumerate(DELAYS):
            sim.reset(_seeds(E))
            _steps(sim, t, rl, [2, 2, 2], torch)
            com = sim.buffer("COM").view(E, -1)
            j = 7
            keep = float(com[e, j])
            for call in range(4):
                if call == 0:
                    com[e, j] = float("nan")
                elif call == 1:
                    com[e, j] = keep
                sim.apply_control()
                v = sim.rows("VOLTS", t.nactu).cpu().numpy()
                bad = ~np.isfinite(v)
                assert bool(bad[e, j]) == (call in when[d]), (d, call)
                bad[e, j] = False
                assert not bad.any(), (d, call)
        sim.check_device()
    finally:
        sim.close()


def test_roket_with_delay_two(torch):
    """ROKET with a uniform delay of 2 frames: its loop filter takes d = 3, the breakdown leaves the loop untouched
    (commands equal those of the same run without it) and its contributors are finite; fractional and per-environment
    delays are refused."""
    from ao_marl_b200.env.ao_env import AoEnv
    from ao_marl_b200.env.config_rl import Config
    cfg = Config(parameters_telescope="production_sh_10x10_2m.py", n_zernike_start_end=[0, 80], n_reverse_filtered_from_cmat=5)
    env = AoEnv(cfg, n_env=2, world_size=3, initial_seed=77, roket=True)
    try:
        sup = env.supervisor
        sup.sim.set_delay(1.5)
        with pytest.raises(NotImplementedError, match="whole frames"):
            sup.init_config_roket(N_total=30, N_preloop=10, agent=None, gamma=1.0)
        sup.sim.set_delay_env([2.0, 1.0])
        with pytest.raises(NotImplementedError, match="one delay"):
            sup.init_config_roket(N_total=30, N_preloop=10, agent=None, gamma=1.0)
        sup.sim.set_delay_env(None)
        sup.sim.set_delay(2.0)
        sup.init_config_roket(N_total=30, N_preloop=10, agent=None, gamma=1.0)
        assert sup.delay == 3
        env.reset()
        a = np.zeros(env.action_size, np.float32)
        for step in range(30):
            env.rl_step(action=a, linear_control=True, apply_control=False, compute_tar_psf=False)
            sup.do_error_breakdown(a)
            env.linear_step()
        com_roket = sup.sim.rows("COM", sup.nactus).clone()
        for name in ("trunc_com", "alias_wfs_com", "H_com", "bp_com", "mod_com"):
            x = getattr(sup, name)
            assert bool(torch.isfinite(x).all()) and float(x[10:].abs().max()) > 0.0, name
    finally:
        env.sim.close()
    ref = AoEnv(cfg, n_env=2, world_size=3, initial_seed=77)
    try:
        ref.sim.set_delay(2.0)
        ref.reset()
        a = np.zeros(ref.action_size, np.float32)
        for _ in range(30):
            ref.rl_step(action=a, linear_control=True, apply_control=True)
            ref.linear_step()
        com_plain = ref.sim.rows("COM", com_roket.shape[1]).clone()
    finally:
        ref.sim.close()
    assert torch.equal(com_roket, com_plain)
