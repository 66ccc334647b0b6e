"""Per-environment guide star, sensor noise and loop gain (aom_set_wfs_noise / aom_set_wfs_noise_env / aom_set_gain_env;
Simulator.set_wfs_noise_env / set_gain, WfsB200.set_noise / set_gs_mag, RtcB200.set_gain with [E] arrays): every
environment of a mixed batch computes exactly what it computes in a uniform batch built with its conditions through
aom_config."""
import copy
import types

import numpy as np
import pytest

# (noise, guide-star magnitude, integrator gain) per environment: none / photon / photon + read noise, four magnitudes
# (the parameter files' 4 and 9 among them), the gains of the parameter files
CONDITIONS = [(-1.0, 4.0, 0.7), (0.0, 9.0, 0.3), (3.0, 6.5, 0.65), (3.0, 11.0, 0.5)]
SEEDS = np.array([1234, 4321, 999, 77], dtype=np.int64)
STEPS = 12


def _nph(t, mag):
    from ao_marl_b200.init.geom import nphotons_for_mags
    c, w = t.config, t.p_wfs
    return nphotons_for_mags(c.p_loop.ittime, w.optthroughput, c.p_tel.diam, w.nxsub, w.zerop, mag)


# ------------------------------------------------------------------------------------------------------------------
def test_magnitude_to_photons_matches_the_builder():
    """nphotons_for_mags (vectorised) equals, as float32, the _nphotons the geometry builder computes for each magnitude
    (and so what Simulator puts in aom_config.nphotons), including the parameter files' own magnitudes 4 and 9."""
    import ctypes
    from ao_marl_b200.config import load_config_from_file
    from ao_marl_b200.init import geom
    from ao_marl_b200.init.geom import nphotons_for_mags
    mags = np.array([4.0, 9.0, 0.0, 5.5, 7.25, 11.0, 13.0, -1.0])
    for name in ("production_sh_10x10_2m.py", "production_sh_40x40_8m_3layers.py",
                 "production_sh_40x40_8m_3layers_d0_noise.py"):
        base = load_config_from_file(name)
        w0, c0 = base.p_wfss[0], base
        vec = nphotons_for_mags(c0.p_loop.ittime, w0.optthroughput, c0.p_tel.diam, w0.nxsub, w0.zerop, mags)
        assert vec.dtype == np.float32 and vec.shape == mags.shape
        scalar = nphotons_for_mags(c0.p_loop.ittime, w0.optthroughput, c0.p_tel.diam, w0.nxsub, w0.zerop, float(mags[1]))
        assert scalar.shape == () and scalar == vec[1]
        for i, m in enumerate(mags):
            c = load_config_from_file(name)
            c.p_wfss[0].gsmag = float(m)
            geom.tel_init(c.p_geom, c.p_tel, c.p_atmos.r0, c.p_loop.ittime, c.p_wfss)
            built = c.p_wfss[0]._nphotons
            f = ctypes.c_float(built).value                  # what aom_config.nphotons holds
            assert np.float32(built) == vec[i] and np.float32(f) == vec[i], (name, m)
        # the file's own magnitude
        c = load_config_from_file(name)
        geom.tel_init(c.p_geom, c.p_tel, c.p_atmos.r0, c.p_loop.ittime, c.p_wfss)
        own = nphotons_for_mags(c.p_loop.ittime, w0.optthroughput, c.p_tel.diam, w0.nxsub, w0.zerop, c.p_wfss[0].gsmag)
        assert own == np.float32(c.p_wfss[0]._nphotons) and float(c.p_wfss[0].gsmag) in (4.0, 9.0)


def test_roket_refuses_per_environment_gains():
    """ROKET's loop filter has one gain: it raises while per-environment gains are in force, and not otherwise."""
    from ao_marl_b200.guardians.roket import Roket
    stub = types.SimpleNamespace(sim=types.SimpleNamespace(gain_env=np.array([0.3, 0.5], np.float32)))
    stub._common_gain = lambda: Roket._common_gain(stub)
    with pytest.raises(NotImplementedError, match="one gain"):
        Roket._common_gain(stub)
    with pytest.raises(NotImplementedError, match="one gain"):
        Roket.do_error_breakdown(stub)
    stub.sim.gain_env = None
    Roket._common_gain(stub)


# ------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


@pytest.fixture(scope="module")
def system10(static10, torch):
    """10x10 tables with a command matrix and two agents (as test_reset_envs' system) whose actors draw exploration."""
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
    """production_sh_40x40_8m_3layers (three layers) with the 43 agents of the benchmark."""
    from ao_marl_b200.rl.layout import RLLayout
    from ao_marl_b200.system import build_tables
    t = build_tables("production_sh_40x40_8m_3layers.py", nfilt=5)
    env_rl = dict(parameters_telescope="production_sh_40x40_8m_3layers.py", n_zernike_start_end=[0, 1260],
                  window_n_zernike=20, include_tip_tilt_windowed=True, n_reverse_filtered_from_cmat=5,
                  delayed_assignment=2)
    rl = RLLayout(t.Btt.shape[1], env_rl, None, world_size=44, seed=0)
    return t, rl


def _with_conditions(t, noise, nph, gain):
    """Tables whose aom_config carries these sensor noise / photon count / gain (the existing uniform path)."""
    u = copy.copy(t)
    u.p_wfs = copy.copy(t.p_wfs)
    u.p_wfs.noise = float(noise)
    u.p_wfs._nphotons = float(nph)
    u.gain = float(gain)
    return u


def _configure(sim, wfs, gemm, keep):
    sim.set_wfs_path(wfs)
    sim.set_gemm_path(gemm)
    sim.step_keeps_image(keep)
    sim.step_with_strehl(True)


def _snap(sim, t, rl, keep):
    E = sim.n_env
    out = {"slopes": sim.rows("SLOPES", t.nslopes), "err": sim.rows("ERR", t.nactu), "com": sim.rows("COM", t.nactu),
           "state": sim.rows("STATE", rl.state_dim), "reward": sim.buffer("REWARD").view(E, rl.n_agents),
           "action": sim.rows("ACTION", rl.action_dim), "strehl": sim.buffer("STREHL").view(E, 4)}
    if keep:
        out["bincube"] = sim.buffer("BINCUBE").view(E, t.p_wfs._nvalid, 256)
    return {k: v.cpu().numpy().copy() for k, v in out.items()}


def _half_step(sim, keep):
    """aom_step mode 0 one call at a time: rl half-step, then the linear half-step."""
    sim.actor_forward()
    sim.rl_control()
    sim.comp_strehl(1.65, phase="both")
    sim.apply_control()
    sim.reward()
    sim.state_begin()
    sim.move_atmos()
    sim.comp_wfs_image(keep_image=keep)
    sim.do_centroids()
    sim.do_control()
    sim.state_end()


def _run(sim, t, rl, keep, half, steps=STEPS):
    sim.reset(SEEDS)
    out = []
    for _ in range(steps):
        if half:
            _half_step(sim, keep)
        else:
            sim.step(mode=0)
        out.append(_snap(sim, t, rl, keep))
    return out


def _mixed(sim, t):
    noise = np.array([c[0] for c in CONDITIONS], np.float32)
    nph = _nph(t, np.array([c[1] for c in CONDITIONS]))
    gain = np.array([c[2] for c in CONDITIONS], np.float32)
    sim.set_wfs_noise_env(noise=noise, nphotons=nph)
    sim.set_gain(gain)
    return noise, nph, gain


# system, sensor path, GEMM path, kept image, half-step calls
CASES = [("10x10", "umma_ws", "tcgen05", False, False), ("10x10", "umma_ws", "tcgen05", True, False),
         ("10x10", "simt", "simt", True, False), ("10x10", "umma", "tf32", False, True),
         ("40x40", "umma_ws", "tcgen05", False, False), ("40x40", "umma", "tcgen05", True, False),
         ("40x40", "simt", "tf32", True, False), ("40x40", "umma_ws", "simt", True, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,wfs,gemm,keep,half", CASES)
def test_mixed_batch_bit_identical(name, wfs, gemm, keep, half, request, torch):
    """Four environments with (noise, magnitude, gain) = (-1, 4, 0.7), (0, 9, 0.3), (3, 6.5, 0.65), (3, 11, 0.5): over 12
    closed-loop steps with exploring agents and the per-frame Strehl, slopes, err, com, state, rewards, actions, Strehl
    and the kept detector cube of each environment equal the same environment of a uniform batch (same seeds) whose
    aom_config carries its conditions."""
    from ao_marl_b200.lib import Simulator
    t, rl = request.getfixturevalue("system10" if name == "10x10" else "system40")
    E = len(CONDITIONS)
    sim = Simulator(t, E, rl)
    try:
        _configure(sim, wfs, gemm, keep)
        noise, nph, gain = _mixed(sim, t)
        got = _run(sim, t, rl, keep, half)
        sim.check_device()
    finally:
        sim.close()
    assert np.abs(got[-1]["com"]).max() > 0 and np.abs(got[-1]["action"]).max() > 0
    for e in range(E):
        ref = Simulator(_with_conditions(t, noise[e], nph[e], gain[e]), E, rl)
        try:
            _configure(ref, wfs, gemm, keep)
            want = _run(ref, t, rl, keep, half)
            ref.check_device()
        finally:
            ref.close()
        for i in range(STEPS):
            for k in want[i]:
                assert np.array_equal(got[i][k][e], want[i][k][e]), (e, i, k)


@pytest.mark.gpu
def test_against_oracle_40x40_d0_noise(torch):
    """production_sh_40x40_8m_3layers_d0_noise, two environments with their own magnitude, noise and gain: each against
    an oracle built with its nphotons / noise / gain -- photon counts teacher-forced and compared as in
    test_gpu_parity40.test_40x40_d0_noise_closed_loop_against_oracle, float quantities at rel 1e-4."""
    import test_gpu_parity40 as par
    from ao_marl_b200.system import build_system, build_tables
    t = build_tables("production_sh_40x40_8m_3layers_d0_noise.py", nfilt=5)
    sim, t, rl = build_system("production_sh_40x40_8m_3layers_d0_noise.py", 2,
                              env_rl=dict(par.ENV_RL_43, delayed_assignment=1), world_size=44, seed=0, tables=t)
    try:
        noise = np.array([3.0, 0.0], np.float32)
        nph = _nph(t, np.array([9.0, 7.0]))
        gain = np.array([0.3, 0.5], np.float32)
        sim.set_wfs_noise_env(noise=noise, nphotons=nph)
        sim.set_gain(gain)
        sim.reset(par.SEEDS)
        envs = [par.oracle_env(_with_conditions(t, noise[e], nph[e], gain[e]), rl, s) for e, s in enumerate(par.SEEDS)]
        rep = par.closed_loop_compare("40x40_d0_noise_per_env", sim, t, rl, envs, 8, torch, noisy=True)
        assert rep["count_mismatch_pixels"] <= 2e-5 * rep["count_pixels"] + 2, rep
        assert rep["phase"] < 2e-5 and rep["bincube"] < par.RTOL, rep
        assert rep["screen_after_reset"] < 3e-5, rep
        for k in ("slopes", "commands", "rewards", "state", "actions"):
            assert rep[k] < par.RTOL, (k, rep)
        sim.check_device()
    finally:
        sim.close()


def _frames(sim, t, n, keep=True, noise=None):
    out = []
    for _ in range(n):
        sim.move_atmos()
        sim.comp_wfs_image(keep_image=keep, noise=noise)
        sim.do_centroids()
        sim.do_control()
        f = {"slopes": sim.rows("SLOPES", t.nslopes), "com": sim.rows("COM", t.nactu)}
        if keep:
            f["bincube"] = sim.buffer("BINCUBE").view(sim.n_env, t.p_wfs._nvalid, 256)
        out.append({k: v.cpu().numpy().copy() for k, v in f.items()})
    return out


def _same(a, b):
    return all(np.array_equal(x[k], y[k]) for x, y in zip(a, b) for k in x)


@pytest.mark.gpu
def test_back_to_uniform_and_noise_free_frames(system10, torch):
    """Both arrays NULL (and the common gain) again: identical to a context that never had per-environment values.
    comp_wfs_image(noise=-1) with per-environment noise in force is noise-free for every environment, scaled by each
    environment's photon count; noise=None draws each environment's own noise."""
    from ao_marl_b200.lib import Simulator
    t, _ = system10
    E = 3
    seeds = SEEDS[:E]
    a, b = Simulator(t, E, rl=None), Simulator(t, E, rl=None)
    try:
        noise, nph = np.array([3.0, 0.0, -1.0], np.float32), _nph(t, np.array([9.0, 6.0, 11.0]))
        a.set_wfs_noise_env(noise=noise, nphotons=nph)
        a.set_gain(np.array([0.2, 0.4, 0.6], np.float32))
        a.reset(seeds); b.reset(seeds)
        free = _frames(a, t, 2, noise=-1.0)
        _frames(b, t, 2, noise=-1.0)
        flux = np.asarray(t.p_wfs._fluxPerSub_list, np.float32)
        for e in range(E):
            tot = free[-1]["bincube"][e].sum(axis=1)
            assert np.allclose(tot, nph[e] * flux, rtol=1e-4), e           # noise-free: the counts are the flux exactly
        a.set_wfs_noise_env(noise=noise * 0 - 1.0, nphotons=nph)           # every environment noise-free
        a.reset(seeds)
        ref = _frames(a, t, 2, noise=-1.0)
        assert _same(free, ref)
        a.set_wfs_noise_env(noise=noise, nphotons=nph)
        a.reset(seeds)
        noisy = _frames(a, t, 1)
        assert not np.array_equal(noisy[0]["bincube"][0], ref[0]["bincube"][0])
        assert np.array_equal(noisy[0]["bincube"][2], ref[0]["bincube"][2])  # noise -1: no draw
        a.set_wfs_noise_env(None, None)
        a.set_gain_env(None)
        a.reset(seeds); b.reset(seeds)
        for noise_arg in (None, 3.0, -1.0):
            assert _same(_frames(a, t, 3, noise=noise_arg), _frames(b, t, 3, noise=noise_arg)), noise_arg
        assert a.wfs_noise_env is None and a.gain_env is None
        a.check_device(); b.check_device()
    finally:
        a.close(); b.close()


@pytest.mark.gpu
def test_noise_free_batch_keeps_the_specialised_kernel(torch):
    """Per-environment noise all -1 (per-environment photon counts too) and no kept image: the frame still runs the
    specialised-warp kernel; one noisy environment moves the frame to the fused kernel."""
    from torch.profiler import ProfilerActivity, profile
    from ao_marl_b200 import tables
    from ao_marl_b200.config import load_config_from_file
    from ao_marl_b200.lib import Simulator
    t = tables.build_static(load_config_from_file("production_sh_40x40_8m_3layers.py"))
    sim = Simulator(t, 2, rl=None)
    try:
        sim.reset(SEEDS[:2])
        sim.comp_wfs_image()                                  # module loads outside the trace

        def kernels(**kw):
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                sim.comp_wfs_image(**kw)
                torch.cuda.synchronize()
            return [e.name for e in prof.events() if "wfs_frame" in e.name]

        sim.set_wfs_noise_env(noise=[-1.0, -1.0], nphotons=_nph(t, np.array([5.0, 10.0])))
        names = kernels()
        assert any("wfs_frame_ws_kernel" in n for n in names) and not any("umma_kernel" in n for n in names), names
        sim.set_wfs_noise_env(noise=[-1.0, 3.0], nphotons=sim.wfs_nphotons_env)
        names = kernels()
        assert any("wfs_frame_umma_kernel" in n for n in names) and not any("ws_kernel" in n for n in names), names
        names = kernels(noise=-1.0)
        assert any("wfs_frame_ws_kernel" in n for n in names), names
        sim.check_device()
    finally:
        sim.close()


@pytest.mark.gpu
def test_reset_envs_with_new_conditions(system10, torch):
    """Environment 1 gets new (noise, magnitude, gain) and reset_envs([1]) after 4 steps: it then equals a fresh batch
    reset with them (plus the linear step that follows a reset); the other environments equal the run without the
    call."""
    from ao_marl_b200.lib import Simulator
    t, rl = system10
    E = 3
    seeds = SEEDS[:E].copy()
    noise0, nph0, gain0 = np.array([3.0, -1.0, 0.0], np.float32), _nph(t, np.array([9.0, 4.0, 6.0])), np.array([0.3, 0.7, 0.5], np.float32)
    noise1, nph1, gain1 = noise0.copy(), nph0.copy(), gain0.copy()
    noise1[1], nph1[1], gain1[1] = 3.0, _nph(t, 10.5), 0.25
    sim = Simulator(t, E, rl)

    def conditions(n, f, g):
        sim.set_wfs_noise_env(noise=n, nphotons=f)
        sim.set_gain(g)

    def steps(k):
        out = []
        for _ in range(k):
            sim.step(mode=0)
            out.append(_snap(sim, t, rl, False))
        return out

    try:
        conditions(noise0, nph0, gain0)
        sim.reset(seeds)
        steps(4)
        conditions(noise1, nph1, gain1)
        sim.reset_envs([1], np.array([555], np.int64))
        a = steps(6)
        conditions(noise0, nph0, gain0)
        sim.reset(seeds)
        steps(4)
        conditions(noise1, nph1, gain1)                      # environment 1 only changes: the others run on unchanged
        b = steps(6)
        seeds_c = seeds.copy()
        seeds_c[1] = 555
        sim.reset(seeds_c)
        sim.state_begin(); sim.move_atmos(); sim.comp_wfs_image(); sim.do_centroids(); sim.do_control(); sim.state_end()
        c = steps(5)
        sim.check_device()
    finally:
        sim.close()
    for i in range(6):
        for k in a[i]:
            assert np.array_equal(a[i][k][[0, 2]], b[i][k][[0, 2]]), (i, k)
    for i in range(1, 6):
        for k in a[i]:
            assert np.array_equal(a[i][k][1], c[i - 1][k][1]), (i, k)


@pytest.mark.gpu
def test_scalar_set_noise_reaches_the_step(system10, torch):
    """WfsB200.set_noise(0, 3.0) and set_gs_mag(0, 9.0) on the noise-free file make sim.step identical to a context
    created with noise 3 and the photons of magnitude 9; set_gs_mag with an [E] array equals per-environment photon
    counts, RtcB200.set_gain(0, [E]) per-environment gains, and a scalar drops them."""
    from ao_marl_b200.lib import Simulator
    from ao_marl_b200.supervisor.components import RtcB200, WfsB200
    t, rl = system10
    E = 3
    assert float(t.p_wfs.noise) < 0
    a = Simulator(t, E, rl)
    b = Simulator(_with_conditions(t, 3.0, _nph(t, 9.0), t.gain), E, rl)
    try:
        config = copy.deepcopy(t.config)                      # set_noise writes the parameter file's value
        wfs, rtc = WfsB200(a, config), RtcB200(a, config, t)
        wfs.set_noise(0, 3.0)
        wfs.set_gs_mag(0, 9.0)
        assert a.wfs_noise == 3.0 and a.wfs_nphotons == float(_nph(t, 9.0))

        def run(sim):
            sim.reset(SEEDS[:E])
            out = []
            for _ in range(5):
                sim.step(mode=0)
                out.append(_snap(sim, t, rl, False))
            return out

        assert _same(run(a), run(b))
        mags, gains = np.array([5.0, 9.0, 12.0]), np.array([0.2, 0.5, 0.9], np.float32)
        wfs.set_gs_mag(0, mags)
        rtc.set_gain(0, gains)
        assert np.array_equal(a.wfs_nphotons_env, _nph(t, mags)) and np.array_equal(rtc.d_control[0].gain, gains)
        assert a.wfs_noise_env is None
        pe = run(a)
        b.set_wfs_noise_env(noise=None, nphotons=_nph(t, mags))
        b.set_gain(gains)
        assert _same(pe, run(b))
        wfs.set_noise(0, [3.0, 0.0, -1.0])
        assert np.array_equal(a.wfs_noise_env, np.array([3.0, 0.0, -1.0], np.float32))
        assert np.array_equal(a.wfs_nphotons_env, _nph(t, mags))          # the photon counts stay
        wfs.set_noise(0, 3.0)
        wfs.set_gs_mag(0, 9.0)
        rtc.set_gain(0, float(t.gain))
        assert a.wfs_noise_env is None and a.wfs_nphotons_env is None and a.gain_env is None
        b.set_wfs_noise_env(None, None)
        b.set_gain_env(None)
        assert _same(run(a), run(b))
        a.check_device(); b.check_device()
    finally:
        a.close(); b.close()


@pytest.mark.gpu
def test_errors(system10, torch):
    """Wrong lengths raise ValueError in Python; non-finite values and photon counts <= 0 return AOM_ERR_INVALID and
    leave the state as it was; the round-1 sensor kernels refuse a frame that reads per-environment sensor values."""
    import ctypes
    from ao_marl_b200.lib import Simulator
    t, _ = system10
    E = 3
    sim = Simulator(t, E, rl=None)
    try:
        sim.reset(SEEDS[:E])
        for bad in ([1.0, 2.0], np.ones(E + 1), np.ones((E, 1))):
            with pytest.raises(ValueError):
                sim.set_wfs_noise_env(noise=bad)
            with pytest.raises(ValueError):
                sim.set_wfs_noise_env(nphotons=bad)
            with pytest.raises(ValueError):
                sim.set_gain(bad)
        with pytest.raises(ValueError, match="not finite"):
            sim.set_wfs_noise_env(noise=[0.0, np.nan, 3.0])
        with pytest.raises(ValueError, match="> 0"):
            sim.set_wfs_noise_env(noise=[0.0, 1.0, 3.0], nphotons=[100.0, 0.0, 50.0])
        with pytest.raises(ValueError, match="> 0"):
            sim.set_wfs_noise_env(nphotons=[100.0, -5.0, 50.0])
        with pytest.raises(ValueError, match="finite"):
            sim.set_wfs_noise_env(nphotons=[100.0, np.inf, 50.0])
        with pytest.raises(ValueError, match="not finite"):
            sim.set_gain([0.3, np.inf, 0.5])
        with pytest.raises(ValueError):
            sim.set_wfs_noise(3.0, 0.0)
        with pytest.raises(ValueError):
            sim.set_wfs_noise(np.nan)
        assert sim.wfs_noise_env is None and sim.wfs_nphotons_env is None and sim.gain_env is None
        # a refused call leaves the values in force as they were
        sim.set_wfs_noise_env(noise=[3.0, 0.0, -1.0])
        x = np.array([0.0, 1.0, 2.0], np.float32)
        y = np.array([1.0, np.nan, 2.0], np.float32)
        assert sim.lib.aom_set_wfs_noise_env(sim._ctx, x.ctypes.data_as(ctypes.c_void_p), y.ctypes.data_as(ctypes.c_void_p)) == -1
        sim.reset(SEEDS[:E])
        sim.comp_wfs_image(keep_image=True)
        cube = sim.buffer("BINCUBE").view(E, t.p_wfs._nvalid, 256).cpu().numpy()
        flux = np.asarray(t.p_wfs._fluxPerSub_list, np.float32)
        assert np.array_equal(cube[1], np.round(cube[1]))                  # photon noise only: whole counts
        assert np.allclose(cube[2].sum(axis=1), sim.wfs_nphotons * flux, rtol=1e-4)   # no noise, common photon count
        sim.set_wfs_noise_env(None, None)
        for path in ("tensor", "tensor_fast", "tensor_reg"):
            sim.set_wfs_path(path)
            sim.comp_wfs_image(noise=3.0)                                   # uniform: still served
            sim.set_wfs_noise_env(noise=[3.0, 0.0, -1.0])
            with pytest.raises(RuntimeError, match="per-environment sensor"):
                sim.comp_wfs_image(noise=3.0)
            sim.comp_wfs_image(noise=-1.0)                                  # noise-free frame: reads none of them
            sim.set_wfs_noise_env(nphotons=[100.0, 200.0, 300.0])
            with pytest.raises(RuntimeError, match="per-environment sensor"):
                sim.comp_wfs_image(noise=-1.0)
            sim.set_wfs_noise_env(None, None)
        sim.set_wfs_path(sim.DEFAULT_WFS_PATH)
        sim.check_device()
    finally:
        sim.close()
