"""The per-episode conditions (aom_condition: amplitude, wind x / y, sensor noise, photon count, integrator gain) live in
one store of the context: aom_get_condition reads back what the setters and aom_load_envs left there, and the Python
properties (Simulator.wfs_noise / wfs_nphotons / gain / *_env, rtc.d_control[0].gain) read it instead of mirroring."""
import copy
import ctypes

import numpy as np
import pytest

E = 4
NAMES = ["AMP", "WIND_X", "WIND_Y", "NOISE", "NPHOTONS", "GAIN"]


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _get(sim, name, layer=0):
    """(common value, per-environment values in force?, each environment's value) through aom_get_condition"""
    from ao_marl_b200.lib import COND
    common, per_env, values = ctypes.c_float(), ctypes.c_int(), np.full(sim.n_env, np.nan, np.float32)
    rc = sim.lib.aom_get_condition(sim._ctx, COND[name], layer, ctypes.byref(common), values.ctypes.data_as(ctypes.c_void_p),
                                   ctypes.byref(per_env))
    assert rc == 0, sim.lib.aom_last_error(sim._ctx)
    return np.float32(common.value), bool(per_env.value), values


def _state(sim):
    return {(k, l): _get(sim, k, l) for k in NAMES for l in range(sim.cfg.n_layers if k in NAMES[:3] else 1)}


def _same_state(x, y):
    return x.keys() == y.keys() and all(x[k][0] == y[k][0] and x[k][1] == y[k][1] and np.array_equal(x[k][2], y[k][2])
                                        for k in x)


def _set_common(sim, name, v):
    if name in NAMES[:3]:
        w = {k: float(_get(sim, k)[0]) for k in NAMES[:3]}
        w[name] = v
        sim.set_layer(0, w["WIND_X"], w["WIND_Y"], w["AMP"])
    elif name == "NOISE":
        sim.set_wfs_noise(v)
    elif name == "NPHOTONS":
        sim.set_wfs_noise(sim.wfs_noise, v)
    else:
        sim.set_gain(v)


def _set_env(sim, name, a):
    if name == "AMP":
        sim.set_layer_amp(0, a)
    elif name in ("WIND_X", "WIND_Y"):
        other = None if a is None else _get(sim, "WIND_Y" if name == "WIND_X" else "WIND_X")[2]
        sim.set_layer_wind(0, *((a, other) if name == "WIND_X" else (other, a)))
    elif name == "NOISE":
        sim.set_wfs_noise_env(noise=a, nphotons=sim.wfs_nphotons_env)
    elif name == "NPHOTONS":
        sim.set_wfs_noise_env(noise=sim.wfs_noise_env, nphotons=a)
    else:
        sim.set_gain_env(a)


def _values(name, c):
    """(new common value, per-environment values) of a condition whose common value is c"""
    return {"AMP": (c * 1.25, c * np.array([1.0, 1.5, 0.5, 2.0])), "WIND_X": (c + 0.125, c + np.array([0.0, 0.25, -0.25, 0.1])),
            "WIND_Y": (c - 0.125, c + np.array([0.1, -0.25, 0.25, 0.0])), "NOISE": (2.0, np.array([-1.0, 0.0, 3.0, 1.0])),
            "NPHOTONS": (c * 0.75, c * np.array([1.0, 0.5, 2.0, 4.0])), "GAIN": (0.45, np.array([0.2, 0.4, 0.6, 0.8]))}[name]


@pytest.mark.gpu
def test_read_back_what_was_set(static10, torch):
    """Each condition: the configured common value, a new common value, per-environment values (the common value set
    while they are in force changes only the common value), and back to the common value."""
    from ao_marl_b200.lib import COND, Simulator
    t = static10
    sim = Simulator(t, E)
    try:
        sim.reset(np.arange(E, dtype=np.int64) + 7)
        cfg = {"AMP": sim.cfg.amp[0], "WIND_X": sim.cfg.deltax[0], "WIND_Y": sim.cfg.deltay[0], "NOISE": sim.cfg.noise,
               "NPHOTONS": sim.cfg.nphotons, "GAIN": sim.cfg.gain}
        for name in NAMES:
            c0 = np.float32(cfg[name])
            c, pe, v = _get(sim, name)
            assert c == c0 and not pe and np.all(v == c0), name
            common, env = _values(name, float(c0))
            env = env.astype(np.float32)
            _set_common(sim, name, common)
            c, pe, v = _get(sim, name)
            assert c == np.float32(common) and not pe and np.all(v == np.float32(common)), name
            _set_env(sim, name, env)
            c, pe, v = _get(sim, name)
            assert c == np.float32(common) and pe and np.array_equal(v, env), name
            _set_common(sim, name, float(c0))
            c, pe, v = _get(sim, name)
            assert c == c0 and pe and np.array_equal(v, env), name
            _set_env(sim, name, None)
            c, pe, v = _get(sim, name)
            assert c == c0 and not pe and np.all(v == c0), name
        assert sim.wfs_noise == np.float32(cfg["NOISE"]) and sim.gain == np.float32(cfg["GAIN"])
        assert sim.wfs_noise_env is None and sim.wfs_nphotons_env is None and sim.gain_env is None
        # NULL outputs are allowed; an unknown condition or a layer out of range is refused
        assert sim.lib.aom_get_condition(sim._ctx, COND["GAIN"], 0, None, None, None) == 0
        assert sim.lib.aom_get_condition(sim._ctx, len(NAMES), 0, None, None, None) == -1
        assert sim.lib.aom_get_condition(sim._ctx, COND["AMP"], sim.cfg.n_layers, None, None, None) == -1
        assert sim.lib.aom_get_condition(sim._ctx, COND["GAIN"], 1, None, None, None) == -1
        sim.check_device()
    finally:
        sim.close()


@pytest.mark.gpu
def test_loaded_conditions_read_back(static10, torch):
    """copy_envs / load_envs of records with another gain, noise and amplitude: the read-back holds the loaded values in
    the loaded slots and every other environment's value as before, and rtc.d_control[0].gain shows the same gains."""
    from ao_marl_b200.lib import Simulator
    from ao_marl_b200.supervisor.components import RtcB200
    t = static10
    a, b = Simulator(t, E), Simulator(t, E)
    try:
        rtc = RtcB200(a, copy.deepcopy(t.config), t)
        for sim in (a, b):
            sim.reset(np.arange(E, dtype=np.int64) + 11)
        amp0 = np.float32(a.cfg.amp[0])
        a_amp = (amp0 * np.array([1.0, 1.25, 1.5, 1.75])).astype(np.float32)
        a.set_layer_amp(0, a_amp)
        rtc.set_gain(0, 0.5)
        b_amp = (amp0 * np.array([2.0, 2.5, 3.0, 3.5])).astype(np.float32)
        b.set_layer_amp(0, b_amp)
        b_noise = np.array([3.0, -1.0, 0.0, 5.0], np.float32)
        b.set_wfs_noise_env(noise=b_noise)
        b.set_gain(0.3)

        a.load_envs([2, 0], b.save_envs([0, 3]))
        gain = np.array([0.3, 0.5, 0.3, 0.5], np.float32)
        noise = np.full(E, np.float32(a.cfg.noise), np.float32)
        noise[[2, 0]] = b_noise[[0, 3]]
        amp = a_amp.copy()
        amp[[2, 0]] = b_amp[[0, 3]]
        assert np.array_equal(_get(a, "AMP")[2], amp)
        assert np.array_equal(a.wfs_noise_env, noise) and a.wfs_nphotons_env is None
        assert np.array_equal(a.gain_env, gain) and np.array_equal(rtc.d_control[0].gain, gain)
        assert a.gain == np.float32(0.5)

        a.copy_envs([2], [1])
        gain[1], noise[1], amp[1] = gain[2], noise[2], amp[2]
        assert np.array_equal(_get(a, "AMP")[2], amp)
        assert np.array_equal(a.wfs_noise_env, noise)
        assert np.array_equal(a.gain_env, gain) and np.array_equal(rtc.d_control[0].gain, gain)
        rtc.set_gain(0, 0.5)
        assert rtc.d_control[0].gain == np.float32(0.5) and a.gain_env is None
        a.check_device()
        b.check_device()
    finally:
        a.close()
        b.close()


@pytest.mark.gpu
def test_non_finite_values_change_nothing(static10, torch):
    """A NaN amplitude (common or per environment), a non-finite common wind or gain, or a NaN in one array of a
    per-environment wind: AOM_ERR_INVALID (ValueError) and every condition reads back as before."""
    from ao_marl_b200.lib import Simulator
    t = static10
    sim = Simulator(t, E)
    try:
        sim.reset(np.arange(E, dtype=np.int64) + 3)
        sim.set_layer_amp(0, np.float32(sim.cfg.amp[0]) * np.array([1.0, 2.0, 3.0, 4.0], np.float32))
        sim.set_gain_env([0.1, 0.2, 0.3, 0.4])
        before = _state(sim)
        dx, dy, amp = float(sim.cfg.deltax[0]), float(sim.cfg.deltay[0]), float(sim.cfg.amp[0])
        bad = [lambda: sim.set_layer_amp(0, [amp, np.nan, amp, amp]),
               lambda: sim.set_layer(0, dx, dy, np.nan),
               lambda: sim.set_layer(0, np.inf, dy, amp),
               lambda: sim.set_layer(0, dx, np.nan, amp),
               lambda: sim.set_gain(np.nan),
               lambda: sim.set_gain(-np.inf),
               lambda: sim.set_layer_wind(0, [dx] * E, [dy, dy, np.nan, dy])]
        for i, call in enumerate(bad):
            with pytest.raises(ValueError, match="not finite"):
                call()
            assert _same_state(_state(sim), before), i
        sim.check_device()
    finally:
        sim.close()
