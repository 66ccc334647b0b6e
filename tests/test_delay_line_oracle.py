"""The reference delay line of the tests (tests/delay_line_ref.py, the oracle's apply_control for delays in [0, 2]): impulse
timing for whole-frame delays, the fractional blend bit for bit against the C library's fmaf, integer delays that select
a row, and ROKET's refusal of delays its loop filter does not model."""
import ctypes
import ctypes.util
import types

import numpy as np
import pytest

from delay_line_ref import DelayOracleEnv, delay_line, fmaf

F32 = np.float32


def _libm_fmaf():
    name = ctypes.util.find_library("m")
    if not name:
        pytest.skip("no C math library")
    f = ctypes.CDLL(name).fmaf
    f.restype = ctypes.c_float
    f.argtypes = [ctypes.c_float] * 3
    return f


def _bits(x):
    return np.asarray(x, F32).view(np.uint32)


def test_fmaf_is_correctly_rounded():
    """fmaf of the reference equals the C library's fmaf bit for bit, on random operands and on ties and cancellations
    where a product rounded first, or a sum rounded twice, would differ."""
    cf = _libm_fmaf()
    r = np.random.default_rng(7)
    a = (r.standard_normal(4000) * 10.0 ** r.integers(-6, 6, 4000)).astype(F32)
    b = (r.standard_normal(4000) * 10.0 ** r.integers(-6, 6, 4000)).astype(F32)
    c = (r.standard_normal(4000) * 10.0 ** r.integers(-12, 12, 4000)).astype(F32)
    eps = np.finfo(F32).eps
    # a product just off a float32, minus its rounded value: exact cancellation residues; and the 0.5 steps of d
    edge_a = np.array([1 + eps, 1 + 2 * eps, 0.5, 0.5, 1 - eps / 2, 3.0, 0.1], F32)
    edge_b = np.array([1 - eps, 1 + eps, 1 + eps, -(1 + eps), 1 + eps, 1 / 3, 0.3], F32)
    edge_c = -(edge_a * edge_b).astype(F32)
    a, b, c = np.concatenate([a, edge_a]), np.concatenate([b, edge_b]), np.concatenate([c, edge_c])
    want = np.array([cf(float(x), float(y), float(z)) for x, y, z in zip(a, b, c)], F32)
    assert np.array_equal(_bits(fmaf(a, b, c)), _bits(want))
    assert _bits(fmaf(a[3], b[3], c[3])) == _bits(want[3])            # scalars too


def test_fractional_blend_is_the_float32_expression():
    """Delays 0.25, 0.5, 1.5, 1.75: volts = fmaf(f, c_(k+1), (1 - f) * c_k) in float32, bit for bit; d = 1.5 is the mean
    of com1 and com2 where that is exact."""
    cf = _libm_fmaf()
    r = np.random.default_rng(3)
    c0, c1, c2 = (r.standard_normal(257).astype(F32) for _ in range(3))
    for d in (0.25, 0.5, 1.5, 1.75):
        k, f = int(d), F32(d - int(d))
        lo, hi = (c0, c1) if k == 0 else (c1, c2)
        p = ((F32(1) - f) * lo).astype(F32)
        want = np.array([cf(float(f), float(h), float(q)) for h, q in zip(hi, p)], F32)
        volts, n1, n2 = delay_line(c0, c1, c2, d)
        assert volts.dtype == F32 and np.array_equal(_bits(volts), _bits(want)), d
        assert np.array_equal(n1, c0) and np.array_equal(n2, c1)
    even = np.array([1.0, -2.0, 0.5], F32)
    assert np.array_equal(delay_line(even, even * 3, even * 5, 1.5)[0], even * 4)


def test_impulse_timing():
    """An impulse in com at call 0 reaches volts at call d for d = 0, 1, 2; d = 0.5 and 1.5 split it over two calls."""
    def run(d, n=5):
        c1 = c2 = np.zeros(1, F32)
        out = []
        for i in range(n):
            v, c1, c2 = delay_line(np.array([1.0 if i == 0 else 0.0], F32), c1, c2, d)
            out.append(float(v[0]))
        return out
    assert run(0) == [1, 0, 0, 0, 0]
    assert run(1) == [0, 1, 0, 0, 0]
    assert run(2) == [0, 0, 1, 0, 0]
    assert run(0.5) == [0.5, 0.5, 0, 0, 0]
    assert run(1.5) == [0, 0.5, 0.5, 0, 0]
    assert run(0.25) == [0.75, 0.25, 0, 0, 0]


def test_integer_delays_select_a_row():
    """A NaN in a row the delay does not read stays out of volts (0 * NaN would not); a fractional delay reads both."""
    nan, one = np.array([np.nan], F32), np.array([1.0], F32)
    for d, rows, finite in ((0, (one, nan, nan), True), (1, (nan, one, nan), True), (2, (nan, nan, one), True),
                            (0.5, (one, nan, one), False), (1.5, (nan, nan, one), False), (1.5, (nan, one, one), True)):
        v = delay_line(*rows, d)[0]
        assert bool(np.isfinite(v[0])) == finite, d


def test_oracle_env_uses_the_three_row_line():
    """DelayOracleEnv's apply_control shifts com -> com1 -> com2 and selects / blends by its delay."""
    env = DelayOracleEnv.__new__(DelayOracleEnv)
    env.tab = {"nactu": 2, "nslopes": 1}
    env.rl = None
    env._clear()
    env.delay = F32(2.0)
    seen = []
    for i in range(4):
        env.com = np.array([i + 1, -(i + 1)], F32)
        env.apply_control()
        seen.append(env.volts.copy())
    assert [float(v[0]) for v in seen] == [0, 0, 1, 2]
    assert np.array_equal(env.com1, [4, -4]) and np.array_equal(env.com2, [3, -3])


def test_roket_refuses_per_environment_and_fractional_delays():
    """ROKET's loop filter delays commands by whole frames, one delay for the batch: it raises for per-environment or
    fractional delays and returns the common whole-frame delay otherwise."""
    from ao_marl_b200.guardians.roket import Roket
    stub = types.SimpleNamespace(sim=types.SimpleNamespace(gain_env=None, controller_env=None, delay=1.0,
                                                           delay_env=np.array([0.0, 2.0], np.float32)))
    stub._common_gain = lambda: Roket._common_gain(stub)
    stub._one_controller = lambda: Roket._one_controller(stub)
    stub._common_delay = lambda: Roket._common_delay(stub)
    with pytest.raises(NotImplementedError, match="one delay"):
        Roket._common_delay(stub)
    with pytest.raises(NotImplementedError, match="one delay"):
        Roket.do_error_breakdown(stub)
    stub.sim.delay_env = None
    stub.sim.delay = 1.5
    with pytest.raises(NotImplementedError, match="whole frames"):
        Roket._common_delay(stub)
    for d in (0.0, 1.0, 2.0):
        stub.sim.delay = d
        assert Roket._common_delay(stub) == int(d)
