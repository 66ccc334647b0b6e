"""Reference of the controller's three-row delay line (aom_apply_control, include/aomarl.h) for the tests: sutra's
comp_voltage, volts = a com + b com1 + c com2, for a delay d in [0, 2] frames, in float32 with the exact expression of the
library.  `DelayOracleEnv` is the numpy closed-loop oracle (oracle/loop.py, delays 0 and 1) with this line in place of its
two-row one."""
import numpy as np

from oracle import loop

F32 = np.float32


def fmaf(a, b, c):
    """float32 fmaf(a, b, c) with one rounding, elementwise.  a * b is exact in float64; the sum is rounded to odd in
    float64 (TwoSum error, then the last bit forced to 1 when inexact), and rounding that to float32 is then correct:
    float64 carries more than two bits beyond float32's 24."""
    a, b, c = (np.asarray(x, F32).astype(np.float64) for x in (a, b, c))
    p = a * b
    s = p + c
    bb = s - p
    err = (p - (s - bb)) + (c - bb)
    bits = np.atleast_1d(s).view(np.int64).copy()
    err = np.atleast_1d(err)
    sign = np.where(np.atleast_1d(s) < 0, -1, 1)
    fix = (err != 0) & ((bits & 1) == 0)
    bits[fix] += np.where(err[fix] > 0, 1, -1) * sign[fix]
    with np.errstate(invalid="ignore", over="ignore"):
        out = bits.view(np.float64).astype(F32)
    return out.reshape(np.shape(s)) if np.ndim(s) else out[0]


def delay_line(com, com1, com2, d):
    """(volts, new com1, new com2) of one aom_apply_control with delay d: an integer delay copies its row, a fractional
    one is fmaf(f, c_(k+1), (1 - f) * c_k) with k = floor(d), f = d - k."""
    d = F32(d)
    assert 0.0 <= d <= 2.0
    rows = [np.asarray(com, F32), np.asarray(com1, F32), np.asarray(com2, F32)]
    k = int(np.floor(d))
    f = F32(d - F32(k))
    if f == 0:
        volts = rows[k].copy()
    else:
        volts = fmaf(f, rows[k + 1], (F32(1) - f) * rows[k])
    return volts, rows[0].copy(), rows[1].copy()


class DelayOracleEnv(loop.OracleEnv):
    """OracleEnv whose apply_control is the three-row delay line with a real delay in [0, 2] (`delay`)."""

    def __init__(self, tab, cmat, Btt=None, P=None, rl=None, seed=1234, delay=1.0):
        super().__init__(tab, cmat, Btt, P, rl, seed)
        self.delay = F32(delay)

    def _clear(self):
        super()._clear()
        self.com2 = np.zeros(self.tab["nactu"], F32)

    def apply_control(self):
        self.volts, self.com1, self.com2 = delay_line(self.com, self.com1, self.com2, self.delay)
