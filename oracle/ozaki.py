"""TEST INFRASTRUCTURE (oracle) -- never imported by the product path.

numpy emulation, bit for bit, of the exact integer contraction of ao_marl_b200/csrc/extrude_i8.cuh (DESIGN.md section
4.2): the screen extrusion (EPI 0) and the controller products (EPI 1 / 2 / 3).

* Input rows: a power-of-two row exponent ev (|x|max 2^-ev in [0.5, 1)) and six signed 7-bit digits per element,
  x 2^-ev = q0 2^-6 + q1 2^-13 + ... + q5 2^-41 + (remainder <= 2^-42).  The products cut float32 rows with float32
  arithmetic (oz_slice_rows_kernel), the extrusion cuts its float64 inputs in float64 (oz_gather_slice_kernel).
* Operator rows: the same six digits and exponent ea, in float64 (oz_slice_operator).
* Level sums: the digit pairs with s + t = g share one integer accumulator; pairs with g < LEV are kept (6 for the
  extrusion, 5 for the products).  They run here as float64 matrix products of digit planes: every partial sum is an
  integer below 2^53, so BLAS computes them exactly, in any order.
* Epilogue: acc = (((a_{L-1} 2^-7 + a_{L-2}) 2^-7 + ...) 2^-7 + a_0) in float64 -- the multiply by 2^-7 is exact, so each
  step is the kernel's fma -- then the scale 2^(ev + ea - 12) and one cast to float32.  EPI 0 adds zref in float64
  before that cast; EPI 2 / 3 negate, and the integrator is float32 fmaf(g, err, com).
"""
import numpy as np

from . import rng

F32, F64 = np.float32, np.float64

SLICES = 6                  # OZ_SLICES: digits of an input row
SLICES_B = 6                # OZ_SLICES_B: digits of an operator row
LEVELS = 6                  # OZ_LEVELS: extrusion keeps s + t <= 5
LEVELS_PRODUCT = 5          # OZ_LEVELS_PRODUCT: controller products keep s + t <= 4
BM, BN, BK = 128, 80, 32    # OZ_BM / OZ_BN / OZ_BK
EV_NONFINITE = 0x40000000   # OZ_EV_NONFINITE: row exponent of an input row holding a NaN or an infinity


def row_exponent(amax):
    """oz_exponent: e with amax 2^-e in [0.5, 1), 0 for amax == 0 (vectorised, float64 input)."""
    amax = np.asarray(amax, F64)
    with np.errstate(invalid="ignore"):
        _, e = np.frexp(np.where(amax > 0, amax, 1.0))
    return np.where(amax > 0, e, 0).astype(np.int64)


def digits(x, scale, ns=SLICES_B):
    """oz_digits: ns signed 7-bit digits of x * scale in float64 -> [ns, *x.shape] (integers, held as float64 for the
    level sums)."""
    t = np.asarray(x, F64) * scale * 64.0
    q = np.empty((ns,) + t.shape, F64)
    for s in range(ns):
        r = np.rint(t)
        q[s] = r
        t = (t - r) * 128.0
    return q


def digits_f32(x, scale, ns=SLICES):
    """oz_digits_f32: the same digits of float32 values, every operation in float32."""
    t = np.asarray(x, F32) * F32(scale) * F32(64.0)
    q = np.empty((ns,) + t.shape, F64)
    with np.errstate(invalid="ignore"):
        for s in range(ns):
            r = np.rint(t)
            q[s] = np.where(np.isfinite(r), r, 0)
            t = (t - r) * F32(128.0)
    return q


def pow2_f32(e):
    """2^e as float32 for |e| <= 126."""
    return ((np.asarray(e, np.int64) + 127) << 23).astype(np.int32).view(F32)


def row_digits_f32(X):
    """oz_slice_rows_kernel on float32 rows X [E, K]: digits [SLICES, E, K] and ev [E] (EV_NONFINITE for a row with a NaN
    or an infinity; its digits are zero here and unused by the epilogue).  The kernel scales by 2^-ev as two float32 factors
    2^-(ev >> 1) and 2^-(ev - (ev >> 1)); both products are exact, so the digits are those of x 2^-ev."""
    X = np.asarray(X, F32)
    fin = np.isfinite(X)
    bad = ~fin.all(axis=1)
    a = np.where(fin, np.abs(X), F32(0))
    ex = row_exponent(a.max(axis=1).astype(F64) if X.shape[1] else np.zeros(X.shape[0]))
    ex[bad] = 0
    h = ex >> 1
    xs = np.where(fin, X, F32(0)) * pow2_f32(-h)[:, None]
    q = digits_f32(xs, pow2_f32(-(ex - h))[:, None], SLICES)
    return q, np.where(bad, EV_NONFINITE, ex)


def operator_digits(W):
    """oz_slice_operator on a float32 operator W [rows, K]: digits [SLICES_B, rows, K] and ea [rows]."""
    W64 = np.asarray(W, F32).astype(F64)
    ea = row_exponent(np.abs(W64).max(axis=1) if W64.shape[1] else np.zeros(W64.shape[0]))
    return digits(W64, np.ldexp(1.0, -ea)[:, None], SLICES_B), ea


def tile_planes(q, tile_rows, kb=None):
    """Digit planes [S, rows, K] in the kernel's tile layout: uint8 [NT][KB][S][tile_rows * 32], 8-row x 16-byte core
    matrices (oz_tile_offset).  Rows beyond `rows` and columns beyond K are zero."""
    S, R, K = q.shape
    NT = -(-R // tile_rows)
    KB = -(-K // BK) if kb is None else kb
    out = np.zeros((NT, KB, S, tile_rows * BK), np.uint8)
    r, k = np.arange(R), np.arange(K)
    rr, kk = r % tile_rows, k % BK
    off = (rr[:, None] >> 3) * 256 + (kk[None, :] >> 4) * 128 + (rr[:, None] & 7) * 16 + (kk[None, :] & 15)
    nt, kbi = np.broadcast_to((r // tile_rows)[:, None], off.shape), np.broadcast_to((k // BK)[None, :], off.shape)
    for s in range(S):
        out[nt, kbi, s, off] = q[s].astype(np.int8).view(np.uint8)
    return out


def level_sums(qa, qb, lev):
    """Integer accumulators [lev, E, N]: acc_g = sum over s + t = g of qa_s . qb_t^T (exact in float64)."""
    E, N = qa.shape[1], qb.shape[1]
    acc = np.zeros((lev, E, N), F64)
    for g in range(lev):
        for s in range(qa.shape[0]):
            t = g - s
            if 0 <= t < qb.shape[0]:
                acc[g] += np.asarray(qa[s], F64) @ np.asarray(qb[t], F64).T
    return acc


def combine(acc):
    """The epilogue's float64 chain: a_{L-1}, then a * 2^-7 + a_g for g = L-2 .. 0 (each step one rounding, as fma)."""
    a = acc[-1].copy()
    for g in range(acc.shape[0] - 2, -1, -1):
        a = a * 0.0078125 + acc[g]
    return a


def product(X, W, lev=LEVELS_PRODUCT):
    """X [E, K] . W[N, K]^T as oz_gemm_kernel<1> computes it: float32 [E, N] (NaN rows for non-finite input rows)."""
    qa, ev = row_digits_f32(X)
    qb, ea = operator_digits(W)
    a = combine(level_sums(qa, qb, lev))
    bad = ev == EV_NONFINITE
    e = np.where(bad, 0, ev)[:, None] + ea[None, :] - 12
    out = np.ldexp(a, e.astype(np.int32)).astype(F32)
    out[bad] = np.nan
    return out


def fmaf(a, b, c):
    """float32 fmaf(a, b, c) with a single rounding.  a b is exact in float64; the float64 sum is rounded to odd (two-sum,
    then a step to the odd neighbour when inexact) so that the final cast to float32 rounds once, correctly."""
    a, b, c = (np.asarray(v, F32).astype(F64) for v in (a, b, c))
    p = a * b
    s = p + c
    return round_to_f32(s, _two_sum_err(p, c, s))


def _two_sum_err(p, c, s):
    with np.errstate(invalid="ignore"):
        bb = s - p
        return (p - (s - bb)) + (c - bb)


def round_to_f32(s, err):
    """Correctly rounded float32 of s + err, where s = fl64(s + err) and err is the exact residual (as from a two-sum or
    math.fsum): round to odd in float64, then cast."""
    s, err = np.asarray(s, F64), np.asarray(err, F64)
    with np.errstate(invalid="ignore"):
        even = (s.view(np.int64) & 1) == 0
        nudge = np.isfinite(s) & (err != 0) & even
        s = np.where(nudge, np.nextafter(s, np.copysign(np.inf, err)), s)
    return s.astype(F32)


def integrate(err, com, gain):
    """EPI 2 / 3 with the loop closed: com + g err in float32 fmaf; gain a scalar or one value per row."""
    g = np.broadcast_to(np.asarray(gain, F32).reshape(-1, 1) if np.ndim(gain) else np.asarray(gain, F32), err.shape)
    return fmaf(g, err, com)


# ---------------------------------------------------------------------------------------------------------------------
# EPI 0: one screen extrusion
def extrusion_inputs(s, istx, amp, noise):
    """The gather of one +x extrusion on the (already transposed / mirrored) float32 screen s [N, N]: float64 inputs
    v = [stencil pixels - zref | noise amp] and zref (float32)."""
    n = s.shape[0]
    zr = s[0, n - 1]
    z = s.reshape(-1)[np.asarray(istx)].astype(F64) - F64(zr)
    return np.concatenate([z, np.asarray(noise, F32).astype(F64) * F64(F32(amp))]), zr


def extrusion_column(v, zr, op):
    """New column of one extrusion: v float64 [E, K], zr float32 [E], op = operator_digits(AB) -> float32 [E, N]."""
    v = np.atleast_2d(v)
    ev = row_exponent(np.abs(v).max(axis=1))
    qa = digits(v, np.ldexp(1.0, -ev)[:, None], SLICES)
    qb, ea = op
    a = combine(level_sums(qa, qb, LEVELS))
    return (np.ldexp(a, (ev[:, None] + ea[None, :] - 12).astype(np.int32)) + np.asarray(zr, F32).astype(F64)[:, None]).astype(F32)


def extrude(screens, op, istx, amp, noises, axis, sign):
    """oracle/aoframe.extrude with the integer contraction behind the new column, for one screen [N, N] or a stack
    [B, N, N] (noises [N] or [B, N]): the x case on the transposed (axis 1) and / or 180-degree rotated (sign < 0)
    screen."""
    s = np.asarray(screens)
    one = s.ndim == 2
    s, noises = np.atleast_3d(s[None] if one else s), np.atleast_2d(noises)
    if axis == 1:
        s = s.swapaxes(1, 2)
    if sign < 0:
        s = s[:, ::-1, ::-1]
    s = np.ascontiguousarray(s)
    vz = [extrusion_inputs(s[b], istx, amp, noises[b]) for b in range(s.shape[0])]
    col = extrusion_column(np.stack([v for v, _ in vz]), np.array([z for _, z in vz], F32), op)
    out = np.empty_like(s)
    out[:, :, :-1] = s[:, :, 1:]
    out[:, :, -1] = col
    if sign < 0:
        out = out[:, ::-1, ::-1]
    if axis == 1:
        out = out.swapaxes(1, 2)
    out = np.ascontiguousarray(out)
    return out[0] if one else out


def extrusion_noise(seed, layer, count, n):
    """Innovations of extrusion `count` of `layer` (the kernel's Philox stream, oracle/rng.py)."""
    return rng.atmos_noise(int(seed), int(layer), int(count), int(n))
