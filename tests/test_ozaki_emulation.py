"""The digit code of the exact integer contraction (extrude_i8_digits.h, built for the host) against its numpy emulation
(oracle/ozaki.py), and the emulation against exact arithmetic and against the float64 oracle.  No GPU needed: the GPU
kernels are compared bit for bit with the same emulation in tests/test_int_contractions.py."""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest

from oracle import aoframe as af
from oracle import ozaki as oz

HERE = os.path.dirname(os.path.abspath(__file__))
F32, F64 = np.float32, np.float64


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    """The CPU harness built fresh from the current headers (a cached build could predate a header change)."""
    out = str(tmp_path_factory.mktemp("harness") / "libharness.so")
    subprocess.run(["g++", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-o", out,
                    os.path.join(HERE, "cpu_kernels", "harness.cpp")], check=True)
    return ctypes.CDLL(out)


def P(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def test_constants_and_tile_offset(harness):
    c = np.zeros(10, np.int32)
    harness.h_oz_constants(P(c))
    assert list(c) == [oz.SLICES, oz.SLICES_B, oz.LEVELS, oz.LEVELS_PRODUCT, oz.BM, oz.BN, oz.BK, oz.BM * oz.BK,
                       oz.BN * oz.BK, oz.EV_NONFINITE]
    seen = set()
    for r in range(oz.BM):
        for k in range(oz.BK):
            o = harness.h_oz_tile_offset(r, k)
            assert o == (r >> 3) * 256 + (k >> 4) * 128 + (r & 7) * 16 + (k & 15)
            seen.add(o)
    assert seen == set(range(oz.BM * oz.BK))          # a permutation of one tile


def adversarial_rows(K, r):
    """float32 rows [n, K] at the edges of the digit code."""
    rows = [np.zeros(K, F32)]                                            # all zero
    one = np.zeros(K, F32); one[K // 2] = F32(-3.75); rows.append(one)   # a single nonzero element
    for k in (0, 5, -7):                                                 # maximum exactly +-2^k (mantissa 0.5: ev = k + 1)
        x = (r.uniform(-1, 1, K) * 2.0 ** k).astype(F32); x[r.integers(K)] = F32((-1) ** k * 2.0 ** k); rows.append(x)
    x = r.uniform(-1, 1, K).astype(F32); x[0] = 1.0                      # elements 2^-17 and 2^-30 below the maximum
    x[K // 3] = F32(2.0 ** -17 * 1.2345); x[(2 * K) // 3] = F32(-2.0 ** -30 * 1.75); x[-1] = F32(2.0 ** -40); rows.append(x)
    x = (r.uniform(-1, 1, K) * 1e-6).astype(F32); x[r.integers(K)] = F32(3.0e3); rows.append(x)   # one outlier
    x = (r.uniform(-1, 1, K) * 2.0 ** -140).astype(F32); rows.append(x)  # subnormal maximum
    rows.append((r.uniform(-1, 1, K) * 2.0 ** 126 * 1.5).astype(F32))   # maximum >= 2^126
    x = r.standard_normal(K).astype(F32); h = K // 2; x[h:2 * h] = -x[:h]; rows.append(x)    # +a / -a pairs
    rows.append(r.standard_normal(K).astype(F32) * F32(1e-3))
    return np.stack(rows)


KS = [1, 31, 32, 33, 87, 128, 513, 2400]
ROWS = [1, 79, 80, 81, 90, 1286]


@pytest.mark.parametrize("K", KS)
def test_operator_slicing_matches_emulation(harness, K):
    """oz_slice_operator (the host slicing aom_set_table runs) gives the emulator's digit planes, byte for byte in the
    kernel's tile layout, and its row exponents, for random and adversarial operators of every row count."""
    r = np.random.default_rng(K)
    for rows in ROWS:
        W = (r.standard_normal((rows, K)) * np.exp(r.uniform(-8, 8, (rows, 1)))).astype(F32)
        adv = adversarial_rows(K, r)
        W[:min(rows, len(adv))] = adv[:rows]
        ld = K + 3
        Wp = np.zeros((rows, ld), F32); Wp[:, :K] = W; Wp[:, K:] = np.nan     # pad columns are never read
        KB, NT = -(-K // oz.BK), -(-rows // oz.BN)
        planes = np.zeros(NT * KB * oz.SLICES_B * oz.BN * oz.BK, np.uint8)
        ea = np.full(NT * oz.BN, -99, np.int32)
        harness.h_oz_slice_operator(P(Wp), rows, ld, K, KB, NT, P(planes), P(ea))
        q, ea_ref = oz.operator_digits(W)
        assert np.array_equal(ea[:rows], ea_ref) and not ea[rows:].any(), (rows, K)
        assert np.array_equal(planes, oz.tile_planes(q, oz.BN).reshape(-1)), (rows, K)
        assert harness.h_oz_operator_finite(P(Wp), rows, ld, K) == 1
        Wp[rows // 2, K - 1] = np.inf
        assert harness.h_oz_operator_finite(P(Wp), rows, ld, K) == 0


def test_digits_match_emulation(harness):
    """oz_digits_f32 (the products' input rows) and oz_digits (extrusion inputs) digit for digit, and oz_exponent, on the
    values and scales the kernels use -- including the two-factor scale of subnormal and huge row maxima."""
    r = np.random.default_rng(7)
    X = np.concatenate([adversarial_rows(K, r) for K in (33, 128, 513)], axis=1)
    ex = oz.row_exponent(np.abs(X).max(axis=1).astype(F64))
    e = np.zeros(len(ex), np.int32)
    harness.h_oz_exponent(len(ex), P(np.abs(X).max(axis=1).astype(F64)), P(e))
    assert np.array_equal(e, ex)
    h = ex >> 1
    xs = (X * oz.pow2_f32(-h)[:, None]).astype(F32).reshape(-1)
    sc = np.broadcast_to(oz.pow2_f32(-(ex - h))[:, None], X.shape).astype(F32).reshape(-1)
    q = np.zeros((oz.SLICES, xs.size), np.int32)
    harness.h_oz_digits_f32(xs.size, P(xs), P(np.ascontiguousarray(sc)), P(q))
    q_ref, ev = oz.row_digits_f32(X)
    assert np.array_equal(ev, ex)
    assert np.array_equal(q, q_ref.reshape(oz.SLICES, -1))
    assert np.abs(q).max() <= 64
    # float64 digits of the extrusion inputs (differences of float32 pixels and products noise * amp)
    v = (X.astype(F64) - X[:, :1].astype(F64)).reshape(-1)
    sc64 = np.ldexp(1.0, -oz.row_exponent(np.abs(v).max())) * np.ones_like(v)
    q = np.zeros((oz.SLICES_B, v.size), np.int32)
    harness.h_oz_digits(v.size, P(v), P(sc64), P(q))
    assert np.array_equal(q, oz.digits(v, sc64, oz.SLICES_B))


def exact_f32(X, W):
    """Correctly rounded float32 of the exact X . W^T (products of float32 values are exact in float64; math.fsum gives
    the correctly rounded float64 sum and its residual), with the exact value's float64 approximation."""
    E, N = X.shape[0], W.shape[0]
    s, res = np.zeros((E, N)), np.zeros((E, N))
    X64, W64 = X.astype(F64), W.astype(F64)
    for e in range(E):
        terms = W64 * X64[e]
        for n in range(N):
            t = terms[n].tolist()
            s[e, n] = math.fsum(t)
            res[e, n] = math.fsum(t + [-s[e, n]])
    return oz.round_to_f32(s, res), s


def error_bound(X, W, lev):
    """Bound on |emulated - exact| before the final float32 rounding, per output (e, n).

    With ev, ea the row exponents, each element is x = 2^ev (sum_s qa_s 2^-(6+7s) + da), |da| <= 2^-42 (half the last
    digit), likewise w with |dw| <= 2^-42, and every digit |q| <= 64.  Then per term k
      |x w - x^ w^| <= |x - x^| |w| + |x^| |w - w^| <= 2^(ev+ea) (2^-42 + 2^-42 (1 + 2^-42))         (truncation)
    and the digit pairs with s + t = g >= lev that are dropped weigh |qa_s qb_t| 2^-(12+7g) <= 2^-7g each, c(g) of them
    (c = 6, 5, 4, 3, 2, 1 for g = 5 .. 10):
      dropped <= 2^(ev+ea) sum_{g >= lev} c(g) 2^-7g.
    The float64 chain of the epilogue rounds lev - 1 times, each at most 2^-53 of a partial sum bounded by
    2^(ev+ea) K sum_g c(g) 2^-7g (< 1.02 K 2^(ev+ea)).  Summed over the K terms:
      B = K 2^(ev+ea) (2^-41 (1 + 2^-43) + sum_{g >= lev} c(g) 2^-7g + (lev - 1) 2^-53 1.02).
    For the products (lev 5) the dropped pairs dominate: about 6 2^-35 of |x|max |W|row max per term.  For the
    extrusion (lev 6): 2^-41 + 5 2^-42 + ... ~ 3.6 2^-41 per term, far below a float32 ulp of any output that is not the
    result of cancellation."""
    K = X.shape[1]
    cnt = {g: min(g, 10 - g) + 1 for g in range(11)}
    c = 2.0 ** -41 * (1 + 2.0 ** -43) + sum(cnt[g] * 2.0 ** (-7 * g) for g in range(lev, 11)) + (lev - 1) * 2.0 ** -53 * 1.02
    _, ev = oz.row_digits_f32(X)
    _, ea = oz.operator_digits(W)
    return K * np.ldexp(c, (ev[:, None] + ea[None, :]).astype(np.int32))


def cancelling_operator(X, r, N):
    """Operator rows whose products with X cancel to about 2^-24 of their terms: the last element of each row fixes the
    sum to ~0 (rounded to float32)."""
    K = X.shape[1]
    W = r.standard_normal((N, K)).astype(F32)
    if K > 1:
        x0 = X[2].astype(F64)                   # a random row with maximum 1
        k = int(np.argmax(np.abs(x0)))
        if x0[k] != 0:
            rest = W.astype(F64) @ x0 - W[:, k].astype(F64) * x0[k]
            W[:, k] = (-rest / x0[k]).astype(F32)
    return W


@pytest.mark.parametrize("lev", [oz.LEVELS_PRODUCT, oz.LEVELS])
@pytest.mark.parametrize("K", [1, 33, 128, 513, 2400])
def test_emulation_within_bound_of_exact(K, lev):
    """The emulated contraction against exact arithmetic on adversarial input rows and operators (random, cancelling,
    adversarial rows): every output within the bound of `error_bound` plus half a float32 ulp.  Prints the fraction of
    outputs that are correctly rounded and the worst error over the bound."""
    r = np.random.default_rng(100 + K + lev)
    X = adversarial_rows(K, r)
    X = X[[i for i in range(len(X)) if np.abs(X[i]).max() < 2.0 ** 100]]      # keep the outputs finite
    N = 24
    W = np.concatenate([r.standard_normal((N // 2, K)).astype(F32), cancelling_operator(X, r, N // 4),
                        adversarial_rows(K, r)[:N // 4]])
    qa, ev = oz.row_digits_f32(X)
    qb, ea = oz.operator_digits(W)
    a = oz.combine(oz.level_sums(qa, qb, lev))
    pre = np.ldexp(a, (ev[:, None] + ea[None, :] - 12).astype(np.int32))       # before the float32 rounding
    got = pre.astype(F32)
    if lev == oz.LEVELS_PRODUCT:
        assert np.array_equal(got.view(np.int32), oz.product(X, W).view(np.int32))
    ref32, ref = exact_f32(X, W)
    B = error_bound(X, W, lev)
    assert (np.abs(pre - ref) <= B).all(), float((np.abs(pre - ref) / np.maximum(B, 1e-300)).max())
    ulp = np.spacing(np.abs(ref32)).astype(F64)
    assert (np.abs(got.astype(F64) - ref) <= B + 0.5 * ulp + 2.0 ** -149).all()
    ratio = float((np.abs(pre - ref) / np.maximum(B, 1e-300)).max())
    exact = float((got == ref32).mean())
    print("K %d lev %d: %.4f of %d outputs correctly rounded, worst error / bound %.3g" % (K, lev, exact, got.size, ratio))
    assert ratio <= 1.0
    if lev == oz.LEVELS:
        assert exact > 0.95                      # rounding differs only next to a float32 rounding boundary


def test_nonfinite_rows_are_nan():
    """A row holding a NaN or an infinity gives a NaN in every output of that row and changes no other row."""
    r = np.random.default_rng(3)
    X = r.standard_normal((5, 40)).astype(F32)
    W = r.standard_normal((7, 40)).astype(F32)
    good = oz.product(X, W)
    X[1, 3], X[3, 39] = np.nan, -np.inf
    out = oz.product(X, W)
    assert np.isnan(out[[1, 3]]).all()
    assert np.array_equal(out[[0, 2, 4]].view(np.int32), good[[0, 2, 4]].view(np.int32))


def test_fmaf_is_single_rounding():
    """The float32 fmaf emulation against exact rational arithmetic, on products and sums built to hit rounding ties."""
    from fractions import Fraction
    r = np.random.default_rng(11)
    a = r.standard_normal(4000).astype(F32)
    b = r.standard_normal(4000).astype(F32)
    c = (-(a.astype(F64) * b.astype(F64))).astype(F32)            # near-total cancellation
    c[::3] = r.standard_normal(c[::3].size).astype(F32)
    c[1::7] = (a[1::7].astype(F64) * b[1::7].astype(F64) * 2.0 ** -25).astype(F32)    # ties and near-ties
    got = oz.fmaf(a, b, c)
    for i in range(a.size):
        ex = Fraction(float(a[i])) * Fraction(float(b[i])) + Fraction(float(c[i]))
        lo = F32(float(ex))                                       # candidate, then the correctly rounded neighbour
        cands = [np.nextafter(lo, F32(-np.inf)), lo, np.nextafter(lo, F32(np.inf))]
        best = min(cands, key=lambda v: (abs(Fraction(float(v)) - ex), int(np.asarray(v).view(np.int32)) & 1))
        assert got[i] == best, (i, a[i], b[i], c[i])


def test_extrusion_emulation_matches_oracle(static10):
    """One EPI 0 extrusion of the 10x10 layer from an identical screen, in every direction: the emulated integer
    contraction against oracle/aoframe.extrude (float64 evaluation, one rounding), within the one-ulp rule of
    test_single_extrusion_is_exact; nearly every pixel identical."""
    t = static10
    n = int(t.dim_screens[0])
    r = np.random.default_rng(5)
    scr = (r.standard_normal((n, n)).cumsum(0).cumsum(1) / n).astype(F32)
    AB = np.concatenate([t.A[0], t.B[0]], axis=1).astype(F32)
    op = oz.operator_digits(AB)
    amp = F32(F32(t.r0_layers[0]) ** F32(-5.0 / 6.0) * F32(0.5 / (2 * np.pi)))
    n_diff = n_tot = 0
    for axis in (0, 1):
        for sign in (1, -1):
            noise = oz.extrusion_noise(77, 0, 2 * n + 3, n)
            got = oz.extrude(scr, op, t.istx[0], amp, noise, axis, sign)
            ref = af.extrude(scr, t.A[0], t.B[0], t.istx[0], amp, noise, axis, sign)
            d = np.abs(got.astype(F64) - ref.astype(F64))
            allowed = np.maximum(np.spacing(np.abs(ref)).astype(F64), 2.0 ** -26 * np.abs(ref).max())
            assert (d <= allowed).all(), float((d / allowed).max())
            n_diff += int((d > 0).sum())
            n_tot += n
    assert n_diff <= 1e-2 * n_tot + 1, (n_diff, n_tot)
