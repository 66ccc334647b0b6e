"""The integer tensor-core contraction (oz_gemm_kernel, extrude_i8.cuh) at its real call sites against its bit-exact numpy
emulation (oracle/ozaki.py) and against float64: the controller products of aom_do_control (err = -cmat s and the
integrator), aom_rl_control (v2m com, m2v modes) and aom_state_end (v2m err), and the screen extrusion.

Batches span several M tiles of 128 environments (E = 127, 128, 129, 300 and the headline 4096), so the per-tile digit
planes, the loader's tile offsets and the ragged last tile are all compared.  Operators get rows of very different
magnitudes, so every N tile of 80 outputs has its own exponents.  The achieved numbers (bit-exact fraction against
float64, errors against the oracle) are printed at the end of the module (pytest -s shows them)."""
import json

import numpy as np
import pytest

from oracle import aoframe as af
from oracle import ozaki as oz

pytestmark = pytest.mark.gpu

F32, F64 = np.float32, np.float64
GEMM_TOL = {"simt": 1e-5, "tf32": 5e-5}        # the tolerances of test_gpu_parity.py::test_gemm_paths
REPORT = {}


def record(test, key, value):
    REPORT.setdefault(test, {})[key] = value


@pytest.fixture(scope="module", autouse=True)
def _print_report():
    yield
    if REPORT:
        print("\ninteger contractions, achieved numbers:\n" + json.dumps(REPORT, indent=1, sort_keys=True))


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def relerr(a, b):
    a, b = np.asarray(a, F64), np.asarray(b, F64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def assert_bits(got, ref, what):
    """Bit-identical float32 arrays; NaN positions must agree (their payloads may differ)."""
    got, ref = np.asarray(got, F32), np.asarray(ref, F32)
    nan = np.isnan(ref)
    assert np.array_equal(np.isnan(got), nan), "%s: NaN positions differ" % what
    diff = (got.view(np.uint32) != ref.view(np.uint32)) & ~nan
    if diff.any():
        e, n = np.argwhere(diff)[0]
        raise AssertionError("%s: %d of %d outputs differ from the emulation, first at row %d column %d: %r != %r"
                             % (what, int(diff.sum()), diff.size, e, n, got[e, n], ref[e, n]))


def tables(par):
    from ao_marl_b200 import tables as tb
    from ao_marl_b200.config import load_config_from_file
    t = tb.build_static(load_config_from_file(par))
    tb.build_basis(t)
    return t


def layout(t, par):
    from ao_marl_b200.rl.layout import RLLayout
    s1 = 80 if "10x10" in par else 1260
    return RLLayout(t.Btt.shape[1], dict(parameters_telescope=par, n_zernike_start_end=[0, s1]), None)


def operator(r, rows, K, spread=6.0):
    """Random float32 operator whose rows differ in magnitude by up to e^(2 spread), with a zero row and a one-element row."""
    W = (r.standard_normal((rows, K)) * np.exp(r.uniform(-spread, spread, (rows, 1)))).astype(F32)
    W[rows // 3] = 0
    W[(2 * rows) // 3, :] = 0
    W[(2 * rows) // 3, K // 2] = F32(-0.625)
    return W


def inputs(r, E, K, adversarial=True, spread=3.0):
    """Per-environment float32 rows with environment scales over e^+-spread, and adversarial rows in the first
    environments: zero, single element, maximum exactly 2^k, subnormal maximum, one outlier."""
    X = (r.standard_normal((E, K)) * np.exp(r.uniform(-spread, spread, (E, 1)))).astype(F32)
    if adversarial and E >= 6:
        X[1] = 0
        X[2] = 0; X[2, K - 1] = F32(1.5)
        X[3] = (r.uniform(-1, 1, K) * 4).astype(F32); X[3, K // 2] = F32(-4.0)
        X[4] = (r.uniform(-1, 1, K) * 2.0 ** -140).astype(F32)
        X[5] = (r.uniform(-1, 1, K) * 1e-6).astype(F32); X[5, 7 % K] = F32(2.0e3)
    return X


def sampled_envs(E, r, n=64):
    """Environments 0, 127, 128, 129, the last row of every M tile, E - 1, and random ones."""
    s = {0, 127, 128, 129, E - 1} | {m * oz.BM + oz.BM - 1 for m in range((E + oz.BM - 1) // oz.BM)}
    s = {e for e in s if e < E}
    rest = np.setdiff1d(np.arange(E), sorted(s))
    s |= set(r.choice(rest, size=min(max(n - len(s), 0), rest.size), replace=False).tolist())
    return np.array(sorted(s))


class Loop:
    """The controller products of one context, run at their call sites and emulated on the environments `envs`."""

    def __init__(self, sim, t, rl, envs, torch):
        self.sim, self.t, self.rl, self.envs, self.torch = sim, t, rl, envs, torch
        self.nm = t.Btt.shape[1]
        sim.set_table("FREEDOM", np.zeros(self.nm, F32))      # the action injection then adds exactly zero

    def upload(self, cmat, v2m, m2v):
        from ao_marl_b200.lib import pad_rows
        self.sim.set_table("CMAT", pad_rows(cmat))
        self.sim.set_table("V2M", pad_rows(v2m))
        self.sim.set_table("M2V", pad_rows(m2v))
        self.cmat, self.v2m, self.m2v = cmat, v2m, m2v

    def rows(self, name, n):
        return self.sim.rows(name, n).cpu().numpy()[self.envs]

    def run(self, S, C, closed, gain):
        """do_control, state_begin / state_end, rl_control; returns the GPU results on the sampled environments."""
        sim, torch, t = self.sim, self.torch, self.t
        sim.rows("SLOPES", t.nslopes).copy_(torch.as_tensor(S, device="cuda"))
        sim.set_command(torch.as_tensor(C, device="cuda"))
        sim.set_loop(closed)
        if np.ndim(gain):
            sim.set_gain_env(gain)
        else:
            sim.set_gain_env(None)
            sim.set_gain(gain)
        sim.do_control()
        out = dict(ERR=self.rows("ERR", t.nactu), COM1=self.rows("COM", t.nactu))
        sim.state_begin()
        sim.state_end()
        out["RES_MODES"] = self.rows("RES_MODES", self.nm)
        sim.rl_control(np.zeros(self.rl.action_dim, F32))
        out["MODES"] = self.rows("MODES", self.nm)
        out["COM2"] = self.rows("COM", t.nactu)
        sim.check_device()
        return out

    def emulate(self, S, C, closed, gain):
        e = self.envs
        S, C = S[e], C[e]
        err = -oz.product(S, self.cmat)
        g = np.asarray(gain, F32)[e] if np.ndim(gain) else F32(gain)
        com = oz.integrate(err, C, g) if closed else C
        modes = oz.product(com, self.v2m)
        return dict(ERR=err, COM1=com, RES_MODES=oz.product(err, self.v2m), MODES=modes, COM2=oz.product(modes, self.m2v))

    def check(self, S, C, closed, gain, what):
        got, ref = self.run(S, C, closed, gain), self.emulate(S, C, closed, gain)
        for k in ref:
            assert_bits(got[k], ref[k], "%s %s" % (what, k))
        # float64 for the record: how often the single rounding lands on the correctly rounded result
        ref64 = -(S[self.envs].astype(F64) @ self.cmat.astype(F64).T)
        fine = np.abs(S[self.envs]).max(axis=1) > 2.0 ** -100
        same = float((got["ERR"][fine] == ref64[fine].astype(F32)).mean())
        record(what, "err_equal_to_rounded_float64", same)
        record(what, "err_rel_to_float64", relerr(got["ERR"][fine], ref64[fine]))
        return got


def product_cases(loop, r, E, what):
    t = loop.t
    S = inputs(r, E, t.nslopes)
    C = inputs(r, E, t.nactu, adversarial=False) * F32(0.01)
    gains = r.uniform(0.1, 0.9, E).astype(F32)
    loop.check(S, C, False, 0.5, what + " open")
    loop.check(S, C, True, 0.37, what + " closed")
    loop.check(S, C, True, gains, what + " closed per-env gain")
    # another operator scale: new exponents for every row
    loop.upload(loop.cmat * F32(2.0 ** -20), loop.v2m * F32(3.0 ** 7), loop.m2v * F32(2.0 ** 9 / 3.0))
    loop.check(S, C, True, 0.37, what + " rescaled operators")


@pytest.mark.parametrize("E", [1, 127, 128, 129, 300])
def test_products_10x10_bit_exact(static10, torch, E):
    """cmat 90 x 128, v2m 87 x 90, m2v 90 x 87: ERR after do_control, RES_MODES after state_end, MODES and COM after
    rl_control equal the emulation bit for bit in every row, loop open and closed, common and per-environment gain, and
    after re-uploading the operators at another scale."""
    from ao_marl_b200.lib import Simulator
    par = "production_sh_10x10_2m.py"
    rl = layout(static10, par)
    sim = Simulator(static10, E, rl, atmosphere=False)
    try:
        r = np.random.default_rng(E)
        loop = Loop(sim, static10, rl, np.arange(E), torch)
        nm = static10.Btt.shape[1]
        loop.upload(operator(r, static10.nactu, static10.nslopes), operator(r, nm, static10.nactu),
                    operator(r, static10.nactu, nm))
        product_cases(loop, r, E, "products10[E=%d]" % E)
    finally:
        sim.close()


@pytest.fixture(scope="module")
def sim40(torch):
    """The headline configuration at E = 4096 (3 layers, 1286 actuators, 2400 slopes, 1283 modes)."""
    from ao_marl_b200.lib import Simulator
    par = "production_sh_40x40_8m_3layers.py"
    t = tables(par)
    rl = layout(t, par)
    sim = Simulator(t, 4096, rl)
    yield sim, t, rl
    sim.close()


def test_products_40x40_E4096_bit_exact(sim40, torch):
    """cmat 1286 x 2400, v2m 1283 x 1286, m2v 1286 x 1283 at E = 4096, compared bit for bit on 64 sampled environments:
    0, 127, 128, 129, the last row of every M tile, 4095 and random ones (rows are independent, so sampling loses
    nothing)."""
    sim, t, rl = sim40
    r = np.random.default_rng(40)
    E = sim.n_env
    loop = Loop(sim, t, rl, sampled_envs(E, r), torch)
    nm = t.Btt.shape[1]
    loop.upload(operator(r, t.nactu, t.nslopes), operator(r, nm, t.nactu), operator(r, t.nactu, nm))
    product_cases(loop, r, E, "products40[E=4096]")


def logical_screens(sim, l, envs):
    n = int(sim.cfg.screen_dim[l])
    idx = sim.torch.as_tensor(envs, device="cuda")
    scr = sim.buffer("SCREEN", l).view(sim.n_env, n, n).index_select(0, idx).cpu().numpy()
    ox = sim.buffer("RING_OX", l).cpu().numpy()[envs]
    oy = sim.buffer("RING_OY", l).cpu().numpy()[envs]
    return [np.roll(scr[i], (-oy[i], -ox[i]), axis=(0, 1)) for i in range(len(envs))]


def check_extrusions(sim, t, envs, seeds, what):
    """One move with winds +/+, -/- and +/- (one x and one y extrusion per layer): every sampled environment's screen
    equals the emulation bit for bit, and the oracle's float64 extrusion from the same screen within one ulp."""
    AB = [np.concatenate([t.A[l], t.B[l]], axis=1).astype(F32) for l in range(t.nscreens)]
    ops = [oz.operator_digits(ab) for ab in AB]             # digits of [A | B], as aom_set_table cuts them
    worst, n_diff, n_tot = 0.0, 0, 0
    for sx, sy in ((1, 1), (-1, -1), (1, -1)):
        for l in range(t.nscreens):
            sim.set_layer(l, 1.0 * sx, 1.0 * sy, float(sim.cfg.amp[l]))
        before = [np.stack(logical_screens(sim, l, envs)) for l in range(t.nscreens)]
        count = [sim.buffer("EXT_COUNT", l).cpu().numpy()[envs] for l in range(t.nscreens)]
        sim.move_atmos()
        for l in range(t.nscreens):
            after = np.stack(logical_screens(sim, l, envs))
            n, amp = int(t.dim_screens[l]), F32(sim.cfg.amp[l])
            s = before[l]
            for j, (axis, sign) in enumerate(((0, sx), (1, sy))):
                noise = np.stack([oz.extrusion_noise(seeds[e], l, int(count[l][i]) + j, n) for i, e in enumerate(envs)])
                ref = np.stack([af.extrude(s[i], t.A[l], t.B[l], t.istx[l], amp, noise[i], axis, sign)
                                for i in range(len(envs))])
                s = oz.extrude(s, ops[l], t.istx[l], amp, noise, axis, sign)
                d = np.abs(s.astype(F64) - ref.astype(F64))
                allowed = np.maximum(np.spacing(np.abs(ref)).astype(F64),
                                     2.0 ** -26 * np.abs(ref).max(axis=(1, 2), keepdims=True))
                worst = max(worst, float((d / allowed).max()))
                n_diff += int((d > 0).sum())
                n_tot += n * len(envs)
            for i, e in enumerate(envs):
                assert_bits(after[i], s[i], "%s layer %d env %d wind %+d/%+d" % (what, l, e, sx, sy))
    record(what, "oracle_worst_error_over_allowed", worst)
    record(what, "oracle_pixels_differing", n_diff)
    record(what, "pixels_written", n_tot)
    assert worst <= 1.0, worst
    assert n_diff <= 1e-2 * n_tot + 1, (n_diff, n_tot)
    sim.check_device()


def test_extrusion_10x10_E300_bit_exact(static10, torch):
    from ao_marl_b200.lib import Simulator
    sim = Simulator(static10, 300, rl=None)
    try:
        seeds = np.arange(300, dtype=np.int64) * 7 + 3
        sim.reset(seeds)
        envs = sampled_envs(300, np.random.default_rng(3), n=300)
        check_extrusions(sim, static10, envs, seeds, "extrusion10[E=300]")
    finally:
        sim.close()


def test_extrusion_40x40_E4096_bit_exact(sim40, torch):
    sim, t, _ = sim40
    seeds = np.arange(4096, dtype=np.int64) + 1000
    sim.reset(seeds)
    check_extrusions(sim, t, sampled_envs(4096, np.random.default_rng(4), n=40), seeds, "extrusion40[E=4096]")


@pytest.fixture(scope="module")
def loop10(static10, torch):
    """A 10x10 context with E = 130 (two M tiles), random operators."""
    from ao_marl_b200.lib import Simulator
    par = "production_sh_10x10_2m.py"
    rl = layout(static10, par)
    sim = Simulator(static10, 130, rl)
    r = np.random.default_rng(9)
    loop = Loop(sim, static10, rl, np.arange(130), torch)
    nm = static10.Btt.shape[1]
    loop.upload(operator(r, static10.nactu, static10.nslopes), operator(r, nm, static10.nactu),
                operator(r, static10.nactu, nm))
    yield loop
    sim.close()


@pytest.mark.parametrize("path", ["simt", "tf32"])
def test_cross_check_paths_against_float64(loop10, path):
    """The same products through the float32 SIMT and 3xTF32 GEMM paths, integrator epilogues included, against
    float64 within the tolerances of test_gemm_paths."""
    t, sim = loop10.t, loop10.sim
    r = np.random.default_rng(17)
    E = sim.n_env
    S = inputs(r, E, t.nslopes, adversarial=False, spread=0.0)
    C = inputs(r, E, t.nactu, adversarial=False, spread=0.0) * F32(0.01)
    gains = r.uniform(0.1, 0.9, E).astype(F32)
    try:
        sim.set_gemm_path(path)
        for closed, gain in ((False, 0.5), (True, 0.37), (True, gains)):
            got = loop10.run(S, C, closed, gain)
            err = -(S.astype(F64) @ loop10.cmat.astype(F64).T)
            g = gains[:, None].astype(F64) if np.ndim(gain) else F64(F32(gain))
            com = C.astype(F64) + g * err if closed else C.astype(F64)
            ref = dict(ERR=err, COM1=com, RES_MODES=got["ERR"].astype(F64) @ loop10.v2m.astype(F64).T,
                       MODES=got["COM1"].astype(F64) @ loop10.v2m.astype(F64).T,
                       COM2=got["MODES"].astype(F64) @ loop10.m2v.astype(F64).T)
            for k, v in ref.items():
                e = relerr(got[k], v)
                key = "cross_check[%s]" % path
                record(key, k, max(e, REPORT.get(key, {}).get(k, 0.0)))
                assert e < GEMM_TOL[path], (path, closed, k, e)
    finally:
        sim.set_gemm_path("tcgen05")
        sim.set_gain_env(None)


@pytest.mark.parametrize("path", ["tcgen05", "simt"])
def test_nonfinite_inputs_poison_their_row_only(loop10, path):
    """A NaN in one slope row makes that row's ERR (and, loop closed, its COM) non-finite; +Inf in one COM row does the
    same through rl_control.  Every other row is bit-identical to a run without the bad row.  The integer path gives NaN
    in every output of the row; the SIMT path may give +-Inf where it gives NaN."""
    t, sim = loop10.t, loop10.sim
    r = np.random.default_rng(23)
    E = sim.n_env
    S = inputs(r, E, t.nslopes, adversarial=False)
    C = inputs(r, E, t.nactu, adversarial=False) * F32(0.01)
    bad_s, bad_c = 129, 3                                  # one in each M tile
    S_bad, C_bad = S.copy(), C.copy()
    S_bad[bad_s, 17] = np.nan
    C_bad[bad_c, 40] = np.inf
    try:
        sim.set_gemm_path(path)
        good = loop10.run(S, C, True, 0.37)
        got = loop10.run(S_bad, C, True, 0.37)
        got_c = loop10.run(S, C_bad, True, 0.37)
    finally:
        sim.set_gemm_path("tcgen05")
    for res, bad, keys in ((got, bad_s, ("ERR", "COM1", "RES_MODES", "MODES", "COM2")), (got_c, bad_c, ("MODES", "COM2"))):
        others = np.setdiff1d(np.arange(E), [bad])
        for k in keys:
            row = res[k][bad]
            if path == "tcgen05":
                assert np.isnan(row).all(), (k, row)
            else:
                assert not np.isfinite(row).any(), (k, row)
            assert_bits(res[k][others], good[k][others], "%s %s other rows" % (path, k))


def test_nonfinite_operator_tables_are_refused(loop10):
    """A NaN or an infinity in CMAT, V2M, M2V or AB raises ValueError and leaves the uploaded operators in force."""
    from ao_marl_b200.lib import pad_rows
    t, sim = loop10.t, loop10.sim
    r = np.random.default_rng(29)
    S = inputs(r, sim.n_env, t.nslopes, adversarial=False)
    C = inputs(r, sim.n_env, t.nactu, adversarial=False) * F32(0.01)
    before = loop10.run(S, C, True, 0.37)
    for name, W in (("CMAT", loop10.cmat), ("V2M", loop10.v2m), ("M2V", loop10.m2v)):
        for bad in (np.nan, np.inf, -np.inf):
            Wb = W.copy()
            Wb[W.shape[0] - 1, W.shape[1] // 2] = bad
            with pytest.raises(ValueError):
                sim.set_table(name, pad_rows(Wb))
    ab = np.concatenate([t.A[0], t.B[0]], axis=1).astype(F32)
    ab[3, 5] = np.nan
    with pytest.raises(ValueError):
        sim.set_table("AB", pad_rows(ab), 0)
    after = loop10.run(S, C, True, 0.37)
    for k in before:
        assert_bits(after[k], before[k], "after refused uploads: %s" % k)
