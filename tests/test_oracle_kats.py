"""Pins of the oracle itself: Random123 known answers for Philox4x32-10, the device math headers
(host build) bit-equal to oracle/rng.py, and the self-consistency KATs of SURVEY.md 8(c)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import aoframe as af
from oracle import loop, rng

HERE = os.path.dirname(os.path.abspath(__file__))


def test_philox_known_answers():
    # Random123 kat_vectors, philox4x32 10 rounds
    kats = [((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
            ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
            ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
             (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))]
    for c, k, want in kats:
        got = tuple(int(v) for v in rng.philox4x32(*c, *k))
        assert got == want


def test_det_math_accuracy():
    r = np.random.default_rng(1)
    x = (r.random(100000) * 0.999 + 1e-6).astype(np.float32)
    assert np.abs(rng.det_log(x) - np.log(x.astype(np.float64))).max() < 2e-6
    c, s = rng.det_sincos2pi(x)
    assert np.abs(c - np.cos(2 * np.pi * x.astype(np.float64))).max() < 3e-7
    assert np.abs(s - np.sin(2 * np.pi * x.astype(np.float64))).max() < 3e-7
    y = (-30 * x).astype(np.float32)
    assert (np.abs(rng.det_exp(y) - np.exp(y.astype(np.float64))) / np.exp(y.astype(np.float64))).max() < 1e-6
    z = rng.atmos_noise(1234, 0, 5, 200000)
    assert abs(z.mean()) < 0.01 and abs(z.std() - 1) < 0.01
    for lam in (0.3, 3.7, 29.9, 30.0, 500.0):
        k = rng.wfs_pixel_noise(7, 0, 1, np.full(200000, lam, np.float32), 0.0)
        assert abs(k.mean() - lam) < 0.02 * max(lam, 1) and abs(k.var() - lam) < 0.05 * max(lam, 1)
        assert np.array_equal(k, np.round(k)) and k.min() >= 0


@pytest.fixture(scope="module")
def harness():
    src = os.path.join(HERE, "cpu_kernels", "harness.cpp")
    out = os.path.join(HERE, "cpu_kernels", "libharness.so")
    if not os.path.exists(out) or os.path.getmtime(out) < os.path.getmtime(src):
        subprocess.run(["g++", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-o", out, src], check=True)
    return ctypes.CDLL(out)


def P(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def test_device_headers_bit_equal_to_oracle(harness):
    """rng.cuh compiled for the host produces the oracle's bits (the GPU runs the same source)."""
    L = harness
    n = 100000
    r = np.random.default_rng(0)
    c = [r.integers(0, 2 ** 32, n, dtype=np.uint32) for _ in range(4)]
    out = np.zeros(4 * n, np.uint32)
    L.h_philox(n, P(c[0]), P(c[1]), P(c[2]), P(c[3]), ctypes.c_uint32(123), ctypes.c_uint32(456), P(out))
    assert np.array_equal(out, np.stack(rng.philox4x32(c[0], c[1], c[2], c[3], 123, 456), 1).reshape(-1))
    x = (r.random(n) * 0.999 + 1e-6).astype(np.float32)
    lg, ex, cc, ss = (np.zeros(n, np.float32) for _ in range(4))
    L.h_det(n, P(x), P(lg), P(ex), P(cc), P(ss))
    c2, s2 = rng.det_sincos2pi(x)
    assert np.array_equal(lg, rng.det_log(x)) and np.array_equal(ex, rng.det_exp(np.float32(-30) * x))
    assert np.array_equal(cc, c2) and np.array_equal(ss, s2)
    z = np.zeros(1001, np.float32)
    L.h_normals(1001, ctypes.c_int64(2 ** 40 + 77), ctypes.c_uint32(9), ctypes.c_uint32(1), ctypes.c_uint32(2), P(z))
    assert np.array_equal(z, rng.atmos_noise(2 ** 40 + 77, 2, 9, 1001))
    for noise in (0.0, 3.0):
        lam = (r.random(n) ** 3 * 200).astype(np.float32)
        lam[:10] = 0
        o = np.zeros(n, np.float32)
        L.h_pixel_noise(n, P(lam), ctypes.c_float(noise), ctypes.c_int64(99), ctypes.c_uint32(5), ctypes.c_uint32(0), P(o))
        assert np.array_equal(o, rng.wfs_pixel_noise(99, 0, 5, lam, noise))


def test_poisson_tail_known_answers(harness):
    """The largest Philox words must give a plausible tail sample, never the loop cap (round-1 advisor finding:
    u01 rounded to exactly 1.0 and the search ran to POISSON_MAXK = 200).  Oracle and device header agree."""
    lams = np.array([0.1, 0.5, 1, 2, 3, 5, 8, 10, 15, 20, 25, 29.9], np.float32)
    words = np.array([0xFFFFFFFF, 0xFFFFFF00, 0xFFFFFE00, 0xFFFFFDFF, 0xFFFFF000, 0x80000000, 0, 0x1FF], np.uint32)
    lam = np.repeat(lams, words.size)
    x0 = np.tile(words, lams.size)
    x1 = np.zeros_like(x0)
    k = rng.poisson_from_words(lam, x0, x1)
    out = np.zeros(lam.size, np.int32)
    harness.h_poisson(lam.size, P(lam), P(x0), P(x1), P(out))
    assert np.array_equal(out, k)
    assert float(rng.u01_open(np.uint32(0xFFFFFFFF))) < 1.0 and float(rng.u01_open(np.uint32(0))) > 0.0
    top = k.reshape(lams.size, words.size)[:, 0]
    # tail sample: beyond the mean, but within a 2^-24 quantile (lam + 12 sqrt(lam) + 12 bounds it generously)
    assert (top < rng.POISSON_MAXK).all()
    assert (top > lams).all() and (top <= lams + 12 * np.sqrt(lams) + 12).all(), top
    # monotone in u
    order = np.argsort(words.astype(np.uint64) >> np.uint64(9), kind="stable")
    kk = k.reshape(lams.size, words.size)[:, order]
    assert (np.diff(kk, axis=1) >= 0).all()


@pytest.mark.parametrize("R", [4, 8])
def test_pruned_dft_matches_fft2(harness, R):
    """fft16.cuh (host build): the kernel's pruned 2-D DFT equals the central Nfft/2 block of numpy's fft2."""
    r = np.random.default_rng(R)
    N, H = 16 * R, 4 * R
    W = 2 * H
    a = (r.standard_normal((16, 16)) + 1j * r.standard_normal((16, 16))).astype(np.complex64)
    inr, ini = np.ascontiguousarray(a.real), np.ascontiguousarray(a.imag)
    inten = np.zeros((W, W), np.float32)
    harness.h_spot(R, P(inr), P(ini), P(inten))
    full = np.zeros((N, N), np.complex128)
    full[:16, :16] = a
    I = np.abs(np.fft.fft2(full)) ** 2
    I = np.roll(np.roll(I, H, 0), H, 1)[:W, :W]
    assert np.abs(inten - I).max() / I.max() < 2e-6


def test_sh_frame_kats(oracle_tab10):
    tab = oracle_tab10
    w, n = tab["wfs"], tab["n"]
    nv = w["nvalid"]
    s = loop.wfs_frame(tab, np.zeros((n, n), np.float32), -1, 0, 0)
    assert np.abs(s).max() < 1e-6                      # flat wavefront -> zero slopes (fixes the halfxy sign)
    theta, pix = 0.05, 2.0 / 160
    ramp = (theta / af.ARCSEC_PER_RAD * np.arange(n) * pix * 1e6).astype(np.float32)
    s = loop.wfs_frame(tab, np.tile(ramp[None, :], (n, 1)), -1, 0, 0)
    assert abs(s[:nv].mean() / theta - 1) < 5e-3 and np.abs(s[nv:]).max() < 1e-5   # tilt x -> x slopes only
    s = loop.wfs_frame(tab, np.tile(ramp[:, None], (1, n)), -1, 0, 0)
    assert abs(s[nv:].mean() / theta - 1) < 5e-3 and np.abs(s[:nv]).max() < 1e-5
    cube = af.sh_bincube(np.tile(ramp[None, :], (n, 1)), tab["mpupil"], w)
    assert np.allclose(cube.sum(axis=(1, 2)), w["nphotons"] * w["fluxPerSub"], rtol=1e-5)


def test_poke_reproduces_stamp(oracle_tab10, static10):
    pz = oracle_tab10["pzt"]
    v = np.zeros(pz["nact"], np.float32)
    v[40] = 3.0
    sh = af.pzt_shape(v, pz["influ"], pz["i1"], pz["j1"], pz["dim"])
    ss = pz["influ"].shape[0]
    x0, y0 = int(pz["i1"][40]), int(pz["j1"][40])
    assert np.array_equal(sh[y0:y0 + ss, x0:x0 + ss], np.float32(3.0) * pz["influ"][:, :, 40].T)
    assert np.count_nonzero(sh) == np.count_nonzero(pz["influ"][:, :, 40])


def test_tt_unit_and_integrator(oracle_tab10, oracle_imat10, static10):
    from ao_marl_b200.init import rtc as rtc_b
    D = oracle_imat10
    nv = oracle_tab10["wfs"]["nvalid"]
    # one unit on the tip-tilt mirror = unitpervolt arcsec of tilt (dm_init.py:683-686)
    assert abs(D[:nv, -2].mean() / static10.p_tt.unitpervolt - 1) < 1e-2
    assert abs(D[nv:, -1].mean() / static10.p_tt.unitpervolt - 1) < 1e-2
    cmat = rtc_b.cmat_with_btt(D, static10.Btt, 0)
    RD = static10.P.astype(np.float64) @ (cmat.astype(np.float64) @ D.astype(np.float64)) @ static10.Btt.astype(np.float64)
    assert np.abs(RD - np.eye(RD.shape[0])).max() < 1e-4          # R.D = I on the controlled modes


def test_closed_loop_statistics(oracle_tab10, oracle_imat10, static10):
    """Closed-loop slope rms of the oracle against the statistic committed by the reference authors
    (real COMPASS, 10x10: std of slopes ~ 0.099 arcsec; BASELINE.md section 2)."""
    from ao_marl_b200.init import rtc as rtc_b
    from ao_marl_b200.rl.layout import load_normalization
    cmat = rtc_b.cmat_with_btt(oracle_imat10, static10.Btt, 0)
    env = loop.OracleEnv(oracle_tab10, cmat, static10.Btt, static10.P, None, seed=3)
    env.reset(3)
    rms = []
    for i in range(150):
        env.apply_control()
        env.linear_step()
        if i >= 30:
            rms.append(env.slopes.std())
    norm, _ = load_normalization("production_sh_10x10_2m.py")
    ref = float(norm["wfs"]["std"].mean())
    assert abs(np.mean(rms) / ref - 1) < 0.25


def test_psf_peak_fit_known_answers():
    """oracle.aoframe.psf_image / fit_peak: flat wavefront -> peak 1 on axis; a pure tilt of a fraction of a pixel leaves
    the fitted peak within 1 % of 1 while the brightest pixel drops; a Gaussian image is fitted exactly."""
    from oracle import aoframe as af
    n, nfft = 64, 256
    yy, xx = np.mgrid[0:n, 0:n] - (n - 1) / 2.0
    pup = (xx ** 2 + yy ** 2) <= (n / 2.0) ** 2
    img = af.psf_image(np.zeros((n, n)), pup, 1.65, nfft)
    assert abs(img[0, 0] - 1.0) < 1e-12 and abs(af.fit_peak(img) - 1.0) < 1e-9
    lam = 1.65
    for shift in (0.2, 0.4):                                   # focal shift in pixels of the nfft grid
        tilt = lam * shift * xx / nfft                          # k * tilt = 2 pi shift x / nfft
        img = af.psf_image(tilt, pup, lam, nfft)
        assert img.max() < 1.0 - 0.02 * shift
        assert abs(af.fit_peak(img) - 1.0) < 0.01
    jj, ii = np.mgrid[0:32, 0:32]
    gimg = 0.7 * np.exp(-((jj - 10.3) ** 2 + (ii - 20.6) ** 2) / 8.0)
    assert abs(af.fit_peak(gimg) - 0.7) < 1e-12


def test_pretiled_actor_weights_layout(harness):
    """gtc_pretile_host (what aom_set_table runs on the actor weights): TF32 hi / lo planes in the UMMA K-major no-swizzle
    tile order gemm_tc_kernel reads with one bulk copy per stage -- hi keeps the leading 11 significant bits, hi + lo is the
    weight exactly, rows / columns beyond the operator are zero, and every element sits at
    [n tile][k block][hi, lo][(r >> 3) * 128 + (k >> 2) * 32 + (r & 7) * 4 + (k & 3)]."""
    L = harness
    L.h_pretile_floats.restype = ctypes.c_longlong
    r = np.random.default_rng(5)
    batch, rows, K = 3, 60, 272                       # the head layer of the 40x40 actors: 2 x 30 outputs, 256 + pad inputs
    ldb, ldc = 272, 64
    W = (r.standard_normal((batch, rows, ldb)) * r.choice([1e-3, 1.0, 50.0], (batch, rows, 1))).astype(np.float32)
    W[:, :, 260:] = 0.0
    per = L.h_pretile_floats(ldc, K)
    NT, nkb = (ldc + 127) // 128, (K + 15) // 16
    assert per == NT * nkb * 2 * 128 * 16
    out = np.full(batch * per, np.nan, np.float32)
    L.h_pretile(P(W), batch, ctypes.c_longlong(rows * ldb), ldb, rows, ldc, K, P(out))
    out = out.reshape(batch, NT, nkb, 2, 128 * 16)
    assert np.isfinite(out).all()
    rr, kk = np.meshgrid(np.arange(128), np.arange(16), indexing="ij")
    off = (rr >> 3) * 128 + (kk >> 2) * 32 + (rr & 7) * 4 + (kk & 3)
    assert len(np.unique(off)) == 128 * 16
    for b in range(batch):
        for kb in range(nkb):
            tile = np.zeros((128, 16), np.float32)
            tile[:rows] = W[b, :, 16 * kb:16 * kb + 16]
            hi = (tile.view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32)
            assert np.array_equal(out[b, 0, kb, 0][off], hi)
            assert np.array_equal(out[b, 0, kb, 1][off], tile - hi)
            assert np.array_equal(out[b, 0, kb, 0][off] + out[b, 0, kb, 1][off], tile)


def _lattice_inputs(t):
    """aom_config fields and host tables of the staged sensor kernels, as Simulator uploads them."""
    from ao_marl_b200.lib import AomConfig, actuator_lattice, separable_factor
    w = t.p_wfs
    cfg = AomConfig()
    cfg.n, cfg.n_layers, cfg.nvalid, cfg.nfft, cfg.nrebin = t.n, t.nscreens, w._nvalid, w._Nfft, w._nrebin
    for l in range(t.nscreens):
        cfg.screen_dim[l] = int(t.dim_screens[l])
    cfg.pzt_pitch, cfg.pzt_grid_n, cfg.pzt_i1_0, cfg.pzt_j1_0, amap = actuator_lattice(t.p_pzt)
    cfg.stamp_size, cfg.pzt_off, cfg.tt_dim, cfg.tt_off = t.p_pzt._influsize, t.pzt_off, t.tt_dim, t.tt_off
    tab = dict(pup=t.mpupil.astype(np.float32), sx=w._tile_origin[:, 1].astype(np.int32),
               sy=w._tile_origin[:, 0].astype(np.int32), stamp=separable_factor(t.p_pzt._influ[:, :, 0]), amap=amap)
    return cfg, tab


def _lattice(harness, cfg, tab):
    """wfl_analyse and the lattice builders (wfs_lattice_host.h): (refusal or None, geom, amap_pad, win, fac)."""
    harness.h_wfs_lattice.restype = ctypes.c_char_p
    GW = cfg.pzt_grid_n + 8
    geom, amap_pad = np.zeros(8, np.int32), np.zeros(GW * GW, np.int16)
    win, fac = np.zeros(cfg.nvalid, np.int32), np.zeros((2, 4, 16), np.float32)
    t = {k: np.ascontiguousarray(v) for k, v in tab.items()}
    why = harness.h_wfs_lattice(ctypes.byref(cfg), P(t["pup"]), P(t["sx"]), P(t["sy"]), P(t["stamp"]), P(t["amap"]),
                                P(geom), P(amap_pad), P(win), P(fac))
    return (why.decode() if why else None), geom, amap_pad, win, fac


@pytest.mark.parametrize("par", ["production_sh_10x10_2m.py",
                                 pytest.param("production_sh_40x40_8m_3layers.py", marks=pytest.mark.slow)])
def test_wfs_lattice_reproduces_mirror(harness, par):
    """The padded actuator map, window origins and stamp factors both staged sensor kernels derive their tables from give,
    for every pixel of every subaperture, the actuators and weights of the mirror sum of the SIMT kernel (wfs_kernels.cuh:
    stamp1d[Y - (j1_0 + 16 gy)] * stamp1d[X - (i1_0 + 16 gx)] over the lattice cells whose stamp covers the pixel)."""
    from ao_marl_b200 import tables
    from ao_marl_b200.config import load_config_from_file
    cfg, tab = _lattice_inputs(tables.build_static(load_config_from_file(par)))
    why, geom, amap_pad, win, fac = _lattice(harness, cfg, tab)
    assert why is None and geom[7] == 1
    GW, gn, ss, nact = geom[6], cfg.pzt_grid_n, cfg.stamp_size, int(tab["amap"].max()) + 1
    stamp, amap = tab["stamp"].astype(np.float64), tab["amap"]

    def factors(origin, base):      # [16 pixels][grid_n cells] stamp factor of the SIMT kernel
        d = origin + cfg.pzt_off + np.arange(16)[:, None] - (base + 16 * np.arange(gn))[None, :]
        return np.where((d >= 0) & (d < ss), stamp[np.clip(d, 0, ss - 1)], 0.0)

    on = amap >= 0
    for k in range(cfg.nvalid):
        fx, fy = factors(tab["sx"][k], cfg.pzt_i1_0), factors(tab["sy"][k], cfg.pzt_j1_0)
        ref = np.zeros((256, nact))
        ref[:, amap[on]] = np.einsum("yg,xh->yxgh", fy, fx).reshape(256, gn * gn)[:, on]
        got = np.zeros((256, nact))
        for jy in range(4):
            for jx in range(4):
                a = amap_pad[win[k] + jy * GW + jx]
                if a >= 0:
                    assert not got[:, a].any()
                    got[:, a] = np.outer(fac[1, jy].astype(np.float64), fac[0, jx].astype(np.float64)).ravel()
        assert np.array_equal(got, ref), k
        assert np.count_nonzero(ref.any(axis=0)) > 0


def test_wfs_lattice_refusals(harness, static10):
    """Geometries outside the staged sensor kernels are refused with the reasons aom_wfs_kernel reports."""
    from ao_marl_b200.lib import AomConfig
    cfg, tab = _lattice_inputs(static10)
    assert _lattice(harness, cfg, tab)[0] is None

    def refusal(cfg_changes={}, **tables):
        c = AomConfig()
        ctypes.memmove(ctypes.byref(c), ctypes.byref(cfg), ctypes.sizeof(cfg))
        for k, v in cfg_changes.items():
            setattr(c, k, v)
        return _lattice(harness, c, dict(tab, **tables))[0]

    pup = tab["pup"].copy()
    y, x = np.argwhere(pup == 1)[np.count_nonzero(pup) // 2]
    pup[y, x] = 0.5
    assert refusal(pup=pup) == "pupil transmission is not binary"
    sx, k = tab["sx"].copy(), cfg.nvalid // 2
    assert sx[k] + 4 + 16 <= cfg.n and 0 < k
    sx[k] += 4                                   # tip-tilt rows stay 16-byte aligned
    assert refusal(sx=sx) == "subapertures not aligned with the actuator lattice"
    assert refusal({"pzt_pitch": 8}) == "actuator pitch is not 16 pixels"
    assert refusal({"n_layers": 5}) == "more than 4 layers"
    assert refusal({"nfft": 128}) == "Nfft != 64"
    amap = tab["amap"].copy()
    amap[amap >= 0] += 40000                     # actuator indices beyond a short
    assert refusal(amap=amap) == "derived tables out of range"
    assert refusal({"pzt_grid_n": 2}) == "derived tables out of range"     # windows leave the padded map
