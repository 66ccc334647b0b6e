"""Pupil and Shack-Hartmann geometry tables (host side, numpy, run once at start-up).

Produces the integer maps and float tables that the reference builds in
shesha/init/geom_init.py (tel_init 49-108, init_wfs_geom 111-165, init_wfs_size 168-340,
compute_nphotons 343-407, init_sh_geom 622-811, geom_init 813-868) with
shesha/util/make_pupil.py:120-200 (generic aperture) and utilities.py:54-61,106-135.
Scope: SH sensors on a generic circular aperture with central obstruction, natural guide star.
Results are compared bit-for-bit (integers) against tests/golden/ref_tables_*.npz.
"""
import numpy as np

RAD2ARCSEC = 3600.0 * 360.0 / (2.0 * np.pi)
DEG2RAD = np.pi / 180.0
ARCSEC2RAD = 2.0 * np.pi / (360.0 * 3600.0)


def fft_goodsize(s):
    return 2 ** (int(np.log2(s)) + 1)


def radial_distance(dim, xc, yc):
    ax = np.arange(dim, dtype=np.float64)
    return np.sqrt((ax[None, :] - xc) ** 2 + (ax[:, None] - yc) ** 2)


def embed_centered(a, size):
    out = np.zeros((size, size))
    o0 = (size - a.shape[0]) // 2
    o1 = (size - a.shape[1]) // 2
    out[o0:o0 + a.shape[0], o1:o1 + a.shape[1]] = a
    return out


def generic_pupil(dim, pupd, p_tel, xc, yc):
    """Disc of diameter pupd minus the central obstruction (make_pupil.py:139-150).
    Spider arms exist in the reference only for spiders_type 'four'/'six'; the production files
    leave it unset, so anything else is refused rather than silently ignored."""
    if p_tel.type_ap not in ("Generic", "generic"):
        raise NotImplementedError("only the generic aperture is on the hot path")
    if p_tel.spiders_type is not None:
        raise NotImplementedError("spider arms are outside the hot-path scope")
    r = radial_distance(dim, xc, yc)
    pup = (r < (pupd + 1.0) / 2.0).astype(np.float32)
    if p_tel.cobs > 0:
        pup -= (r < (pupd * p_tel.cobs + 1.0) * 0.5).astype(np.float32)
    return pup


def geom_init(p_geom, p_tel, padding=2):
    """Pupil supports: spupil (pupdiam), mpupil (+2 px guard each side), ipupil (power-of-two)."""
    p_geom.ssize = int(2 ** np.ceil(np.log2(p_geom.pupdiam) + 1))
    p_geom.cent = p_geom.ssize / 2 - 0.5
    p_geom._p1 = int(np.ceil(p_geom.cent - p_geom.pupdiam / 2.0))
    p_geom._p2 = int(np.floor(p_geom.cent + p_geom.pupdiam / 2.0))
    p_geom.pupdiam = p_geom._p2 - p_geom._p1 + 1
    p_geom._n = p_geom.pupdiam + 2 * padding
    p_geom._n1 = p_geom._p1 - padding
    p_geom._n2 = p_geom._p2 + padding
    c = p_geom.pupdiam / 2.0 - 0.5
    p_geom._spupil = generic_pupil(p_geom.pupdiam, p_geom.pupdiam, p_tel, c, c).astype(np.float32)
    p_geom._ipupil = embed_centered(p_geom._spupil, p_geom.ssize).astype(np.float32)
    p_geom._mpupil = embed_centered(p_geom._spupil, p_geom._n).astype(np.float32)
    p_geom._apodizer = np.ones(p_geom._spupil.shape, dtype=np.int32)
    p_geom._pixsize = p_tel.diam / p_geom.pupdiam
    p_geom.is_init = True


def init_wfs_size(p_wfs, r0, p_tel):
    """Array sizes of one SH sensor (geom_init.py:168-340, SH branches only)."""
    if p_wfs.type != "sh":
        raise NotImplementedError("only Shack-Hartmann sensors are on the hot path")
    r0 = r0 * (p_wfs.Lambda * 2) ** (6.0 / 5)
    subapdiam = p_tel.diam / float(p_wfs.nxsub)
    lam = p_wfs.Lambda * 1.0e-6
    if p_wfs._pdiam <= 0:
        # free geometry (the sensor that defines the pupil sampling): 6 phase points per r0, >= 16
        pdiam = max(int(6 * subapdiam / r0), 16)
        if (pdiam * p_wfs.nxsub) % 2:
            pdiam += 1
        nrebin = max(2, int(2 * subapdiam * p_wfs.pixsize / lam / RAD2ARCSEC) + 1)
        Nfft = fft_goodsize(int(pdiam / subapdiam * nrebin / p_wfs.pixsize * RAD2ARCSEC * lam))
    else:
        pdiam = p_wfs._pdiam
        Nfft = fft_goodsize(2 * pdiam)
    qpixsize = (pdiam * lam / subapdiam * RAD2ARCSEC) / Nfft
    ratio = p_wfs.pixsize / qpixsize
    nrebin = int(ratio) + 1 if ratio - int(ratio) > 0.5 else int(ratio)
    pixsize = nrebin * qpixsize
    if pixsize * p_wfs.npix > qpixsize * Nfft:
        Ntot = fft_goodsize(int(pixsize * p_wfs.npix / qpixsize) + 1)
    else:
        Ntot = Nfft
    if Ntot % 2 != Nfft % 2:
        Ntot += 1
    p_wfs._pdiam = pdiam
    p_wfs.pixsize = pixsize
    p_wfs._qpixsize = qpixsize
    p_wfs._Nfft = Nfft
    p_wfs._Ntot = Ntot
    p_wfs._nrebin = nrebin
    p_wfs._subapd = p_tel.diam / p_wfs.nxsub


def compute_nphotons(ittime, optthroughput, diam, nxsub, zerop, gsmag):
    """Photons per full subaperture per frame, natural guide star (geom_init.py:343-407)."""
    if zerop == 0:
        zerop = 1.0e11
    return zerop * 10.0 ** (-0.4 * gsmag) * ittime * optthroughput * (diam / nxsub) ** 2.0


def nphotons_for_mags(ittime, optthroughput, diam, nxsub, zerop, gsmag):
    """float32 photon counts of compute_nphotons for a scalar or an array of guide-star magnitudes.  Each value is the
    scalar formula in float64 rounded once to float32, as the builder's _nphotons reaches aom_config.nphotons."""
    mags = np.asarray(gsmag, dtype=np.float64)
    out = np.array([compute_nphotons(ittime, optthroughput, diam, nxsub, zerop, float(m)) for m in mags.reshape(-1)],
                   dtype=np.float64)
    return out.astype(np.float32).reshape(mags.shape)


def init_sh_geom(p_wfs, r0, p_tel, p_geom, ittime):
    """Valid subapertures and the phasemap / binmap / halfxy tables (geom_init.py:622-811)."""
    nx, pd, npix = p_wfs.nxsub, p_wfs._pdiam, p_wfs.npix
    p_wfs.nPupils = 1
    start = np.linspace(0, p_geom.pupdiam, nx + 1)[:-1].astype(np.int64) + 2
    mp = p_geom._mpupil
    # illuminated fraction of every subaperture tile
    flux = np.array([[mp[i:i + pd, j:j + pd].sum() for j in start] for i in start],
                    dtype=np.float32) / pd ** 2.0
    isvalid = (flux >= p_wfs.fracsub).astype(np.int32)
    p_wfs._isvalid = isvalid
    p_wfs._nvalid = int(isvalid.sum())
    p_wfs._fluxPerSub = flux.copy()
    cols, rows = np.nonzero(isvalid.T)       # list order: outer over isvalid columns
    validx = rows.astype(np.int32)
    validy = cols.astype(np.int32)
    p_wfs._validpuppixx = validx * pd + 2
    p_wfs._validpuppixy = validy * pd + 2
    n = p_geom._n
    oy = start[validy]
    ox = start[validx]
    t = np.arange(pd)
    flat = (oy[None, None, :] + t[:, None, None]) * n + (ox[None, None, :] + t[None, :, None])
    p_wfs._phasemap = flat.reshape(pd * pd, p_wfs._nvalid).astype(np.int32)
    p_wfs._tile_origin = np.stack([oy, ox], axis=1).astype(np.int32)   # (row, col) per valid subap
    p_wfs._validsubsx = validx * npix
    p_wfs._validsubsy = validy * npix

    # half-pixel shift of the spot so that an even detector is centred between pixels
    ramp = np.linspace(0, 2 * np.pi, p_wfs._Nfft + 1)[:pd] / 2.0
    halfxy = ramp[None, :] + ramp[:, None]
    if npix % 2 == 1 and p_wfs._nrebin % 2 == 1:
        halfxy = np.zeros((pd, pd))
    p_wfs._halfxy = halfxy.astype(np.float32)

    if p_wfs._Ntot != p_wfs._Nfft:
        raise NotImplementedError("extended field of view (Ntot != Nfft) is outside the hot-path scope")
    p_wfs._hrmap = np.zeros((2, 2), dtype=np.int32)

    # binmap[:, p]: flat FFT-native indices of the nrebin^2 high-res pixels summed into pixel p
    Ntot, nr = p_wfs._Ntot, p_wfs._nrebin
    side = nr * npix
    lo = (Ntot - side) // 2 + (1 if side % 2 != Ntot % 2 else 0)
    if p_wfs.gsalt > 0:
        raise NotImplementedError("laser guide stars are outside the hot-path scope")
    # high-res coordinate (centred frame) -> FFT-native coordinate is a roll by Ntot//2
    c = np.arange(side)
    native = (lo + c + Ntot // 2) % Ntot                      # per axis
    lr = c // nr
    yy, xx = np.meshgrid(native, native, indexing="ij")
    ly, lx = np.meshgrid(lr, lr, indexing="ij")
    pix = (lx + ly * npix).reshape(-1)
    flat = (xx + yy * Ntot).reshape(-1)
    binmap = np.zeros((nr * nr, npix * npix), dtype=np.int64)
    order = np.lexsort((flat, pix))                            # ascending flat index inside a pixel
    binmap[:] = flat[order].reshape(npix * npix, nr * nr).T
    p_wfs._binmap = binmap.astype(np.int32)

    p_wfs._nphotons = compute_nphotons(ittime, p_wfs.optthroughput, p_tel.diam, nx, p_wfs.zerop,
                                       p_wfs.gsmag)
    # upload order of the illuminated fractions (wfs_init.py:145)
    p_wfs._fluxPerSub_list = flux.T[np.nonzero(isvalid.T)].astype(np.float32)


def init_wfs_geom(p_wfs, r0, p_tel, p_geom, ittime):
    if p_geom.pupdiam:
        pdiam = p_geom.pupdiam // p_wfs.nxsub + (1 if p_geom.pupdiam % p_wfs.nxsub > 0 else 0)
    else:
        pdiam = -1
    p_wfs._pdiam = pdiam
    init_wfs_size(p_wfs, r0, p_tel)
    if not p_geom.is_init:
        p_geom.pupdiam = p_wfs._pdiam * p_wfs.nxsub
        geom_init(p_geom, p_tel)
    init_sh_geom(p_wfs, r0, p_tel, p_geom, ittime)


def tel_init(p_geom, p_tel, r0, ittime, p_wfss):
    """Geometry of every sensor; the one with the most subapertures (LAST among ties, as
    np.argsort(...)[-1] picks it, geom_init.py:79-94) fixes the pupil sampling."""
    first = int(np.argsort([w.nxsub for w in p_wfss])[-1])
    init_wfs_geom(p_wfss[first], r0, p_tel, p_geom, ittime)
    for i, w in enumerate(p_wfss):
        if i != first:
            init_wfs_geom(w, r0, p_tel, p_geom, ittime)
