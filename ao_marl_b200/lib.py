"""ctypes binding of libaomarl.so (include/aomarl.h) and the `Simulator` that owns one GPU context.

PyTorch is used only as the owner of user-visible device memory and streams: every context buffer is
exposed as a zero-copy torch view (``__cuda_array_interface__``).  There is no CPU path: loading the
library or creating a context without a CUDA device raises.
"""
import ctypes
import os

import numpy as np

from .csrc import build as _build

MAX_LAYERS = 8


def LD(n):
    return (int(n) + 15) & ~15


class AomConfig(ctypes.Structure):
    _fields_ = (
        [("n_env", ctypes.c_int32), ("n", ctypes.c_int32), ("n_layers", ctypes.c_int32),
         ("screen_dim", ctypes.c_int32 * MAX_LAYERS), ("stencil_size", ctypes.c_int32 * MAX_LAYERS),
         ("deltax", ctypes.c_float * MAX_LAYERS), ("deltay", ctypes.c_float * MAX_LAYERS),
         ("amp", ctypes.c_float * MAX_LAYERS), ("wfs_xoff", ctypes.c_float * MAX_LAYERS),
         ("wfs_yoff", ctypes.c_float * MAX_LAYERS)]
        + [(k, ctypes.c_int32) for k in ("nxsub", "nvalid", "pdiam", "npix", "nfft", "nrebin")]
        + [(k, ctypes.c_float) for k in ("lambda_um", "nphotons", "noise", "pixsize", "cog_offset")]
        + [(k, ctypes.c_int32) for k in ("wfs_index", "pzt_nact", "stamp_size", "pzt_off", "pzt_pitch",
                                         "pzt_grid_n", "pzt_i1_0", "pzt_j1_0", "tt_dim", "tt_off",
                                         "nactu", "nslopes", "nmodes")]
        + [("gain", ctypes.c_float), ("delay", ctypes.c_int32), ("n_hist", ctypes.c_int32),
           ("state_modes", ctypes.c_int32), ("state_dim", ctypes.c_int32)]
        + [(k, ctypes.c_float) for k in ("env_act_scale", "env_act_bias", "pol_act_scale", "pol_act_bias",
                                         "log_sig_min", "log_sig_max")]
        + [(k, ctypes.c_int32) for k in ("n_agents", "actor_in", "actor_hidden", "actor_out", "action_dim")]
        + [("reward_factor", ctypes.c_float)])


TABLES = ["AB", "STENCIL", "MPUPIL", "HALFXY", "SUB_X0", "SUB_Y0", "FLUX", "STAMP1D", "ACT_MAP", "TT_PLANES",
          "CMAT", "V2M", "M2V", "FREEDOM", "ACTION_MAP", "STATE_MAP", "NORM_DM_MEAN", "NORM_DM_STD",
          "NORM_RES_MEAN", "NORM_RES_STD", "AGENT_IDX", "AGENT_ACT", "AGENT_REWARD", "ACTOR_W1", "ACTOR_B1",
          "ACTOR_W2", "ACTOR_B2", "ACTOR_WH", "ACTOR_BH", "GEO_PROJ", "GEO_SIFN", "DENOISER", "DENOISER_TC"]
T = {name: i for i, name in enumerate(TABLES)}
BUFFERS = ["SCREEN", "RING_OX", "RING_OY", "SLOPES", "ERR", "COM", "VOLTS", "BINCUBE", "PHASE", "MODES",
           "RES_MODES", "STATE", "REWARD", "ACTION", "ACTION_MEAN", "STREHL", "GEO_COM", "GEO_VOLTS", "STREHL_GEO", "GEO_PROJ",
           "EXT_COUNT"]
B = {name: i for i, name in enumerate(BUFFERS)}
_INT_BUFFERS = {"RING_OX", "RING_OY", "EXT_COUNT"}
OPTIONS = ["WFS_PATH", "GEMM_PATH", "TIME_WFS", "GEO", "DENOISE", "PUPIL_PATH", "KEEP_IMAGE", "STREHL", "STREHL_LAMBDA_NM", "EXTRUDE_PATH", "STREHL_PEAK", "PSF_NFFT", "DENOISE_PATH"]
O = {name: i for i, name in enumerate(OPTIONS)}

EXPORTS = ["aom_config_size", "aom_create", "aom_destroy", "aom_last_error", "aom_set_table", "aom_get_buffer",
           "aom_device_count_launches", "aom_set_option", "aom_check_device", "aom_reset", "aom_reset_envs", "aom_move_atmos", "aom_set_layer", "aom_set_layer_amp", "aom_set_layer_wind", "aom_comp_wfs_image", "aom_set_wfs_noise", "aom_set_wfs_noise_env", "aom_wfs_kernel", "aom_wfs_time_ms", "aom_raytrace_wfs",
           "aom_comp_strehl", "aom_reset_strehl", "aom_do_control_geo", "aom_apply_control_geo", "aom_denoise", "aom_set_bincube", "aom_do_centroids", "aom_do_centroids_geom", "aom_do_control", "aom_set_command", "aom_apply_control",
           "aom_set_gain", "aom_set_gain_env", "aom_set_loop", "aom_reset_dm", "aom_set_dm_volts", "aom_rl_control",
           "aom_state_begin", "aom_state_end", "aom_reward", "aom_actor_forward", "aom_step", "aom_gemm_tn",
           "aom_pixel_noise"]

_lib = None


def load_library():
    """Load (building first if the sources are newer) libaomarl.so; raises if it cannot be had."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB
    if _build.needs_build():
        try:
            _build.build()
        except Exception as exc:  # no nvcc on the box: use the shipped binary if there is one
            if not os.path.exists(path):
                raise RuntimeError("libaomarl.so is missing and cannot be built: %s" % exc)
    lib = ctypes.CDLL(path)
    vp, i32, f32, i64, u32, sz = (ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_int64,
                                  ctypes.c_uint32, ctypes.c_size_t)
    lib.aom_config_size.restype = sz
    lib.aom_last_error.restype = ctypes.c_char_p
    lib.aom_last_error.argtypes = [vp]
    lib.aom_create.argtypes = [ctypes.POINTER(AomConfig), ctypes.POINTER(vp)]
    lib.aom_destroy.argtypes = [vp]
    lib.aom_destroy.restype = None
    lib.aom_set_table.argtypes = [vp, i32, i32, vp, sz]
    lib.aom_get_buffer.argtypes = [vp, i32, i32, ctypes.POINTER(vp), ctypes.POINTER(sz)]
    lib.aom_device_count_launches.argtypes = [vp, ctypes.POINTER(ctypes.c_uint64)]
    lib.aom_set_option.argtypes = [vp, i32, i32]
    lib.aom_check_device.argtypes = [vp]
    lib.aom_reset.argtypes = [vp, vp, vp]
    lib.aom_reset_envs.argtypes = [vp, i32, vp, vp, vp]
    lib.aom_move_atmos.argtypes = [vp, vp]
    lib.aom_set_layer.argtypes = [vp, i32, f32, f32, f32]
    lib.aom_set_layer_amp.argtypes = [vp, i32, vp]
    lib.aom_set_layer_wind.argtypes = [vp, i32, vp, vp]
    lib.aom_comp_wfs_image.argtypes = [vp, i32, f32, vp]
    lib.aom_set_wfs_noise.argtypes = [vp, f32, f32]
    lib.aom_set_wfs_noise_env.argtypes = [vp, vp, vp]
    lib.aom_raytrace_wfs.argtypes = [vp, i32, vp]
    lib.aom_wfs_time_ms.argtypes = [vp, ctypes.POINTER(f32), ctypes.POINTER(i32)]
    lib.aom_wfs_kernel.argtypes = [vp]
    lib.aom_wfs_kernel.restype = ctypes.c_char_p
    lib.aom_comp_strehl.argtypes = [vp, i32, f32, i32, vp]
    lib.aom_reset_strehl.argtypes = [vp, vp]
    lib.aom_do_control_geo.argtypes = [vp, vp]
    lib.aom_apply_control_geo.argtypes = [vp, vp]
    lib.aom_denoise.argtypes = [vp, vp, vp, i64, vp]
    lib.aom_do_centroids_geom.argtypes = [vp, i32, ctypes.c_float, vp]
    lib.aom_set_bincube.argtypes = [vp, vp, vp]
    lib.aom_do_centroids.argtypes = [vp, vp]
    lib.aom_do_control.argtypes = [vp, vp]
    lib.aom_set_command.argtypes = [vp, vp, i32, vp]
    lib.aom_apply_control.argtypes = [vp, i32, vp]
    lib.aom_set_gain.argtypes = [vp, f32]
    lib.aom_set_gain_env.argtypes = [vp, vp]
    lib.aom_set_loop.argtypes = [vp, i32]
    lib.aom_reset_dm.argtypes = [vp, vp]
    lib.aom_set_dm_volts.argtypes = [vp, vp, i32, vp]
    lib.aom_rl_control.argtypes = [vp, vp, vp]
    lib.aom_state_begin.argtypes = [vp, vp]
    lib.aom_state_end.argtypes = [vp, vp]
    lib.aom_reward.argtypes = [vp, f32, vp]
    lib.aom_actor_forward.argtypes = [vp, i32, vp]
    lib.aom_step.argtypes = [vp, i32, i32, vp]
    lib.aom_gemm_tn.argtypes = [vp, vp, i32, vp, i32, vp, i32, i32, i32, i32, vp, i32, vp]
    lib.aom_pixel_noise.argtypes = [vp, vp, vp, i64, f32, i64, u32, u32, vp]
    if lib.aom_config_size() != ctypes.sizeof(AomConfig):
        raise RuntimeError("aom_config layout mismatch between aomarl.h and lib.py")
    _lib = lib
    return lib


class _DeviceView:
    """Zero-copy description of a device buffer for torch.as_tensor."""

    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False),
                                         "version": 2, "strides": None}


def pad_rows(a, ld=None):
    """[rows, k] -> float32 [rows, LD(k)] with zero padding (the layout every K-major operand uses)."""
    a = np.asarray(a, dtype=np.float32)
    ld = LD(a.shape[-1]) if ld is None else ld
    out = np.zeros(a.shape[:-1] + (ld,), dtype=np.float32)
    out[..., :a.shape[-1]] = a
    return np.ascontiguousarray(out)


def separable_factor(stamp, rtol=2e-6):
    """f with stamp ~= outer(f, f); raises when the actuator stamp is not separable."""
    stamp = np.asarray(stamp, dtype=np.float64)
    a, b = np.unravel_index(np.argmax(stamp), stamp.shape)
    peak = stamp[a, b]
    f = stamp[:, b] / np.sqrt(peak)
    err = np.abs(np.outer(f, f) - stamp).max() / peak
    if err > rtol or np.abs(stamp - stamp.T).max() > rtol * peak:
        raise NotImplementedError("actuator stamp is not separable/symmetric (err %.2e)" % err)
    return f.astype(np.float32)


def actuator_lattice(p_pzt):
    """(pitch, grid_n, i1_0, j1_0, act_map) of the square actuator lattice, or raises."""
    pitch = float(p_pzt._pitch)
    if not pitch.is_integer():
        raise NotImplementedError("non-integer actuator pitch %.4f px" % pitch)
    pitch = int(pitch)
    i1, j1 = np.asarray(p_pzt._i1, dtype=np.int64), np.asarray(p_pzt._j1, dtype=np.int64)
    base = min(i1.min(), j1.min())
    gx, gy = (i1 - base), (j1 - base)
    if (gx % pitch).any() or (gy % pitch).any():
        raise NotImplementedError("actuators are not on an integer lattice")
    gx //= pitch
    gy //= pitch
    grid_n = int(max(gx.max(), gy.max())) + 1
    amap = -np.ones(grid_n * grid_n, dtype=np.int32)
    amap[gy * grid_n + gx] = np.arange(i1.size, dtype=np.int32)
    return pitch, grid_n, int(base), int(base), amap


class Simulator:
    """One GPU context: E batched environments of one AO configuration.

    tables : ao_marl_b200.tables.StaticTables
    rl     : optional ao_marl_b200.rl.layout.RLLayout (state / action / agent tables)
    """

    def __init__(self, tables, n_env, rl=None, atmosphere=True, stream=None):
        import torch
        if not torch.cuda.is_available():
            raise RuntimeError("ao_marl_b200 needs a CUDA device: there is no CPU path")
        self.torch = torch
        self.lib = load_library()
        self.tables = t = tables
        self.n_env = int(n_env)
        self.rl = rl
        w = t.p_wfs
        cfg = AomConfig()
        cfg.n_env = self.n_env
        cfg.n = t.n
        cfg.n_layers = t.nscreens if atmosphere else 0
        for l in range(cfg.n_layers):
            cfg.screen_dim[l] = int(t.dim_screens[l])
            cfg.stencil_size[l] = int(len(t.istx[l]))
            cfg.deltax[l] = float(t.deltax[l])
            cfg.deltay[l] = float(t.deltay[l])
            cfg.amp[l] = float(np.float32(np.float32(t.r0_layers[l]) ** np.float32(-5.0 / 6.0)
                                          * np.float32(0.5 / (2 * np.pi))))
            cfg.wfs_xoff[l] = float(t.wfs_xoff[l])
            cfg.wfs_yoff[l] = float(t.wfs_yoff[l])
        cfg.nxsub, cfg.nvalid, cfg.pdiam, cfg.npix = w.nxsub, w._nvalid, w._pdiam, w.npix
        cfg.nfft, cfg.nrebin = w._Nfft, w._nrebin
        cfg.lambda_um, cfg.nphotons, cfg.noise = w.Lambda, w._nphotons, w.noise
        cfg.pixsize, cfg.cog_offset, cfg.wfs_index = t.cog_scale, t.cog_offset, t.wfs_index
        pitch, grid_n, i1_0, j1_0, amap = actuator_lattice(t.p_pzt)
        cfg.pzt_nact, cfg.stamp_size, cfg.pzt_off = t.p_pzt._ntotact, t.p_pzt._influsize, t.pzt_off
        cfg.pzt_pitch, cfg.pzt_grid_n, cfg.pzt_i1_0, cfg.pzt_j1_0 = pitch, grid_n, i1_0, j1_0
        cfg.tt_dim, cfg.tt_off = t.tt_dim, t.tt_off
        cfg.nactu, cfg.nslopes = t.nactu, t.nslopes
        cfg.nmodes = int(t.Btt.shape[1]) if getattr(t, "Btt", None) is not None else 0
        cfg.gain, cfg.delay = t.gain, int(round(t.delay))
        cfg.reward_factor = 1000.0
        if float(t.delay) not in (0.0, 1.0):
            raise NotImplementedError("controller delay must be 0 or 1 frame")
        if rl is not None:
            rl.fill_config(cfg)
        self.cfg = cfg
        self._ctx = ctypes.c_void_p()
        rc = self.lib.aom_create(ctypes.byref(cfg), ctypes.byref(self._ctx))
        if rc != 0:
            msg = self.lib.aom_last_error(self._ctx).decode()
            if self._ctx:
                self.lib.aom_destroy(self._ctx)
                self._ctx = ctypes.c_void_p()
            raise (ValueError if rc == -1 else RuntimeError)("aom_create: " + msg)
        self._stream = stream
        self._views = {}
        # sensor noise / photon count / integrator gain: common values and the per-environment float32 [E] arrays in
        # force (None: the common value), as the context holds them
        self.wfs_noise, self.wfs_nphotons = float(np.float32(cfg.noise)), float(np.float32(cfg.nphotons))
        self.wfs_noise_env = self.wfs_nphotons_env = self.gain_env = None
        # focal-plane grid of the target image (p_geom._ipupil, geom_init: 2^ceil(log2(pupdiam) + 1)) for the PSF core
        try:
            self.psf_nfft = int(np.asarray(t.config.p_geom._ipupil).shape[0])
        except Exception:
            self.psf_nfft = int(2 ** np.ceil(np.log2(max(int(t.n) - 4, 2)) + 1))
        self._check(self.lib.aom_set_option(self._ctx, O["PSF_NFFT"], self.psf_nfft), "aom_set_option")
        self._upload_static(amap)
        if cfg.nmodes:
            self.set_basis(t.Btt, t.P)
        if getattr(t, "cmat", None) is not None:
            self.set_command_matrix(t.cmat)
        if getattr(t, "geo_proj", None) is not None:
            self.set_geo(t.geo_proj, t.geo_sifn)
        if rl is not None:
            rl.upload(self)

    # -- plumbing ------------------------------------------------------------------------------
    def _check(self, rc, what):
        if rc != 0:
            msg = self.lib.aom_last_error(self._ctx).decode()
            raise (ValueError if rc == -1 else RuntimeError)("%s: %s" % (what, msg))

    @property
    def stream(self):
        s = self._stream if self._stream is not None else self.torch.cuda.current_stream()
        return ctypes.c_void_p(s.cuda_stream)

    def set_table(self, name, arr, index=0):
        arr = np.ascontiguousarray(arr)
        self._check(self.lib.aom_set_table(self._ctx, T[name], index, arr.ctypes.data_as(ctypes.c_void_p),
                                           arr.nbytes), "aom_set_table(%s)" % name)

    def buffer(self, name, index=0):
        """Flat zero-copy torch view of a context buffer."""
        key = (name, index)
        if key not in self._views:
            ptr, cnt = ctypes.c_void_p(), ctypes.c_size_t()
            self._check(self.lib.aom_get_buffer(self._ctx, B[name], index, ctypes.byref(ptr), ctypes.byref(cnt)),
                        "aom_get_buffer(%s)" % name)
            typ = "<i4" if name in _INT_BUFFERS else "<f4"
            self._views[key] = self.torch.as_tensor(_DeviceView(ptr.value, (cnt.value,), typ), device="cuda")
        return self._views[key]

    def rows(self, name, n, index=0):
        """[E, n] view (pad columns dropped) of a per-environment vector buffer."""
        flat = self.buffer(name, index)
        return flat.view(self.n_env, -1)[:, :n]

    def launches(self):
        n = ctypes.c_uint64()
        self.lib.aom_device_count_launches(self._ctx, ctypes.byref(n))
        return n.value

    DEFAULT_WFS_PATH = "umma_ws"
    WFS_PATHS = {"umma": 0, "umma_fast": 1, "simt": 2, "tensor_reg": 3, "tensor": 4, "tensor_fast": 5, "umma_ws": 6}

    def set_wfs_path(self, name):
        """Select the Shack-Hartmann frame kernel: 'umma_ws' (default: both DFT stages on tcgen05, specialised warps), 'umma'
        (the same pipeline fused in every warp; also serves noisy / image-keeping frames of the default), 'umma_fast', 'simt'
        (float32 FFT cross-check), 'tensor' / 'tensor_fast' / 'tensor_reg' (the round-1 mma.sync kernels)."""
        self._check(self.lib.aom_set_option(self._ctx, O["WFS_PATH"], self.WFS_PATHS[name]), "aom_set_option")

    def wfs_kernel(self):
        """Name of the kernel the next frame launches (and, via last_error, why the staged one is not used)."""
        return self.lib.aom_wfs_kernel(self._ctx).decode()

    def time_wfs(self, on=True):
        """Bracket every sensor-kernel launch with CUDA events (read the mean with wfs_time_ms)."""
        self._check(self.lib.aom_set_option(self._ctx, O["TIME_WFS"], 1 if on else 0), "aom_set_option")

    def wfs_time_ms(self):
        """(mean device time in ms, number of launches) of the sensor kernel since the last call."""
        ms, n = ctypes.c_float(), ctypes.c_int()
        self._check(self.lib.aom_wfs_time_ms(self._ctx, ctypes.byref(ms), ctypes.byref(n)), "aom_wfs_time_ms")
        return float(ms.value), int(n.value)

    def set_extrude_path(self, name):
        """Contraction behind the screen extrusion: 'i8' (default: exact integer digits on tcgen05) or 'ffma' (float32)."""
        self._check(self.lib.aom_set_option(self._ctx, O["EXTRUDE_PATH"], {"i8": 0, "ffma": 1}[name]), "aom_set_option")

    GEMM_PATHS = {"tcgen05": 0, "simt": 1, "tf32": 2}

    def set_gemm_path(self, name):
        """Select the GEMM kernel of the env-batched contractions: 'tcgen05' (default) or 'simt'."""
        self._check(self.lib.aom_set_option(self._ctx, O["GEMM_PATH"], self.GEMM_PATHS[name]), "aom_set_option")

    def check_device(self):
        """Synchronise and raise if a kernel reported an asynchronous error."""
        self._check(self.lib.aom_check_device(self._ctx), "aom_check_device")

    def close(self):
        if self._ctx:
            self._views.clear()
            self.lib.aom_destroy(self._ctx)
            self._ctx = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- tables --------------------------------------------------------------------------------
    def _upload_static(self, amap):
        t, w = self.tables, self.tables.p_wfs
        for l in range(self.cfg.n_layers):
            ab = np.concatenate([t.A[l], t.B[l]], axis=1)
            self.set_table("AB", pad_rows(ab), l)
            self.set_table("STENCIL", np.asarray(t.istx[l], dtype=np.int32), l)
        self.set_table("MPUPIL", t.mpupil.astype(np.float32))
        self.set_table("HALFXY", w._halfxy.astype(np.float32))
        self.set_table("SUB_X0", w._tile_origin[:, 1].astype(np.int32))
        self.set_table("SUB_Y0", w._tile_origin[:, 0].astype(np.int32))
        self.set_table("FLUX", w._fluxPerSub_list.astype(np.float32))
        self.set_table("STAMP1D", separable_factor(t.p_pzt._influ[:, :, 0]))
        self.set_table("ACT_MAP", amap)
        self.set_table("TT_PLANES", np.ascontiguousarray(t.p_tt._influ.transpose(2, 1, 0), dtype=np.float32))

    def set_basis(self, Btt, P):
        self.set_table("M2V", pad_rows(Btt))
        self.set_table("V2M", pad_rows(P))

    def set_command_matrix(self, cmat):
        cmat = np.asarray(cmat, dtype=np.float32)
        if cmat.shape != (self.cfg.nactu, self.cfg.nslopes):
            raise ValueError("Dimension mismatch")
        self.set_table("CMAT", pad_rows(cmat))
        self.cmat = cmat

    def env_seeds(self, seed):
        """int64 [E] seeds from a scalar (environment e gets seed + e, so E == 1 keeps the reference's
        single stream) or from an explicit array."""
        seed = np.asarray(seed, dtype=np.int64)
        if seed.ndim == 0:
            return seed + np.arange(self.n_env, dtype=np.int64)
        if seed.shape != (self.n_env,):
            raise ValueError("Dimension mismatch")
        return seed

    # -- ops (thin, asynchronous on the current stream) -----------------------------------------
    def reset(self, seeds):
        seeds = np.ascontiguousarray(np.broadcast_to(np.asarray(seeds, dtype=np.int64), (self.n_env,)))
        self._check(self.lib.aom_reset(self._ctx, seeds.ctypes.data_as(ctypes.c_void_p), self.stream), "aom_reset")

    def reset_envs(self, envs, seeds):
        """Restart the environments `envs` (distinct indices, int [n]) with `seeds` (int [n]) while the others run on
        (aom_reset_envs).  Their next step acts as the linear step after a reset: its rl half-step is ignored, its reward
        is 0 and the state it leaves is their s0.  Set the new episode's conditions first (set_layer_amp / set_layer_wind
        with [E] arrays): the start-up of the screens already uses them."""
        envs, seeds = np.asarray(envs), np.asarray(seeds)
        if envs.ndim != 1 or seeds.shape != envs.shape:
            raise ValueError("reset_envs: envs and seeds must be 1-D arrays of the same length")
        if envs.size and (envs.dtype.kind not in "iu" or seeds.dtype.kind not in "iu"):
            raise TypeError("reset_envs: envs and seeds must be integer arrays")
        if envs.size and (envs.min() < 0 or envs.max() >= self.n_env):
            raise ValueError("reset_envs: environment index out of range [0, %d)" % self.n_env)
        if np.unique(envs).size != envs.size:
            raise ValueError("reset_envs: duplicate environment index")
        envs = np.ascontiguousarray(envs, dtype=np.int32)
        seeds = np.ascontiguousarray(seeds, dtype=np.int64)
        self._check(self.lib.aom_reset_envs(self._ctx, int(envs.size), envs.ctypes.data_as(ctypes.c_void_p),
                                            seeds.ctypes.data_as(ctypes.c_void_p), self.stream), "aom_reset_envs")

    def move_atmos(self):
        self._check(self.lib.aom_move_atmos(self._ctx, self.stream), "aom_move_atmos")

    def set_layer(self, layer, deltax, deltay, amp):
        self._check(self.lib.aom_set_layer(self._ctx, int(layer), float(deltax), float(deltay), float(amp)),
                    "aom_set_layer")

    def set_layer_wind(self, layer, deltax, deltay):
        """Wind step of one layer per environment (pixels / frame, float [E] each; a scalar broadcasts); None, None
        returns the layer to its common wind (set_layer).  Accumulators continue from the common one."""
        if deltax is None and deltay is None:
            self._check(self.lib.aom_set_layer_wind(self._ctx, int(layer), None, None), "aom_set_layer_wind")
            return
        dx = np.ascontiguousarray(np.broadcast_to(np.asarray(deltax, dtype=np.float32), (self.n_env,)))
        dy = np.ascontiguousarray(np.broadcast_to(np.asarray(deltay, dtype=np.float32), (self.n_env,)))
        self._check(self.lib.aom_set_layer_wind(self._ctx, int(layer), dx.ctypes.data_as(ctypes.c_void_p),
                                                dy.ctypes.data_as(ctypes.c_void_p)), "aom_set_layer_wind")

    def set_layer_amp(self, layer, amp):
        """Innovation amplitude of one layer per environment (float [E]); None restores the common amplitude."""
        if amp is None:
            self._check(self.lib.aom_set_layer_amp(self._ctx, int(layer), None), "aom_set_layer_amp")
            return
        amp = np.ascontiguousarray(np.broadcast_to(np.asarray(amp, dtype=np.float32), (self.n_env,)))
        self._check(self.lib.aom_set_layer_amp(self._ctx, int(layer), amp.ctypes.data_as(ctypes.c_void_p)), "aom_set_layer_amp")

    def _env_array(self, x, what):
        """float32 [E] from a scalar (broadcast) or a length-E sequence; ValueError otherwise."""
        a = np.asarray(x, dtype=np.float32)
        if a.ndim == 0:
            a = np.full(self.n_env, a, dtype=np.float32)
        if a.shape != (self.n_env,):
            raise ValueError("%s: expected a scalar or %d values, got shape %s" % (what, self.n_env, a.shape))
        return np.ascontiguousarray(a)

    def set_wfs_noise(self, noise, nphotons=None):
        """Common sensor noise (<0 none, 0 photon, >0 photon + read noise in e-) and photons per subaperture and frame
        (None: unchanged).  aom_step and comp_wfs_image(noise=None) use them; per-environment values stay in force."""
        nph = self.wfs_nphotons if nphotons is None else nphotons
        self._check(self.lib.aom_set_wfs_noise(self._ctx, float(noise), float(nph)), "aom_set_wfs_noise")
        self.wfs_noise, self.wfs_nphotons = float(np.float32(noise)), float(np.float32(nph))

    def set_wfs_noise_env(self, noise=None, nphotons=None):
        """Sensor noise and photon count per environment (scalar or [E] each; None: that quantity's common value).  A
        noisy frame then draws each environment's own noise, and every frame is scaled by its own photon count."""
        P = lambda a: None if a is None else a.ctypes.data_as(ctypes.c_void_p)
        n = None if noise is None else self._env_array(noise, "set_wfs_noise_env(noise)")
        f = None if nphotons is None else self._env_array(nphotons, "set_wfs_noise_env(nphotons)")
        self._check(self.lib.aom_set_wfs_noise_env(self._ctx, P(n), P(f)), "aom_set_wfs_noise_env")
        self.wfs_noise_env, self.wfs_nphotons_env = n, f

    def comp_wfs_image(self, atmos=True, dms=True, keep_image=False, noise=None, advance_frame=True):
        """noise None: the common noise, or with per-environment noise in force a noisy frame (each environment's own);
        a value < 0: noise-free for every environment."""
        flags = (1 if atmos else 0) | (2 if dms else 0) | (4 if keep_image else 0) | (0 if advance_frame else 8)
        if noise is None:
            noise = 0.0 if self.wfs_noise_env is not None else self.wfs_noise
        noise = float(noise)
        self._check(self.lib.aom_comp_wfs_image(self._ctx, flags, noise, self.stream), "aom_comp_wfs_image")

    def do_centroids_geom(self, atmos=True, dms=True, geo=False):
        """Geometric slopes (mean phase gradient per subaperture) of the sensor-direction phase -> SLOPES."""
        flags = (1 if atmos else 0) | (2 if dms else 0) | (0x100 if geo else 0)
        alpha = 0.206265 / float(self.tables.p_wfs._subapd)
        self._check(self.lib.aom_do_centroids_geom(self._ctx, flags, alpha, self.stream), "aom_do_centroids_geom")

    def raytrace_wfs(self, atmos=True, dms=True, geo=False):
        flags = (1 if atmos else 0) | (2 if dms else 0) | (0x100 if geo else 0)
        self._check(self.lib.aom_raytrace_wfs(self._ctx, flags, self.stream), "aom_raytrace_wfs")
        return self.buffer("PHASE").view(self.n_env, self.cfg.n, self.cfg.n)

    def comp_strehl(self, lambda_um, atmos=True, dms=True, accumulate=True, geo=False, phase="both", peak=False):
        """Pupil phase variance -> AOM_B_STREHL [E, 4] = (SE, LE, variance, mean variance); geo=True: the target
        behind the geometric controller's mirrors (AOM_B_STREHL_GEO).  phase: "both" (trace now and publish), "trace"
        (TargetCompass.raytrace: sweep now, keep pending) or "publish" (comp_tar_image / comp_strehl on the pending sums).
        peak: SE / LE from the brightest pixel of the 3 x 3 PSF core with a three-point fit (comp_strehl(do_fit=True))
        instead of the on-axis pixel."""
        flags = ((1 if atmos else 0) | (2 if dms else 0) | (0x100 if geo else 0) | (0x800 if peak else 0)
                 | {"both": 0, "trace": 0x200, "publish": 0x400}[phase])
        self._check(self.lib.aom_comp_strehl(self._ctx, flags, float(lambda_um), 1 if accumulate else 0, self.stream),
                    "aom_comp_strehl")
        return self.buffer("STREHL_GEO" if geo else "STREHL").view(self.n_env, 4)

    def set_geo(self, proj, sifn):
        """Upload the geometric controller's tables (ao_marl_b200.init.geo.build_geo)."""
        proj = np.asarray(proj, dtype=np.float32)
        if proj.shape != (self.cfg.nactu, self.cfg.nactu) or np.shape(sifn) != (self.cfg.nactu,):
            raise ValueError("Dimension mismatch")
        self.set_table("GEO_PROJ", pad_rows(proj))
        self.set_table("GEO_SIFN", np.asarray(sifn, dtype=np.float32))

    def do_control_geo(self):
        """rtc.do_control(geo controller, sources=target): AOM_B_GEO_COM = least-squares mirror fit of the turbulence."""
        self._check(self.lib.aom_do_control_geo(self._ctx, self.stream), "aom_do_control_geo")
        return self.rows("GEO_COM", self.cfg.nactu)

    def apply_control_geo(self):
        self._check(self.lib.aom_apply_control_geo(self._ctx, self.stream), "aom_apply_control_geo")

    def set_pupil_path(self, name):
        """Kernels behind comp_strehl / do_control_geo: 'sweep' (default) or 'pixel' (cross-check path)."""
        self._check(self.lib.aom_set_option(self._ctx, O["PUPIL_PATH"], {"sweep": 0, "pixel": 1}[name]), "aom_set_option")

    def step_with_denoiser(self, on=True):
        """aom_step runs the fused denoiser between the sensor frame and the centroider (AOM_OPT_DENOISE)."""
        self._check(self.lib.aom_set_option(self._ctx, O["DENOISE"], 1 if on else 0), "aom_set_option")

    def step_keeps_image(self, on=True):
        """aom_step keeps every frame's detector cube in AOM_B_BINCUBE (AOM_OPT_KEEP_IMAGE)."""
        self._check(self.lib.aom_set_option(self._ctx, O["KEEP_IMAGE"], 1 if on else 0), "aom_set_option")

    def strehl_from_peak(self, on=True):
        """Every Strehl evaluation (aom_comp_strehl and the one inside aom_step) uses the fitted PSF-core peak."""
        self._check(self.lib.aom_set_option(self._ctx, O["STREHL_PEAK"], 1 if on else 0), "aom_set_option")

    def step_with_strehl(self, on=True, lambda_um=1.65, pure_delay_0=False):
        """aom_step evaluates the target Strehl every frame, as the reference's next_part_two does by default
        (compute_tar_psf=True, rlSupervisor.py:944-947): with the voltages the target was traced with in next_part_one, or
        (pure_delay_0, the reference's modification_online) re-traced after apply_control."""
        self._check(self.lib.aom_set_option(self._ctx, O["STREHL_LAMBDA_NM"], int(round(lambda_um * 1000))), "aom_set_option")
        self._check(self.lib.aom_set_option(self._ctx, O["STREHL"], (2 if pure_delay_0 else 1) if on else 0), "aom_set_option")

    def step_with_geo(self, on=True):
        """aom_step also runs the geometric controller every frame (AOM_OPT_GEO)."""
        self._check(self.lib.aom_set_option(self._ctx, O["GEO"], 1 if on else 0), "aom_set_option")

    def reset_strehl(self):
        self._check(self.lib.aom_reset_strehl(self._ctx, self.stream), "aom_reset_strehl")

    def set_denoiser(self, packed, packed_tc=None):
        """Upload the denoiser's parameters (ao_marl_b200.denoiser.pack_weights; packed_tc = pack_weights_tc's
        (weight tiles, float parameters) for the tensor-core kernel)."""
        self.set_table("DENOISER", np.asarray(packed, dtype=np.float32))
        if packed_tc is not None:
            tiles, prm = packed_tc
            blob = np.concatenate([np.asarray(prm, np.float32).view(np.uint8), np.asarray(tiles, np.uint16).view(np.uint8)])
            self.set_table("DENOISER_TC", blob)

    def set_denoise_path(self, name):
        """'tcgen05' (default) or 'simt' (float32 FFMA cross-check kernel)."""
        self._check(self.lib.aom_set_option(self._ctx, O["DENOISE_PATH"], {"tcgen05": 0, "simt": 1}[name]), "aom_set_option")

    def denoise(self, cube=None, out=None):
        """Fused CNN denoiser.  cube None: the last frame's detector cube, in place, feeding the next do_centroids;
        otherwise a CUDA float32 tensor [..., 256] (or [..., 16, 16]), returns the denoised tensor of the same shape."""
        if cube is None:
            self._check(self.lib.aom_denoise(self._ctx, None, None, 0, self.stream), "aom_denoise")
            return self.buffer("BINCUBE").view(self.n_env, self.cfg.nvalid, 256)
        torch = self.torch
        x = cube if (cube.is_cuda and cube.dtype == torch.float32 and cube.is_contiguous()) else \
            cube.to(device="cuda", dtype=torch.float32).contiguous()
        if x.numel() % 256:
            raise ValueError("Dimension mismatch")
        y = torch.empty_like(x) if out is None else out
        if x.numel() == 0:
            return y                                         # an empty tensor has no device pointer to hand over
        self._check(self.lib.aom_denoise(self._ctx, ctypes.c_void_p(x.data_ptr()), ctypes.c_void_p(y.data_ptr()),
                                         x.numel() // 256, self.stream), "aom_denoise")
        return y

    def set_bincube(self, cube):
        self._cube_keepalive = cube
        self._check(self.lib.aom_set_bincube(self._ctx, ctypes.c_void_p(cube.data_ptr()), self.stream),
                    "aom_set_bincube")

    def do_centroids(self):
        self._check(self.lib.aom_do_centroids(self._ctx, self.stream), "aom_do_centroids")

    def do_control(self):
        self._check(self.lib.aom_do_control(self._ctx, self.stream), "aom_do_control")

    def _rows_arg(self, x, n):
        torch = self.torch
        x = torch.as_tensor(x, dtype=torch.float32, device="cuda")
        if x.dim() == 1:
            x = x.unsqueeze(0).expand(self.n_env, -1)
        if x.shape[0] != self.n_env or x.shape[1] != n:
            raise ValueError("Dimension mismatch")
        return x.contiguous()

    def set_command(self, com):
        x = self._rows_arg(com, self.cfg.nactu)
        self._check(self.lib.aom_set_command(self._ctx, ctypes.c_void_p(x.data_ptr()), x.shape[1], self.stream),
                    "aom_set_command")

    def set_dm_volts(self, volts):
        x = self._rows_arg(volts, self.cfg.nactu)
        self._check(self.lib.aom_set_dm_volts(self._ctx, ctypes.c_void_p(x.data_ptr()), x.shape[1], self.stream),
                    "aom_set_dm_volts")

    def apply_control(self, comp_voltage=True):
        self._check(self.lib.aom_apply_control(self._ctx, int(bool(comp_voltage)), self.stream), "aom_apply_control")

    def set_gain(self, g):
        """Integrator gain: a scalar sets the common gain (per-environment gains stay in force, as aom_set_gain); an [E]
        array sets one gain per environment (set_gain_env)."""
        if np.ndim(g) == 0:
            self._check(self.lib.aom_set_gain(self._ctx, float(g)), "aom_set_gain")
        else:
            self.set_gain_env(g)

    def set_gain_env(self, g):
        """One integrator gain per environment ([E]; a scalar broadcasts); None: back to the common gain."""
        a = None if g is None else self._env_array(g, "set_gain_env")
        self._check(self.lib.aom_set_gain_env(self._ctx, None if a is None else a.ctypes.data_as(ctypes.c_void_p)),
                    "aom_set_gain_env")
        self.gain_env = a

    def set_loop(self, closed):
        self._check(self.lib.aom_set_loop(self._ctx, int(bool(closed))), "aom_set_loop")

    def reset_dm(self):
        self._check(self.lib.aom_reset_dm(self._ctx, self.stream), "aom_reset_dm")

    def rl_control(self, action=None):
        ptr = ctypes.c_void_p(0)
        if action is not None:
            a = self.torch.as_tensor(action, dtype=self.torch.float32, device="cuda")
            if a.dim() == 1:
                a = a.unsqueeze(0).expand(self.n_env, -1)
            if a.shape != (self.n_env, self.cfg.action_dim):
                raise ValueError("Dimension mismatch")
            self.rows("ACTION", self.cfg.action_dim).copy_(a)
        self._check(self.lib.aom_rl_control(self._ctx, ptr, self.stream), "aom_rl_control")

    def state_begin(self):
        self._check(self.lib.aom_state_begin(self._ctx, self.stream), "aom_state_begin")

    def state_end(self):
        self._check(self.lib.aom_state_end(self._ctx, self.stream), "aom_state_end")

    def reward(self, factor=1000.0):
        self._check(self.lib.aom_reward(self._ctx, float(factor), self.stream), "aom_reward")

    def actor_forward(self, eval_mode=False):
        self._check(self.lib.aom_actor_forward(self._ctx, int(bool(eval_mode)), self.stream), "aom_actor_forward")

    def step(self, mode=0, eval_mode=False, atmos_done=False):
        """One env-step of the whole batch.  atmos_done: the caller already ran move_atmos for this step (for example
        on a second stream while the actions were on their way from the host)."""
        self._check(self.lib.aom_step(self._ctx, int(mode) | (8 if atmos_done else 0), int(bool(eval_mode)), self.stream),
                    "aom_step")

    def gemm_tn(self, A, Bm, bias=None, relu=False):
        """C = A . Bm^T on padded device tensors [M, ld] / [N, ld]; returns [M, LD(N)] (test entry point)."""
        torch = self.torch
        M, N = A.shape[0], Bm.shape[0]
        C = torch.empty((M, LD(N)), dtype=torch.float32, device="cuda")
        bp = ctypes.c_void_p(bias.data_ptr()) if bias is not None else ctypes.c_void_p(0)
        self._check(self.lib.aom_gemm_tn(self._ctx, ctypes.c_void_p(A.data_ptr()), A.shape[1],
                                         ctypes.c_void_p(Bm.data_ptr()), Bm.shape[1], ctypes.c_void_p(C.data_ptr()),
                                         C.shape[1], M, N, min(A.shape[1], Bm.shape[1]), bp, int(relu), self.stream),
                    "aom_gemm_tn")
        return C

    def pixel_noise(self, lam, noise, seed, frame, wfs):
        out = self.torch.empty_like(lam)
        self._check(self.lib.aom_pixel_noise(self._ctx, ctypes.c_void_p(lam.data_ptr()), ctypes.c_void_p(out.data_ptr()),
                                             lam.numel(), float(noise), int(seed), int(frame), int(wfs), self.stream),
                    "aom_pixel_noise")
        return out
