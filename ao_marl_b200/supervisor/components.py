"""Component objects of the supervisor: the same method names and argument meaning as the reference's
shesha/supervisor/components/{atmos,wfs,dm,rtc,target,telescope}Compass.py, each a thin stream-ordered
call into libaomarl.so through `ao_marl_b200.lib.Simulator`.

Every per-environment array carries a leading batch dimension E; with E == 1 getters return numpy
arrays of the reference's shapes (float32), otherwise device tensors [E, ...] (no host copy).
"""
import numpy as np

from ..init.geom import DEG2RAD, nphotons_for_mags


class _Base:
    def __init__(self, sim, config):
        self._sim = sim
        self._config = config

    def _out(self, t):
        """[E, ...] device tensor -> reference-shaped numpy when E == 1."""
        if self._sim.n_env == 1:
            return t[0].detach().cpu().numpy()
        return t


class TelescopeB200(_Base):
    pass


class AtmosB200(_Base):
    """atmosCompass.py:50-161"""

    def __init__(self, sim, config):
        super().__init__(sim, config)
        self.is_enable = True

    def enable_atmos(self, enable):
        self.is_enable = enable

    def move_atmos(self):
        self._sim.move_atmos()

    def reset_turbu(self, seed):
        """Reseed and regenerate every layer.  `seed` may be a scalar (environment e gets seed + e, Simulator.env_seeds,
        so that E == 1 reproduces the reference's single stream) or an int64 array [E]."""
        self._sim.reset(self._sim.env_seeds(seed))

    def _amp(self, layer, r0=None):
        a = self._config.p_atmos
        r0_px = (a.r0 if r0 is None else np.asarray(r0, dtype=np.float64)) / (a.frac[layer] ** (3.0 / 5.0) * a.pupixsize)
        amp = np.float32(r0_px) ** np.float32(-5.0 / 6.0) * np.float32(0.5 / (2 * np.pi))
        return float(np.float32(amp)) if np.ndim(amp) == 0 else np.asarray(amp, dtype=np.float32)

    def set_r0(self, r0, *, reset_seed=-1):
        """atmosCompass.py:79-101.  `r0` may be a scalar (every environment) or an array [E]: one seeing condition per
        environment of the batch (the reference changes the r0 of its single simulator at run time, train_rpc.py:429-449)."""
        a = self._config.p_atmos
        if np.ndim(r0) == 0:
            a.r0 = float(r0)
            for l in range(a.nscreens):
                self._sim.set_layer(l, a._deltax[l], a._deltay[l], self._amp(l))
                self._sim.set_layer_amp(l, None)
        else:
            r0 = np.asarray(r0, dtype=np.float64)
            if r0.shape != (self._sim.n_env,):
                raise ValueError("Dimension mismatch")
            for l in range(a.nscreens):
                self._sim.set_layer_amp(l, self._amp(l, r0))
        if reset_seed != -1:
            seed = np.random.randint(int(1e4)) if reset_seed == 0 else reset_seed
            self._sim.reset(self._sim.env_seeds(1234 + seed))

    def _wind_step(self, windspeed, winddir):
        """(deltax, deltay) in pixels per frame of one wind speed (m/s) and direction (degrees)."""
        c = self._config
        lin = c.p_geom.pupdiam / c.p_tel.diam * windspeed * np.cos(DEG2RAD * c.p_geom.zenithangle) * c.p_loop.ittime
        return lin * np.sin(DEG2RAD * winddir + np.pi), lin * np.cos(DEG2RAD * winddir + np.pi)

    def set_wind(self, screen_index, *, windspeed=None, winddir=None):
        """atmosCompass.py:79-135.  `windspeed` and `winddir` may each be a scalar or an array [E] (one wind per
        environment of the batch; a scalar broadcasts against the other, an omitted one is the layer's current value).
        Both scalar: the layer's common wind, recorded in p_atmos as in the reference, and any per-environment wind of
        the layer is dropped.  Otherwise the winds go to the environments only (p_atmos keeps the common wind); every
        environment continues from the layer's current sub-pixel position."""
        a = self._config.p_atmos
        l = screen_index
        if np.ndim(windspeed) == 0 and np.ndim(winddir) == 0:
            if windspeed is not None:
                a.windspeed[l] = windspeed
            if winddir is not None:
                a.winddir[l] = winddir
            a._deltax[l], a._deltay[l] = self._wind_step(a.windspeed[l], a.winddir[l])
            # a change of sign needs no new stencil here: mirroring is index arithmetic in the kernels
            self._sim.set_layer(l, a._deltax[l], a._deltay[l], self._amp(l))
            self._sim.set_layer_wind(l, None, None)
            return
        E = self._sim.n_env
        speed = np.asarray(a.windspeed[l] if windspeed is None else windspeed, dtype=np.float64)
        direction = np.asarray(a.winddir[l] if winddir is None else winddir, dtype=np.float64)
        for v in (speed, direction):
            if v.ndim != 0 and v.shape != (E,):
                raise ValueError("Dimension mismatch")
        speed, direction = np.broadcast_to(speed, (E,)), np.broadcast_to(direction, (E,))
        # element by element with the scalar formula on values of p_atmos' own types (float32 in the parameter files):
        # the same operations as a common wind of that value, so each environment moves exactly as such a batch would
        ts, td = np.asarray(a.windspeed).dtype.type, np.asarray(a.winddir).dtype.type
        steps = [self._wind_step(ts(speed[e]), td(direction[e])) for e in range(E)]
        self._sim.set_layer_wind(l, np.array([d[0] for d in steps], np.float32), np.array([d[1] for d in steps], np.float32))

    def get_atmos_layer(self, indx):
        """Logical (un-rotated) screen(s) of layer `indx`."""
        import torch
        sim = self._sim
        n = int(sim.cfg.screen_dim[indx])
        scr = sim.buffer("SCREEN", indx).view(sim.n_env, n, n)
        ox = sim.buffer("RING_OX", indx).cpu().numpy()
        oy = sim.buffer("RING_OY", indx).cpu().numpy()
        out = torch.stack([torch.roll(scr[e], (-int(oy[e]), -int(ox[e])), dims=(0, 1)) for e in range(sim.n_env)])
        return self._out(out)


class WfsB200(_Base):
    """wfsCompass.py + sourceCompass.py:54-85.  raytrace only records what the next frame must contain; the
    fused kernel evaluates the phase per subaperture inside compute_wfs_image."""

    def __init__(self, sim, config, wfs_index=0):
        super().__init__(sim, config)
        self._index = wfs_index
        self._atm = False
        self._dms = False
        self.keep_image = False

    def _chk(self, i):
        if i != self._index:
            raise NotImplementedError("only the sensor driving controller 0 is on the hot path")

    def raytrace(self, index, *, tel=None, atm=None, dms=None, ncpa=True, reset=True):
        self._chk(index)
        if reset:
            self._atm = self._dms = False
        if atm is not None and getattr(atm, "is_enable", True):
            self._atm = True
        if dms is not None:
            self._dms = True

    def compute_wfs_image(self, wfs_index, *, noise=True):
        self._chk(wfs_index)
        # noise=True: the common noise, or each environment's own (Simulator.comp_wfs_image(noise=None))
        self._sim.comp_wfs_image(atmos=self._atm, dms=self._dms, keep_image=self.keep_image,
                                 noise=None if noise else -1.0)

    def set_noise(self, wfs_index, noise, *, seed=1234):
        """Sensor noise (<0 none, 0 photon, >0 photon + read noise in e-): a scalar sets the common value and drops
        per-environment noise, an [E] array sets one value per environment.  Both reach aom_step and compute_wfs_image."""
        self._chk(wfs_index)
        sim = self._sim
        if np.ndim(noise) == 0:
            sim.set_wfs_noise(float(noise))
            sim.set_wfs_noise_env(noise=None, nphotons=sim.wfs_nphotons_env)
            self._config.p_wfss[wfs_index].noise = noise
        else:
            sim.set_wfs_noise_env(noise=noise, nphotons=sim.wfs_nphotons_env)

    def set_gs_mag(self, wfs_index, mag):
        """Guide-star magnitude, scalar or [E]: photons per subaperture and frame from compute_nphotons with this
        sensor's integration time, throughput, telescope diameter, nxsub and zero point (geom_init.py:343-407).  A scalar
        sets the common photon count and drops per-environment ones; an [E] array sets one per environment."""
        self._chk(wfs_index)
        c, sim = self._config, self._sim
        w = c.p_wfss[wfs_index]
        nph = nphotons_for_mags(c.p_loop.ittime, w.optthroughput, c.p_tel.diam, w.nxsub, w.zerop, mag)
        if np.ndim(mag) == 0:
            sim.set_wfs_noise(sim.wfs_noise, float(nph))
            sim.set_wfs_noise_env(noise=sim.wfs_noise_env, nphotons=None)
        else:
            sim.set_wfs_noise_env(noise=sim.wfs_noise_env, nphotons=nph)

    def reset_noise(self, seed):
        """Noise streams are keyed by the environment seed and the frame counter: reseeding happens in
        AtmosB200.reset_turbu (one aom_reset covers both, rlSupervisor.py:240-241)."""

    def get_wfs_phase(self, wfs_index):
        self._chk(wfs_index)
        return self._out(self._sim.raytrace_wfs(atmos=self._atm, dms=self._dms))

    def get_bincube(self):
        """[E, nvalid, npix, npix] spots of the last frame computed with keep_image=True."""
        c = self._sim.cfg
        return self._sim.buffer("BINCUBE").view(self._sim.n_env, c.nvalid, c.npix, c.npix)

    def get_wfs_image(self, wfs_index):
        """Detector mosaic (rlSupervisor.py:857-874 layout: spot k at [validsubsy[k], validsubsx[k]] in [y, x])."""
        import torch
        self._chk(wfs_index)
        c = self._sim.cfg
        w = self._config.p_wfss[wfs_index]
        cube = self.get_bincube()
        side = c.nxsub * c.npix
        img = torch.zeros((self._sim.n_env, side, side), device=cube.device)
        for k in range(c.nvalid):
            x0, y0 = int(w._validsubsx[k]), int(w._validsubsy[k])
            img[:, y0:y0 + c.npix, x0:x0 + c.npix] = cube[:, k]
        return self._out(img)

    def set_bincube(self, cube):
        """Replace the detector spots before centroiding (denoiser path, rlSupervisor.py:876-891)."""
        import torch
        c = self._sim.cfg
        cube = torch.as_tensor(cube, dtype=torch.float32, device="cuda").reshape(self._sim.n_env, c.nvalid, 256)
        self._sim.set_bincube(cube.contiguous())


class DmB200(_Base):
    """dmCompass.py:50-160.  dm_index follows the parameter file's p_dms list."""

    def __init__(self, sim, config, pzt_index, tt_index):
        super().__init__(sim, config)
        self._pzt, self._tt = pzt_index, tt_index

    def reset_dm(self, dm_index=-1):
        self._sim.reset_dm()

    def set_command(self, commands, *, dm_index=None, shape_dm=True):
        import torch
        sim = self._sim
        v = sim.rows("VOLTS", sim.cfg.nactu)
        x = torch.as_tensor(commands, dtype=torch.float32, device="cuda")
        if x.dim() == 1:
            x = x.unsqueeze(0).expand(sim.n_env, -1)
        if dm_index is None:
            if x.shape[1] != sim.cfg.nactu:
                raise ValueError("Dimension mismatch")
            v.copy_(x)
        elif dm_index == self._pzt:
            if x.shape[1] != sim.cfg.pzt_nact:
                raise ValueError("Dimension mismatch")
            v[:, :sim.cfg.pzt_nact].copy_(x)
        elif dm_index == self._tt:
            if x.shape[1] != 2:
                raise ValueError("Dimension mismatch")
            v[:, sim.cfg.pzt_nact:].copy_(x)
        else:
            raise NotImplementedError("DM %d is not driven by controller 0" % dm_index)

    def get_dm_shape(self, indx):
        raise NotImplementedError("mirror surfaces are evaluated per subaperture inside the fused kernel; "
                                  "use wfs.raytrace(dms=...) + wfs.get_wfs_phase for the surface seen by the sensor")


class _Controller:
    """Stand-in for ``rtc._rtc.d_control[i]`` (ao_env.py:957, train_rpc.py:84 read .gain / call .set_gain; sutra's
    controller also has .delay / set_delay)."""

    def __init__(self, sim, ctype):
        self._sim = sim
        self.type = ctype

    @property
    def gain(self):
        """The integrator gain in force: the common one, or the float32 [E] per-environment gains."""
        g = self._sim.gain_env
        return self._sim.gain if g is None else g

    def set_gain(self, g):
        """A scalar sets the gain of every environment (and drops per-environment gains); an [E] array one gain per
        environment."""
        if np.ndim(g) == 0:
            self._sim.set_gain(float(g))
            self._sim.set_gain_env(None)
        else:
            self._sim.set_gain_env(g)

    @property
    def delay(self):
        """The controller delay in frames in force: the common one, or the float32 [E] per-environment delays."""
        d = self._sim.delay_env
        return self._sim.delay if d is None else d

    def set_delay(self, d):
        """A scalar in [0, 2] sets the delay of every environment (and drops per-environment delays); an [E] array one
        delay per environment."""
        if np.ndim(d) == 0:
            self._sim.set_delay(float(d))
            self._sim.set_delay_env(None)
        else:
            self._sim.set_delay_env(d)


class _RtcHandle:
    def __init__(self, controls):
        self.d_control = controls


class RtcB200(_Base):
    """rtcCompass.py:55-630: controller 0 = least-squares integrator; when the parameter file lists a geometric
    controller (type "geo"), do_control / apply_control / get_command / get_voltages also accept its index."""

    def __init__(self, sim, config, tables):
        super().__init__(sim, config)
        self._tables = tables
        self._geo = next((i for i, c in enumerate(config.p_controllers) if getattr(c, "type", "") == "geo"), None)
        controls = [_Controller(sim, "ls")]
        if self._geo is not None:
            while len(controls) < self._geo:
                controls.append(None)
            controls.append(_Controller(sim, "geo"))
        self._rtc = _RtcHandle(controls)
        self.d_control = self._rtc.d_control

    def _is_geo(self, i):
        return i != 0 and i == self._geo and getattr(self._tables, "geo_proj", None) is not None

    def _chk(self, i):
        if i != 0:
            raise NotImplementedError("controller %d: only the LS integrator (0) serves this call" % i)

    def do_centroids(self, controller_index):
        self._chk(controller_index)
        self._sim.do_centroids()

    def do_control(self, controller_index, **kw):
        if self._is_geo(controller_index):
            self._sim.do_control_geo()
            return
        self._chk(controller_index)
        self._sim.do_control()

    def apply_control(self, controller_index, *, comp_voltage=True):
        if self._is_geo(controller_index):
            self._sim.apply_control_geo()
            return
        self._chk(controller_index)
        self._sim.apply_control(comp_voltage)

    def do_clipping(self, controller_index):
        self._chk(controller_index)   # +-1e5 V limits are never reached on this path

    def get_slopes(self, controller_index):
        self._chk(controller_index)
        return self._out(self._sim.rows("SLOPES", self._sim.cfg.nslopes))

    def get_err(self, controller_index):
        self._chk(controller_index)
        return self._out(self._sim.rows("ERR", self._sim.cfg.nactu))

    def get_command(self, controller_index):
        if self._is_geo(controller_index):
            return self._out(self._sim.rows("GEO_COM", self._sim.cfg.nactu))
        self._chk(controller_index)
        return self._out(self._sim.rows("COM", self._sim.cfg.nactu))

    def get_voltages(self, controller_index):
        if self._is_geo(controller_index):
            return self._out(self._sim.rows("GEO_VOLTS", self._sim.cfg.nactu))
        self._chk(controller_index)
        return self._out(self._sim.rows("VOLTS", self._sim.cfg.nactu))

    def set_command(self, controller_index, com):
        self._chk(controller_index)
        if np.shape(com)[-1] != self._sim.cfg.nactu:
            raise ValueError("Dimension mismatch")
        self._sim.set_command(com)

    def reset_command(self, controller_index=None):
        import torch
        self._sim.set_command(torch.zeros((self._sim.n_env, self._sim.cfg.nactu), device="cuda"))

    def set_gain(self, controller_index, gain):
        self._chk(controller_index)
        self.d_control[0].set_gain(gain)

    def get_interaction_matrix(self, controller_index):
        self._chk(controller_index)
        return self._tables.imat

    def get_command_matrix(self, controller_index):
        self._chk(controller_index)
        return self._sim.cmat

    def set_command_matrix(self, controller_index, cmat):
        self._chk(controller_index)
        self._sim.set_command_matrix(cmat)

    def open_loop(self, controller_index=None, reset=True):
        self._sim.set_loop(False)
        if reset:
            self.reset_command()

    def close_loop(self, controller_index=None):
        self._sim.set_loop(True)


class TargetB200(_Base):
    """targetCompass.py (next-row scope) without the focal-plane image: get_strehl() = [SE, LE, phase variance, mean
    variance] with SE = |<exp(i k phi)>|^2 over the pupil -- the on-axis intensity ratio, i.e. the peak of the PSF the
    reference's FFT gives for a tilt-free residual (Marechal's exp(-sigma^2) for small ones) -- and LE its mean over the
    frames; with peak_fit (default) SE / LE are the brightest pixel of the 3 x 3 PSF core on the reference's focal grid,
    refined by a three-point fit per axis (comp_strehl(do_fit=True)); the full image only exists on demand (get_tar_image).  One sweep kernel (aom_comp_strehl) evaluates the on-axis
    phase per pupil pixel and reduces it without materialising it; the figures live in AOM_B_STREHL."""

    def __init__(self, sim, config, tables, eager_trace=False):
        super().__init__(sim, config)
        self._tables = tables
        self._flags = {}
        # eager_trace: raytrace() sweeps the pupil at once, as sutra does, so that a Strehl published later refers to the
        # mirrors of the moment of the trace (the reference's ordering when apply_control falls between
        # next_part_one's target trace and next_part_two's comp_strehl).  Default: the sweep runs when the image is asked
        # for -- one sweep per frame instead of one per trace, equal to the reference's "pure delay 0" ordering.
        self.eager_trace = bool(eager_trace)
        self._pending = set()
        # SE / LE from the brightest pixel of the PSF core with a three-point fit, as the reference's
        # comp_strehl(do_fit=True) default; False: the on-axis pixel (cheaper sweep)
        self.peak_fit = True
        # target i looks through the mirrors of the geometric controller when its dms are that controller's
        # (parameter layout "geo": target 1 <-> DMs [1, 3] <-> controller 1)
        geo = next((c for c in config.p_controllers if getattr(c, "type", "") == "geo"), None)
        gd = sorted(int(d) for d in geo.ndm) if geo is not None else None
        self._geo_targets = {i for i, tg in enumerate(config.p_targets)
                             if gd is not None and sorted(int(d) for d in tg.dms_seen) == gd}

    def _is_geo(self, index):
        return index in self._geo_targets and getattr(self._tables, "geo_proj", None) is not None

    def raytrace(self, index, *, tel=None, atm=None, dms=None, ncpa=True, reset=True):
        a, d = (False, False) if reset else self._flags.get(index, (False, False))
        if atm is not None and getattr(atm, "is_enable", True):
            a = True
        if dms is not None:
            d = True
        self._flags[index] = (a, d)
        if self.eager_trace:
            lam = float(self._config.p_targets[index].Lambda)
            self._sim.comp_strehl(lam, atmos=a, dms=d, geo=self._is_geo(index), phase="trace", peak=self.peak_fit)
            self._pending.add(index)

    def comp_tar_image(self, tarNum, *, puponly=0, compLE=True):
        lam = float(self._config.p_targets[tarNum].Lambda)
        a, d = self._flags.get(tarNum, (False, False))
        phase = "publish" if (self.eager_trace and tarNum in self._pending) else "both"
        self._sim.comp_strehl(lam, atmos=a, dms=d, accumulate=bool(compLE), geo=self._is_geo(tarNum), phase=phase,
                              peak=self.peak_fit)

    def comp_strehl(self, tarNum, *, do_fit=True):
        pass

    def reset_strehl(self, tar_index):
        self._sim.reset_strehl()

    def get_strehl(self, tar_index, *, do_fit=True):
        """[SE, LE, variance, mean variance]: floats when E == 1 (targetCompass.py:139-159), else [E] device tensors."""
        s = self._sim.buffer("STREHL_GEO" if self._is_geo(tar_index) else "STREHL").view(self._sim.n_env, 4)
        if self._sim.n_env == 1:
            return [float(x) for x in s[0].cpu()]
        return [s[:, i] for i in range(4)]

    def get_tar_image(self, tar_index, *, expo_type="se", envs=None):
        """Short-exposure PSF on the reference's Nfft x Nfft focal grid, centred (np.fft.fftshift of sutra's d_image_se,
        targetCompass.py:69-87), in units of the diffraction-limited peak.  An on-demand getter for plots and checks, not
        part of the step: the phase of the selected environments (default: the first) is materialised and transformed
        with torch.fft.  The long-exposure image is not kept -- only its 3 x 3 core feeds the LE Strehl."""
        if expo_type != "se":
            raise NotImplementedError("only the 3 x 3 core of the long-exposure image is accumulated (LE Strehl)")
        import torch
        sim = self._sim
        a, d = self._flags.get(tar_index, (True, True))
        envs = [0] if envs is None else list(envs)
        g = self._config.p_geom
        pd = int(g.pupdiam)
        off = (int(g._n) - pd) // 2
        ph = sim.raytrace_wfs(atmos=a, dms=d)[envs, off:off + pd, off:off + pd].double()
        pup = torch.as_tensor(np.asarray(g._spupil) > 0, device=ph.device)
        k = 2 * np.pi / float(self._config.p_targets[tar_index].Lambda)
        field = torch.polar(pup.double().expand_as(ph), k * ph)
        nf = sim.psf_nfft
        img = torch.fft.fft2(field, s=(nf, nf)).abs().square() / float(pup.sum()) ** 2
        img = torch.fft.fftshift(img, dim=(-2, -1)).float()
        return img[0].cpu().numpy() if (sim.n_env == 1 or len(envs) == 1) else img

    def get_tar_phase(self, tar_index, *, pupil=False):
        a, d = self._flags.get(tar_index, (False, False))
        return self._out(self._sim.raytrace_wfs(atmos=a, dms=d))
