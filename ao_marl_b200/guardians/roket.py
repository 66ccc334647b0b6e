"""ROKET -- error breakdown of the closed loop (SURVEY.md 8(f) rank 4, second half).

Reference: guardians/roket_generalized_rl.py:171-376 (`Roket(RlSupervisor)`: `init_config_roket`, `do_error_breakdown`,
`error_breakdown`, `cov_cor`, `save_in_hdf5`), driven by src/error_budget/error_budget_multiple_agents.py:306-343:

    env.rl_step(a, apply_control=False, compute_tar_psf=False); supervisor.do_error_breakdown(a); env.linear_step()

What it estimates, per frame and actuator: the part of the command error that comes from the detector noise, from the
centroiding (non linearity / truncation), from aliasing, from the filtered modes, from the loop delay (bandwidth), from
tomography and from the RL correction, each propagated through the integrator's loop filter, plus the fitting error (the
variance of the phase the mirrors cannot reproduce).  Here every environment of the batch gets its own breakdown: all
buffers are device tensors [frames, E, nactu] and the loop filters are batched products.

How each contributor is measured on this simulator (the arithmetic of the reference's calls lives in sutra; semantics [S]):

  noise        the same frame once more without detector noise -> centroids -> err E ; buffer = Derr - E
  non linearity geometric slopes of the same sensor phase (aom_do_centroids_geom) -> err F ; buffer = E - gamma F
  aliasing     the part of the phase orthogonal to the mirrors, phi_atm - proj(phi_atm) = atmosphere seen through the
               geometric controller's mirrors, measured with geometric slopes -> err Ageom.  (The reference projects the
               sensor's residual phase, atmosphere + main mirrors; the main mirrors' shape lies in the span of the influence
               functions, so its projection removes it exactly and the orthogonal part is the same.  On this repository's
               four-mirror parameter files the literal call sequence of the reference -- wfs.raytrace(dms, reset=False)
               after apply_control(1) -- would add the main mirrors a second time; the intended quantity of the original
               COMPASS ROKET is built here.)
  fitting      variance of that orthogonal phase over the pupil (aom_comp_strehl through the geometric mirrors)
  B            the geometric controller's command (least-squares fit of the target phase); filtered modes = its
               components on the modes the command matrix filters, commanded modes = the rest
  bandwidth    the frame-to-frame change of the commanded modes through the loop filter
  tomography   commanded modes of the sensor direction minus those of the target direction: identically zero for the
               on-axis single-sensor systems of this repository, kept for the reference's output layout
  zeta         the RL correction Btt . (action * freedom), delayed like a command, through the loop filter

Loop filter.  On this simulator the breakdown of frame i sees the command c[i] that already contains the error of the
frame's measurement, and that measurement saw the turbulence of frame i through the mirrors of command c[i-d],
d = controller delay + 1 (apply_control's delay line):   c[i] = c[i-1] + g (-R s[i]),  s[i] = D (c[i-d] - B[i]) + ...
Writing every part of -R s[i] separately gives, exactly,
    x[i]  = x[i-1]  - g gamma R D x[i-d]  + g b[i]                                (noise, non linearity, aliasing, tomography)
    bp[i] = bp[i-1] - g gamma R D bp[i-d] - (B[i] - B[i-1]) + g gamma R D (B[i] - B[i-d])        (bandwidth)
and  c[i] - B_commanded[i] = sum of the x[i] + bp[i]  (checked in tests/test_roket.py).  The reference indexes its buffers
with COMPASS's timing (b[i-d] drives x[i], the bandwidth term has no second bracket, roket_generalized_rl.py:190-260);
the quantities are the same contributions to the command.                       (R = cmat, D = imat)
"""
import numpy as np

from ..supervisor.rlSupervisor import RlSupervisor


class Roket(RlSupervisor):
    """RlSupervisor with the error breakdown.  Needs a parameter file with the geometric controller (controller 1)."""

    def __init__(self, config, config_rl=None, **kw):
        super().__init__(config, config_rl, **kw)
        if self.geo_index is None:
            raise ValueError("ROKET needs the geometric controller of the parameter file (p_controllers[1].type == 'geo')")
        self.iter_number = 0

    def _common_gain(self):
        """The loop filter of the breakdown uses one gain g for the whole batch."""
        if self.sim.gain_env is not None:
            raise NotImplementedError("ROKET's loop filter has one gain for the whole batch: per-environment gains "
                                      "(set_gain with an [E] array) are not supported; set a scalar gain")

    def reset_envs(self, envs, seeds):
        """Not available: the error-breakdown buffers ([N_total, E, .]) hold one run of the whole batch."""
        raise NotImplementedError("ROKET's breakdown buffers are whole-batch: use reset()")

    # -- buffers ----------------------------------------------------------------------------------------------------------
    def init_config_roket(self, N_total=3000, N_preloop=1000, agent=None, nfiltered=None, gamma=1.0, include_tip_tilt=True,
                          n_zernike_start=None, n_zernike_end=None):
        import torch
        assert N_total >= N_preloop
        self._common_gain()
        t, E = self.tables, self.n_env
        dev = "cuda"
        self.agent, self.include_tip_tilt = agent, include_tip_tilt
        self.nfiltered = int(self.n_reverse_filtered_from_cmat if nfiltered is None else nfiltered)
        self.N_preloop, self.gamma, self.n, self.iter_number = int(N_preloop), float(gamma), int(N_total), 0
        self.n_zernike_start, self.n_zernike_end = n_zernike_start, n_zernike_end
        self.nactus, self.nslopes = int(t.nactu), int(t.nslopes)
        z = lambda *shape: torch.zeros(shape, dtype=torch.float32, device=dev)
        na, ns, n = self.nactus, self.nslopes, self.n
        for name in ("com", "noise_com", "noise_buf", "alias_wfs_com", "ageom", "wf_com", "tomo_com", "tomo_buf", "trunc_com",
                     "trunc_buf", "H_com", "mod_com", "bp_com", "rl_commands", "zeta_contributor"):
            setattr(self, name, z(n, E, na))
        for name in ("alias_meas", "trunc_meas", "slopes"):
            setattr(self, name, z(n, E, ns))
        self.fit = z(n, E)
        self.centroid_gain = z(E)
        self.centroid_gain2 = z(E)
        self.Btt = torch.as_tensor(np.asarray(self.modes2volts, np.float32), device=dev)          # [nactu, nmodes]
        # volts -> modes with the FULL geometric covariance (piezo <-> tip-tilt cross terms included): the least-squares
        # command of the geometric controller may carry tilt on the piezo mirror, which compute_btt's block-diagonal
        # P = Btt^T Delta does not see (the reference loads Btt Btt^T into the geometric controller instead,
        # roket_generalized_rl.py:157-158: same effect).  For commands of the main loop the two projections coincide.
        from ..init.geo import influence_rows
        IF = influence_rows(t)
        npup = float((np.asarray(t.mpupil) != 0).sum())
        delta_full = (IF @ IF.T).toarray() / npup
        self.P = torch.as_tensor((np.asarray(self.modes2volts, np.float64).T @ delta_full).astype(np.float32), device=dev)  # [nmodes, nactu]
        self.cmat = torch.as_tensor(np.asarray(t.cmat, np.float32), device=dev)                   # R [nactu, nslopes]
        self.D = torch.as_tensor(np.asarray(t.imat, np.float32), device=dev)                      # D [nslopes, nactu]
        self.RD = self.cmat @ self.D
        self.g = float(self.config.p_controllers[0].gain)
        self.gRD = self.g * self.gamma * self.RD
        self.delay = int(round(float(self.config.p_controllers[0].delay))) + 1
        nm = self.P.shape[0]
        keep = torch.ones(nm, dtype=torch.bool, device=dev)
        if self.nfiltered > 0:
            keep[nm - self.nfiltered - 2:nm - 2] = False                # the filtered modes sit just before tip-tilt
        self._keep = keep
        self.SR = self.SR2 = None
        self.cov = self.cor = None

    # -- helpers ----------------------------------------------------------------------------------------------------------
    def _filter(self, com, buf, i, scale):
        """x[i] = x[i-1] - gRD x[i-d] + scale * buf[i]  (frames before the first read zeros)."""
        prev = com[i - 1] if i >= 1 else 0.0
        back = com[i - self.delay] @ self.gRD.T if i >= self.delay else 0.0
        com[i] = prev - back + scale * buf[i]

    def _err_of_current_slopes(self):
        """err = -cmat . slopes for the slopes just written, without integrating (the loop is opened for the call)."""
        sim = self.sim
        sim.set_loop(False)
        try:
            sim.do_control()
        finally:
            sim.set_loop(True)
        return sim.rows("ERR", self.nactus).clone(), sim.rows("SLOPES", self.nslopes).clone()

    @staticmethod
    def _centroid_gain(e, f):
        """Least-squares gain between two command errors (shesha.util.rtc_util.centroid_gain): <e, f> / <f, f> per env."""
        den = (f * f).sum(dim=1)
        return (e * f).sum(dim=1) / den.clamp_min(1e-30)

    # -- one frame --------------------------------------------------------------------------------------------------------
    def do_error_breakdown(self, a=None):
        """roket_generalized_rl.py:171-188: record the RL command of this frame, run the breakdown, then apply the (RL
        corrected) command and evaluate the target."""
        import torch
        self._common_gain()
        i = self.iter_number
        if a is not None and i < self.n:
            act = torch.as_tensor(a, dtype=torch.float32, device="cuda")
            if act.dim() == 1:
                act = act.unsqueeze(0).expand(self.n_env, -1)
            nm = self.Btt.shape[1]
            rl = torch.zeros((self.n_env, nm), device="cuda")
            rng = self.obtain_action_range_modal(None)
            idx = torch.as_tensor([r if r >= 0 else nm + r for r in rng], device="cuda")
            rl[:, idx] = act[:, :idx.numel()] * torch.as_tensor(np.asarray(self.freedom_vector, np.float32), device="cuda")[idx]
            self.rl_commands[i] = rl @ self.Btt.T
        self.error_breakdown()
        self.rtc.apply_control(0)
        self.raytrace_target(0)
        self.target.comp_tar_image(0)
        self.target.comp_strehl(0)
        self.iter_number += 1

    def error_breakdown(self):
        i = self.iter_number
        if i >= self.n:
            raise IndexError("ROKET buffers hold %d frames" % self.n)
        sim, g, gam = self.sim, self.g, self.gamma
        na = self.nactus
        Dcom = sim.rows("COM", na).clone()
        Derr = sim.rows("ERR", na).clone()
        Dslopes = sim.rows("SLOPES", self.nslopes).clone()
        self.com[i] = Dcom
        self.slopes[i] = Dslopes
        try:
            # noise: the same frame without detector noise
            sim.comp_wfs_image(noise=-1.0, advance_frame=False)
            sim.do_centroids()
            E, E_meas = self._err_of_current_slopes()
            self.noise_buf[i] = Derr - E
            self._filter(self.noise_com, self.noise_buf, i, g)
            # sampling / truncation: geometric slopes of the same phase
            sim.do_centroids_geom(atmos=True, dms=True)
            F, F_meas = self._err_of_current_slopes()
            self.trunc_meas[i] = E_meas - F_meas
            self.trunc_buf[i] = E - gam * F
            self._filter(self.trunc_com, self.trunc_buf, i, g)
            self.centroid_gain += self._centroid_gain(E, F)
            self.centroid_gain2 += self._centroid_gain(Derr, F)
            # projection of the atmosphere on the mirrors (geometric controller) and what is left
            sim.do_control_geo()
            sim.apply_control_geo()
            B = sim.rows("GEO_COM", na).clone()
            sim.do_centroids_geom(atmos=True, dms=True, geo=True)          # atmosphere through the geometric mirrors
            A, A_meas = self._err_of_current_slopes()
            self.ageom[i] = A
            self.alias_meas[i] = A_meas
            self._filter(self.alias_wfs_com, self.ageom, i, gam * g)
            lam = float(self.config.p_targets[0].Lambda)
            self.fit[i] = sim.comp_strehl(lam, atmos=True, dms=True, accumulate=False, geo=True)[:, 2]
            # filtered and commanded modes of the ideal command
            modes = B @ self.P.T
            self.H_com[i] = (modes * (~self._keep)) @ self.Btt.T
            self.mod_com[i] = (modes * self._keep) @ self.Btt.T
            # bandwidth
            C = self.mod_com[i] - (self.mod_com[i - 1] if i >= 1 else 0.0)
            lag = self.mod_com[i] - (self.mod_com[i - self.delay] if i >= self.delay else 0.0)
            prev = self.bp_com[i - 1] if i >= 1 else 0.0
            self.bp_com[i] = prev - (self.bp_com[i - self.delay] @ self.gRD.T if i >= self.delay else 0.0) - C + lag @ self.gRD.T
            # RL correction
            prev = self.zeta_contributor[i - 1] if i >= 1 else 0.0
            back = self.zeta_contributor[i - self.delay] @ self.gRD.T if i >= self.delay else 0.0
            self.zeta_contributor[i] = prev - back + self.rl_commands[i]
            # tomography: sensor direction = target direction here
            self.wf_com[i] = self.mod_com[i]
            self.tomo_buf[i] = self.mod_com[i] - self.wf_com[i]
            prev = self.tomo_com[i - 1] if i >= 1 else 0.0
            back = self.tomo_com[i - self.delay] @ self.gRD.T if i >= self.delay else 0.0
            self.tomo_com[i] = prev - back - g * gam * (self.tomo_buf[i] @ self.RD.T)
        finally:
            # the loop continues from the state it had: command, error, slopes of the real (noisy) frame
            sim.set_command(Dcom)
            sim.rows("ERR", na).copy_(Derr)
            sim.rows("SLOPES", self.nslopes).copy_(Dslopes)

    # -- results ----------------------------------------------------------------------------------------------------------
    def contributors(self):
        d = {"noise": self.noise_com, "non linearity": self.trunc_com, "aliasing": self.alias_wfs_com,
             "filtered modes": self.H_com, "bandwidth": self.bp_com, "tomography": self.tomo_com}
        if self.agent is not None:
            d["zeta_com"] = self.zeta_contributor
        return d

    def cov_cor(self):
        """roket_generalized_rl.py:443-486: covariance / correlation of the contributors in the modal basis, summed over
        the modes, per environment: cov [E, k, k]."""
        import torch
        n1 = min(self.iter_number, self.n)
        bufs = [b[self.N_preloop:n1] @ self.P.T for b in self.contributors().values()]      # [frames, E, nmodes]
        k = len(bufs)
        cov = torch.zeros((self.n_env, k, k), device="cuda")
        for a in range(k):
            for b in range(a, k):
                c = ((bufs[a] * bufs[b]).mean(0) - bufs[a].mean(0) * bufs[b].mean(0)).sum(-1)
                cov[:, a, b] = c
                cov[:, b, a] = c
        s = torch.diagonal(cov, dim1=1, dim2=2)
        den = torch.sqrt((s.unsqueeze(2) * s.unsqueeze(1)).clamp_min(0))
        cor = torch.where(den > 0, cov / den.clamp_min(1e-30), torch.zeros_like(cov))
        self.cov, self.cor = cov, cor
        return cov, cor

    def strehl_from_breakdown(self):
        """exp(-(2 pi / lambda)^2 (sum of the contributors' modal variances + fitting)): ROKET's consistency figure next
        to the measured long-exposure Strehl."""
        import torch
        cov, _ = self.cov_cor()
        n1 = min(self.iter_number, self.n)
        var = torch.diagonal(cov, dim1=1, dim2=2).sum(-1) + self.fit[self.N_preloop:n1].mean(0)
        lam = float(self.config.p_targets[0].Lambda)
        return torch.exp(-var * (2 * np.pi / lam) ** 2)

    def save(self, savename):
        """The reference's HDF5 fields (roket_generalized_rl.py:378-441) as one .npz (h5py is not a dependency here)."""
        n0, n1 = self.N_preloop, min(self.iter_number, self.n)
        cov, cor = self.cov_cor()
        host = lambda x: x.detach().cpu().numpy()
        out = {k: host(v[n0:n1]).transpose(1, 2, 0) for k, v in self.contributors().items()}      # [E, nactu, frames]
        out.update({"wf_com": host(self.wf_com[n0:n1]).transpose(1, 2, 0), "com": host(self.com[n0:n1]).transpose(1, 2, 0),
                    "slopes": host(self.slopes[n0:n1]).transpose(1, 2, 0),
                    "alias_meas": host(self.alias_meas[n0:n1]).transpose(1, 2, 0),
                    "trunc_meas": host(self.trunc_meas[n0:n1]).transpose(1, 2, 0),
                    "fitting": host(self.fit[n0:n1].mean(0)), "P": host(self.P), "Btt": host(self.Btt), "R": host(self.cmat),
                    "D": host(self.D), "cov": host(cov), "cor": host(cor),
                    "centroid_gain": host(self.centroid_gain) / max(n1 - n0, 1),
                    "centroid_gain2": host(self.centroid_gain2) / max(n1 - n0, 1),
                    "SR": np.asarray(self.SR if self.SR is not None else np.nan),
                    "SR2": np.asarray(self.SR2 if self.SR2 is not None else np.nan)})
        np.savez_compressed(savename, **out)

    save_in_hdf5 = save
