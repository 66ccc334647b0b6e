"""RlSupervisor: the reference's RL split of the AO frame behind the same method surface
(shesha/supervisor/rlSupervisor.py:60-1051; construction order of genericSupervisor.py:116-142),
batched over E environments and executed by libaomarl.so.

    sup = RlSupervisor(config, config_rl, initial_seed=1234, n_env=4096)
    sup.reset(); sup.next_part_one(); sup.next_part_two(action)

`config` is a parameter set (ao_marl_b200.config.load_config_from_file), `config_rl` anything with
``.env_rl`` / ``.sac`` / ``.autoencoder`` dicts as the reference's Config object has
(src/reinforcement_learning/config/GlobalConfig.py).
"""
import numpy as np

from .. import calibration, tables as tables_mod
from ..init import geo as geo_b
from ..init import rtc as rtc_b
from ..lib import Simulator
from ..rl.layout import RLLayout
from .components import AtmosB200, DmB200, RtcB200, TargetB200, TelescopeB200, WfsB200


class _Basis:
    """Holder for supervisor.basis (ModalBasis optimizer, modalBasis.py:102-164)."""

    def __init__(self, tables):
        self._t = tables

    def compute_modes_to_volts_basis(self, dms=None, p_dms=None, modal_basis_type="Btt"):
        if modal_basis_type != "Btt":
            raise NotImplementedError("only the Btt basis is on the hot path")
        return self._t.Btt, self._t.P


class RlSupervisor:
    def __init__(self, config, config_rl, *, build_cmat_with_modes=True, initial_seed=1234, autoencoder=None,
                 cacao=False, n_env=1, world_size=None, tables=None, norm=None, zn_norm=None, policy_seed=0):
        if cacao:
            raise NotImplementedError("CACAO publishing is outside the hot-path scope")
        self.cacao = False
        self.config = config
        self.config_rl = config_rl
        env_rl = config_rl.env_rl
        env_rl.setdefault("which_basis", "Btt")
        self.n_modes_start_end = env_rl["n_zernike_start_end"]
        self.n_reverse_filtered_from_cmat = env_rl["n_reverse_filtered_from_cmat"]
        self.include_tip_tilt = env_rl["include_tip_tilt"]
        # modification_online ("pure delay 0", rlSupervisor.py:936-940): the target is re-traced right after apply_control,
        # so the published Strehl already contains the new command; DelayedMDP shortens its window accordingly
        self.pure_delay_0 = bool(env_rl["modification_online"])
        self.autoencoder = autoencoder
        self.freedom_vector_actuator_space = None
        self.initial_seed = initial_seed
        self.current_seed = initial_seed
        self.iter = 0
        self.is_init = False
        self.past_command_rl = None

        # static tables -> interaction matrix on the GPU -> Btt -> command matrix
        t = tables if tables is not None else tables_mod.build_static(config)
        if getattr(t, "imat", None) is None:
            t.imat = calibration.measure_imat(t)
        if getattr(t, "Btt", None) is None:
            tables_mod.build_basis(t)
        nfilt = self.n_reverse_filtered_from_cmat if (build_cmat_with_modes and env_rl["which_basis"] == "Btt") else -1
        if getattr(t, "cmat", None) is None or getattr(t, "nfilt", None) != max(nfilt, 0):
            t.nfilt = max(nfilt, 0)
            t.cmat = rtc_b.cmat_with_btt(t.imat, t.Btt, t.nfilt)
        # second controller of the "geo" parameter layouts: least-squares fit of the mirrors to the target phase
        self.geo_index = next((i for i, c in enumerate(config.p_controllers) if getattr(c, "type", "") == "geo"), None)
        if self.geo_index is not None and getattr(t, "geo_proj", None) is None:
            geo_b.build_geo(t)
        self.tables = t
        self.modes2volts, self.volts2modes = t.Btt, t.P
        sac = getattr(config_rl, "sac", None)
        self.rl = RLLayout(t.Btt.shape[1], env_rl, sac, world_size, norm=norm, zn_norm=zn_norm, seed=policy_seed)
        self.freedom_vector = self.rl.freedom
        self.sim = Simulator(t, n_env, self.rl)
        self.n_env = int(n_env)
        if autoencoder is not None and hasattr(autoencoder, "attach"):
            autoencoder.attach(self.sim)  # per-subaperture CNN on the fused kernel (aom_denoise)

        ctrl = config.p_controllers[0]
        self.tel = TelescopeB200(self.sim, config)
        self.atmos = AtmosB200(self.sim, config)
        self.dms = DmB200(self.sim, config, int(ctrl.ndm[0]), int(ctrl.ndm[1]))
        # faithful ordering of the target trace: without pure delay 0 the Strehl of next_part_two refers to the mirrors of
        # the trace in next_part_one (eager sweep at raytrace); with it the sweep after apply_control is the reference's own
        self.target = TargetB200(self.sim, config, t, eager_trace=not self.pure_delay_0)
        self.wfs = WfsB200(self.sim, config, t.wfs_index)
        self.rtc = RtcB200(self.sim, config, t)
        self.basis = _Basis(t)
        self.calibration = None
        self.is_init = True
        self.action_range_for_roket = self.obtain_action_range_modal(np.zeros(t.nactu))

    # -- default methods (rlSupervisor.py:196-246) -----------------------------------------------
    def get_config(self):
        return self.config

    def get_frame_counter(self):
        return self.iter

    def load_freedom_vector_from_env(self, normalization_bool):
        self.freedom_vector = self.rl.freedom if normalization_bool else None

    def set_sim_seed(self, seed):
        self.current_seed = seed

    def obtain_and_set_cmat_filtered(self, modes_filtered):
        cmat = rtc_b.cmat_with_btt(self.tables.imat, self.modes2volts, max(modes_filtered, 0))
        self.rtc.set_command_matrix(0, cmat)
        return cmat

    def reset(self):
        """atmos.reset_turbu + wfs.reset_noise + target.reset_strehl + dms.reset_dm + integrator reset: a single
        aom_reset regenerates the screens from the seeds and clears mirrors, delay line, integrator and histories."""
        self.past_command_rl = None
        self.atmos.reset_turbu(self.current_seed)
        self.wfs.reset_noise(self.current_seed)
        for tar_index in range(len(self.config.p_targets)):
            self.target.reset_strehl(tar_index)
        self.rtc.close_loop()

    def reset_envs(self, envs, seeds):
        """Restart the environments `envs` with `seeds` while the others run on (aom_reset_envs): everything reset() does,
        for those environments only.  Their next next_part_two is ignored (no action, no Strehl) and their next
        next_part_one + state leave their s0.  Conditions of the new episode (atmos.set_r0 / set_wind with [E] arrays)
        must be set before the call, so that the start-up of their screens uses them."""
        self.sim.reset_envs(envs, seeds)

    def get_m_pupil(self):
        return self.config.p_geom._mpupil

    def get_s_pupil(self):
        return self.config.p_geom._spupil

    def get_i_pupil(self):
        return self.config.p_geom._ipupil

    # -- control (rlSupervisor.py:677-836) ---------------------------------------------------------
    def obtain_action_range_modal(self, final_command_modal):
        if self.n_modes_start_end[0] >= 0:
            rng = list(range(self.n_modes_start_end[0], self.n_modes_start_end[1]))
            return rng + [-2, -1] if self.include_tip_tilt else rng
        return list(range(self.modes2volts.shape[1]))

    def rl_control(self, action, ncontrol, evaluation_rl_full_action=False):
        """com <- m2v . (v2m . com + scatter((a * std + mean) * freedom)); scaling constants live in the context."""
        if self.config_rl.env_rl["level"] != "correction":
            raise NotImplementedError
        self.sim.rl_control(action)

    def raytrace_target(self, ncontrol):
        t = ncontrol
        if self.atmos.is_enable:
            self.target.raytrace(t, tel=self.tel, atm=self.atmos, dms=self.dms)
        else:
            self.target.raytrace(t, tel=self.tel, dms=self.dms)

    def autoencoder_denoising(self):
        """bincube -> denoiser -> back into the centroider input, all on the device (rlSupervisor.py:876-891
        does a host round trip and a python loop over subapertures)."""
        if getattr(self.autoencoder, "sim", None) is self.sim:
            self.sim.denoise()            # fused kernel, in place, feeds the next do_centroids
            return
        cube = self.wfs.get_bincube()
        E, nv = cube.shape[0], cube.shape[1]
        den = self.autoencoder.predict(cube.reshape(E * nv, 16, 16))
        self.wfs.set_bincube(den.reshape(E, nv, 256))

    # -- the two half-steps (rlSupervisor.py:900-1051) ------------------------------------------------
    def next_part_two(self, action, linear_control=False, tar_trace=None, apply_control=True, compute_tar_psf=True,
                      evaluation_rl_full_action=False):
        if not linear_control:
            self.rl_control(action, 0, evaluation_rl_full_action)
        if apply_control:
            self.rtc.apply_control(0)
            if self.pure_delay_0:
                self.raytrace_target(0)
        if compute_tar_psf:
            self.target.comp_tar_image(0)
            self.target.comp_strehl(0)

    def generic_delay_0_next(self, *, move_atmos=True, ncontrol=0, tar_trace=None, wfs_trace=None, do_control=True,
                             apply_control=True, compute_tar_psf=True):
        """rlSupervisor.py:329-394: the vanilla frame with the target re-traced right after apply_control (used by the
        reference's dataset dumps, obtain_dataset_autoencoder.py:85-88)."""
        if move_atmos and self.atmos is not None:
            self.atmos.move_atmos()
        self.next_part_one_integrator(ncontrol=ncontrol, do_control=do_control)
        if apply_control:
            self.rtc.apply_control(ncontrol)
            self.raytrace_target(ncontrol)
        if compute_tar_psf:
            self.target.comp_tar_image(0)
            self.target.comp_strehl(0)
        self.iter += 1

    def next_part_one_integrator(self, *, ncontrol=0, do_control=True):
        self.raytrace_target(ncontrol)
        w = self.tables.wfs_index
        if self.atmos.is_enable:
            self.wfs.raytrace(w, tel=self.tel, atm=self.atmos)
        else:
            self.wfs.raytrace(w, tel=self.tel)
        if not self.config.p_wfss[w].open_loop and self.dms is not None:
            self.wfs.raytrace(w, dms=self.dms, ncpa=False, reset=False)
        self.wfs.keep_image = self.autoencoder is not None
        self.wfs.compute_wfs_image(w)
        if self.autoencoder is not None:
            self.autoencoder_denoising()
        if do_control:
            self.rtc.do_centroids(ncontrol)
            self.rtc.do_control(ncontrol)

    def next_part_one_geo(self, *, ncontrol=1, do_control=True, geometric_apply_control=True):
        """rlSupervisor.py:989-1013: target trace through the atmosphere, projection, apply, trace through the mirrors."""
        t = ncontrol
        if self.atmos.is_enable:
            self.target.raytrace(t, tel=self.tel, atm=self.atmos, ncpa=False)
        else:
            self.target.raytrace(t, tel=self.tel, ncpa=False)
        if do_control and self.rtc is not None:
            self.rtc.do_control(ncontrol, sources=None, source_index=t)
            if geometric_apply_control:
                self.rtc.apply_control(ncontrol)
            self.target.raytrace(t, dms=self.dms, ncpa=True, reset=False)

    def next_part_one(self, *, move_atmos=True, tar_trace=None, wfs_trace=None, do_control=True,
                      geometric_apply_control=True, geo=False):
        """rlSupervisor.py:1015-1051.  The reference runs every controller of the parameter file each frame; the
        geometric one only feeds the "fitting error" curves, so here it is opt-in (geo=True, or
        ``sim.step_with_geo()`` for the fused step)."""
        if move_atmos and self.atmos is not None:
            self.atmos.move_atmos()
        self.next_part_one_integrator(ncontrol=0, do_control=do_control)
        if geo and self.geo_index is not None:
            self.next_part_one_geo(ncontrol=self.geo_index, do_control=do_control,
                                   geometric_apply_control=geometric_apply_control)
        self.iter += 1

    def next(self, *, move_atmos=True, nControl=0, tar_trace=None, wfs_trace=None, do_control=True,
             apply_control=True, compute_tar_psf=True):
        """Vanilla closed-loop frame (genericSupervisor.py:180-243)."""
        if move_atmos:
            self.atmos.move_atmos()
        self.next_part_one_integrator(ncontrol=nControl, do_control=do_control)
        if apply_control:
            self.rtc.apply_control(nControl)
        if compute_tar_psf:
            self.target.comp_tar_image(0)
            self.target.comp_strehl(0)
        self.iter += 1

    def next_normalization(self, linear_control_through_modal=False, **kw):
        """One integrator frame returning v2m . voltages (rlSupervisor.py:591-657); the phase-projection
        estimate of the reference (second return value) is outside the hot-path scope."""
        self.next(**{k: v for k, v in kw.items() if k in ("move_atmos", "do_control", "apply_control",
                                                          "compute_tar_psf")})
        import torch
        v = self.sim.rows("VOLTS", self.sim.cfg.nactu)
        modes = v @ torch.as_tensor(self.volts2modes, device=v.device).T
        return (modes[0].cpu().numpy() if self.n_env == 1 else modes), []
