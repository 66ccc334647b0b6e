"""AoEnv: the gym-style environment of the reference (src/reinforcement_learning/environment/ao_env.py:18-978)
over the batched B200 supervisor.  Same method names and step sequencing; states, rewards and actions gain a
leading environment dimension E (squeezed to the reference's shapes when E == 1).

Hot path kept on the device: the state assembly of linear_step (v2m projections, history deque,
standardisation; ao_env.py:470-583, 871-909) is one aom_state_begin/aom_state_end pair, the default reward
(avg_squared_modes_<factor>, ao_env.py:845-853) one reduction kernel.
"""
import numpy as np

from ..config import load_config_from_file
from ..supervisor.rlSupervisor import RlSupervisor


class AoEnv:
    def __init__(self, config_rl, normalization_bool=True, build_cmat_with_modes=True, initial_seed=-1,
                 geo_policy_testing=False, roket=False, n_env=1, world_size=None, tables=None, autoencoder=None):
        if geo_policy_testing:
            raise NotImplementedError("the GEO policy-testing driver is outside the hot-path scope")
        if not normalization_bool:
            raise NotImplementedError("un-normalised states are outside the hot-path scope")
        self.normalization_bool = normalization_bool
        self.config_rl = config_rl
        self.n_env = int(n_env)
        config = load_config_from_file(config_rl.env_rl["parameters_telescope"])
        if roket:                      # ao_env.py:118-125: the supervisor with the error breakdown
            from ..guardians.roket import Roket as Supervisor
        else:
            Supervisor = RlSupervisor
        self.supervisor = Supervisor(config, config_rl, build_cmat_with_modes=build_cmat_with_modes,
                                     initial_seed=initial_seed, autoencoder=autoencoder, n_env=n_env,
                                     world_size=world_size, tables=tables)
        rl = self.supervisor.rl
        self.sim = self.supervisor.sim
        self.norm_parameters = rl.norm
        self.wfs_shape = (self.supervisor.tables.nslopes,)
        self.dm_shape = (rl.state_modes,)
        self.state_size = rl.state_dim
        self.action_size = rl.action_dim
        self.reward_type = config_rl.env_rl["reward_type"]
        self.verbose = config_rl.env_rl.get("verbose", False)

    # -- helpers -------------------------------------------------------------------------------------
    def _out(self, t):
        return t[0].detach().cpu().numpy() if self.n_env == 1 else t

    def set_sim_seed(self, seed):
        self.supervisor.set_sim_seed(seed)

    def is_geometric_controller_present(self):
        return False

    def standardise(self, inpt, key):
        p = self.norm_parameters[key]
        return (inpt - p["mean"]) / p["std"]

    def set_gain(self, g):
        g0 = g[0] if np.ndim(g) else g
        if not np.isscalar(g0):
            raise ValueError("Cannot set array gain w/ generic + integrator law")
        self.supervisor.rtc._rtc.d_control[0].set_gain(g0)

    # -- gym surface ---------------------------------------------------------------------------------
    def reset(self, normalization_loop=False, return_dict=False, geometric_do_control=False,
              geometric_apply_control=True):
        self.supervisor.reset()          # also zero-fills the command history (ao_env.py:336-347)
        self.supervisor.iter = 0
        if normalization_loop:
            return None
        return self.linear_step(return_dict, geometric_do_control, geometric_apply_control)

    def reset_envs(self, envs, seeds):
        """Autoreset of the environments `envs` with `seeds` (RlSupervisor.reset_envs): their next rl_step is ignored
        (reward 0) and their next linear_step returns their s0, while every other environment runs on.  Set the new
        episode's conditions (set_r0 / set_wind with [E] arrays) before the call."""
        self.supervisor.reset_envs(envs, seeds)

    def state(self):
        return self.sim.rows("STATE", self.state_size)

    def linear_step(self, return_dict=False, geometric_do_control=False, geometric_apply_control=True):
        """raytrace + WFS frame + centroids + integrator, then the normalised state.  geometric_do_control also runs the
        parameter file's geometric controller (the reference runs it every frame, ao_env.py:885; opt-in here)."""
        self.sim.state_begin()                         # s_dm_before_linear = rtc.get_command(0)
        self.supervisor.next_part_one(geometric_apply_control=geometric_apply_control, geo=geometric_do_control)
        self.sim.state_end()
        s = self.state()
        if return_dict:
            rl = self.supervisor.rl
            return {k: self._out(s[:, a:b]) for k, (a, b) in rl.indices_of_state.items()}
        return self._out(s)

    def calculate_reward(self, target=0, reward_type=None):
        """Global reward: -factor * mean over the action range of (v2m . d_err)^2 (ao_env.py:845-853);
        reward_type "strehl_ratio_se" / "strehl_ratio_le": the Strehl figures of `target` (ao_env.py:587-602)."""
        if reward_type in ("strehl_ratio_se", "strehl_ratio_le"):
            self.supervisor.target.raytrace(target, atm=self.supervisor.atmos, dms=self.supervisor.dms)
            self.supervisor.target.comp_tar_image(target)
            return self.supervisor.target.get_strehl(target)[0 if reward_type.endswith("_se") else 1]
        rl = self.supervisor.rl
        import torch
        res = self.sim.rows("RES_MODES", rl.nmodes)
        idx = torch.as_tensor(rl.action_map.astype(np.int64), device=res.device)
        r = -rl.reward_factor * res[:, idx].pow(2).mean(dim=1)
        return float(r[0]) if self.n_env == 1 else r

    def agent_rewards(self):
        """Per-agent rewards [E, n_agents] (TrainerRPC.divide_rewards_for_agents, train_rpc.py:402-416)."""
        rl = self.supervisor.rl
        self.sim.reward(rl.reward_factor)
        return self.sim.buffer("REWARD").view(self.n_env, rl.n_agents)

    def rl_step(self, action, linear_control=False, geometric_do_control=False, evaluation_rl_full_action=False,
                apply_control=True, compute_tar_psf=False):
        """rl_control + apply_control (+ target statistics when compute_tar_psf).  The reference computes the
        long-exposure PSF every frame (rlSupervisor.py:944-947); here it is opt-in."""
        self.supervisor.next_part_two(action=action, linear_control=linear_control,
                                      evaluation_rl_full_action=evaluation_rl_full_action,
                                      apply_control=apply_control, compute_tar_psf=compute_tar_psf)
        r = self.calculate_reward()
        if geometric_do_control and self.supervisor.geo_index is not None:
            # fitting-only Strehl of the target behind the geometric controller's mirrors (ao_env.py:928-937)
            return r, False, "", self.calculate_reward(target=1, reward_type="strehl_ratio_se")   # target 1, as the reference
        return r, False, ""

    def normalization_step(self, linear_control_through_modal=False):
        return self.supervisor.next_normalization(linear_control_through_modal)
