"""RL-side layout of one experiment: which Btt modes the agents act on, how the state vector is laid
out, how it is split between agents, the normalisation inputs and the actors.

Restates the configuration logic spread over the reference's
  RlSupervisor.obtain_action_range_modal / load_freedom_parameter_modal_space  (shesha/supervisor/rlSupervisor.py:677-691, 255-282)
  AoEnv.define_state_action_space / load_norm_parameters / transform_state_to_zernike (src/.../environment/ao_env.py:154-214, 251-306, 482-505)
  TrainerRPC.create_agents_dictionary / prepare_indices_of_state / get_state_shape_worker / load_soft_actor_critic (src/.../rpc_training/train_rpc.py:265-379)
and turns it into the integer / float tables of include/aomarl.h.
"""
import os

import numpy as np

from . import helper_states as hs
from .policy import GaussianPolicy, pack_actors

DATA_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "data", "normalization")

DEFAULT_ENV_RL = dict(
    n_zernike_start_end=[-1, -1], include_tip_tilt=True, window_n_zernike=-1, include_tip_tilt_windowed=False,
    tt_treated_as_mode=False, n_reverse_filtered_from_cmat=0, number_of_previous_dm=2, number_of_previous_wfs=0,
    number_of_previous_dm_residuals=0, state_dm_before_linear=True, state_dm_after_linear=False, state_wfs=False,
    state_dm_residual=True, normalization_std_inside_environment=1.0, normalization_mean_inside_environment=0.0,
    norm_scale_zernike_actions=10.0, reward_type="avg_squared_modes_1000", delayed_assignment=1,
    modification_online=False, level="correction", basis="zernike_space", which_basis="Btt",
    max_steps_per_episode=1000, custom_freedom_path=None, parameters_telescope=None)
DEFAULT_SAC = dict(hidden_size_actor=256, num_layers_actor=2, activation="relu", gaussian_mu=0.0, gaussian_std=1.0,
                   LOG_SIG_MAX=2.0, initialize_last_layer_0=True, initialize_last_layer_near_0=False, gamma=0.1,
                   batch_size=256, lr=3e-4, tau=0.005, alpha=0.2, automatic_entropy_tuning=True)


def load_normalization(parameters_telescope):
    name = os.path.basename(parameters_telescope)
    name = name[:-3] if name.endswith(".py") else name
    path = os.path.join(DATA_DIR, name + ".npz")
    if not os.path.exists(path) and name.endswith("_d0_noise"):
        # the reference ships the statistics of its magnitude-9 noisy configuration under this name
        # (normalization_production_sh_40x40_8m_3layers_noise_M9_zernike_space.pickle)
        path = os.path.join(DATA_DIR, name[:-len("_d0_noise")] + "_noise_M9.npz")
    if not os.path.exists(path):
        raise FileNotFoundError("no normalisation statistics shipped for %s" % name)
    z = np.load(path)
    norm = {k: {s: z["%s_%s" % (k, s)] for s in ("mean", "std", "max", "min")} for k in ("dm", "wfs", "dm_residual")}
    return norm, z["zn_norm"].copy()


class RLLayout:
    def __init__(self, nmodes, env_rl=None, sac=None, world_size=None, norm=None, zn_norm=None, seed=0,
                 policies=None):
        self.env_rl = e = dict(DEFAULT_ENV_RL, **(env_rl or {}))
        self.sac = s = dict(DEFAULT_SAC, **(sac or {}))
        self.nmodes = int(nmodes)
        for k in ("state_wfs", "state_dm_after_linear"):
            if e[k]:
                raise NotImplementedError("state block %s is outside the hot-path scope" % k)
        if e["number_of_previous_wfs"] or e["number_of_previous_dm_residuals"]:
            raise NotImplementedError("only the command history is kept in the state")
        if not (e["state_dm_before_linear"] and e["state_dm_residual"]):
            raise NotImplementedError("state needs dm_before_linear and dm_residual")
        if e["level"] != "correction" or e["basis"] != "zernike_space" or e["tt_treated_as_mode"]:
            raise NotImplementedError("only level=correction / basis=zernike_space is on the hot path")
        if norm is None or zn_norm is None:
            norm, zn_norm = load_normalization(e["parameters_telescope"])
        if len(zn_norm) != self.nmodes:
            raise ValueError("Dimension mismatch: %d normalisation modes, %d Btt modes" % (len(zn_norm), self.nmodes))
        self.freedom = (np.asarray(zn_norm, np.float32) / np.float32(e["norm_scale_zernike_actions"])).astype(np.float32)

        s0, s1 = e["n_zernike_start_end"]
        if s0 >= 0:
            rng = list(range(s0, s1)) + ([self.nmodes - 2, self.nmodes - 1] if e["include_tip_tilt"] else [])
        else:
            rng = list(range(self.nmodes))
        self.action_map = np.asarray(rng, dtype=np.int32)
        self.action_dim = len(rng)
        windowed = e["window_n_zernike"] > -1
        self.state_map = np.arange(self.nmodes, dtype=np.int32) if (windowed or s0 < 0) else self.action_map.copy()
        self.state_modes = len(self.state_map)
        self.n_hist = int(e["number_of_previous_dm"])
        self.state_keys = (["dm_history_%d" % (self.n_hist - i) for i in range(self.n_hist)]
                           + ["dm_before_linear", "dm_residual"])
        self.state_dim = len(self.state_keys) * self.state_modes
        self.indices_of_state = {k: [i * self.state_modes, (i + 1) * self.state_modes]
                                 for i, k in enumerate(self.state_keys)}
        self.norm = {k: {st: np.asarray(v[st], np.float32)[self.state_map] for st in ("mean", "std")}
                     for k, v in norm.items() if k in ("dm", "dm_residual")}
        self.reward_factor = float(e["reward_type"].split("_")[-1]) if "avg_squared_modes_" in e["reward_type"] else None
        if self.reward_factor is None:
            raise NotImplementedError("reward %s is outside the hot-path scope" % e["reward_type"])

        # agents
        self.world_size = world_size
        if world_size is None:
            self.agents = {}
        else:
            self.agents, self.total_controlled, self.local_controlled = hs.agents_dictionary(
                self.nmodes, s0, s1, world_size, e["include_tip_tilt"])
        self.n_agents = len(self.agents)
        if self.n_agents:
            self.modes_chosen = hs.get_modes_chosen(self.agents, self.indices_of_state, e,
                                                    e["n_reverse_filtered_from_cmat"], self.nmodes,
                                                    self.total_controlled, s0)
            for wid, rngw in self.agents.items():
                want = hs.state_shape_worker(rngw, e, wid, self.n_agents)
                if want != len(self.modes_chosen[wid]):
                    raise ValueError("agent %d: state split has %d entries, expected %d"
                                     % (wid, len(self.modes_chosen[wid]), want))
            self.actor_in = max(len(v) for v in self.modes_chosen.values())
            self.actor_out = max(v[1] - v[0] for v in self.agents.values())
            self.hidden = int(s["hidden_size_actor"])
            self.agent_idx = -np.ones((self.n_agents, self.actor_in), np.int32)
            self.agent_act = -np.ones((self.n_agents, self.actor_out), np.int32)
            self.agent_reward = np.zeros((self.n_agents, 2), np.int32)
            for a, wid in enumerate(sorted(self.agents)):
                mc = self.modes_chosen[wid]
                self.agent_idx[a, :len(mc)] = mc
                lo, hi = hs.action_slots(self.agents[wid], self.nmodes, self.total_controlled, s0,
                                         e["include_tip_tilt"])
                self.agent_act[a, :hi - lo] = np.arange(lo, hi)
                self.agent_reward[a] = self.agents[wid]
            if policies is None:
                import torch
                gen_state = torch.random.get_rng_state()
                torch.manual_seed(seed)
                policies = [GaussianPolicy(len(self.modes_chosen[wid]), self.agents[wid][1] - self.agents[wid][0],
                                           hidden_dim=self.hidden, num_layers=int(s["num_layers_actor"]),
                                           activation=s["activation"],
                                           initialize_last_layer_zero=bool(s["initialize_last_layer_0"]),
                                           initialize_last_layer_near_zero=bool(s["initialize_last_layer_near_0"]),
                                           action_scale=s["gaussian_std"], action_bias=s["gaussian_mu"],
                                           LOG_SIG_MAX=s["LOG_SIG_MAX"]) for wid in sorted(self.agents)]
                torch.random.set_rng_state(gen_state)
            self.policies = policies
        else:
            self.actor_in = self.actor_out = self.hidden = 0
            self.policies = []

    # -- context plumbing ------------------------------------------------------------------------
    def fill_config(self, cfg):
        e, s = self.env_rl, self.sac
        cfg.n_hist, cfg.state_modes, cfg.state_dim = self.n_hist, self.state_modes, self.state_dim
        cfg.env_act_scale = float(e["normalization_std_inside_environment"])
        cfg.env_act_bias = float(e["normalization_mean_inside_environment"])
        cfg.pol_act_scale, cfg.pol_act_bias = float(s["gaussian_std"]), float(s["gaussian_mu"])
        cfg.log_sig_min, cfg.log_sig_max = -20.0, float(s["LOG_SIG_MAX"])
        cfg.n_agents, cfg.actor_in, cfg.actor_hidden, cfg.actor_out = (self.n_agents, self.actor_in, self.hidden,
                                                                      self.actor_out)
        cfg.action_dim = self.action_dim
        cfg.reward_factor = float(self.reward_factor)

    def upload(self, sim):
        sim.set_table("FREEDOM", self.freedom)
        sim.set_table("ACTION_MAP", self.action_map)
        sim.set_table("STATE_MAP", self.state_map)
        sim.set_table("NORM_DM_MEAN", self.norm["dm"]["mean"])
        sim.set_table("NORM_DM_STD", self.norm["dm"]["std"])
        sim.set_table("NORM_RES_MEAN", self.norm["dm_residual"]["mean"])
        sim.set_table("NORM_RES_STD", self.norm["dm_residual"]["std"])
        if self.n_agents:
            sim.set_table("AGENT_IDX", self.agent_idx)
            sim.set_table("AGENT_ACT", self.agent_act)
            sim.set_table("AGENT_REWARD", self.agent_reward)
            self.upload_actors(sim)

    def upload_actors(self, sim, slot=0, policies=None):
        """Upload the actors (this layout's policies, or `policies`, one GaussianPolicy per agent) into policy slot
        `slot` of the simulator (Simulator.set_controller_env chooses the slot of each environment)."""
        pols = self.policies if policies is None else policies
        if len(pols) != self.n_agents:
            raise ValueError("upload_actors: %d policies for %d agents" % (len(pols), self.n_agents))
        for name, arr in pack_actors(pols, self.actor_in, self.hidden, self.actor_out).items():
            sim.set_table(name, arr, index=slot)
