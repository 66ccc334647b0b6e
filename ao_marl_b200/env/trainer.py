"""In-process multi-agent rollout loop: TrainerRPC.episode without RPC
(src/reinforcement_learning/rpc_training/train_rpc.py:503-553, 620-648, 706-757): the master process of the
reference asks one remote SAC worker per agent for an action over torch.distributed.rpc and steps one
simulator; here every agent's actor and every environment advance in one aom_step on the device.
"""
import numpy as np

from ..rl.delayed_mdp import DelayedMDP


class BatchedRollout:
    def __init__(self, env, seed=1234):
        self.env = env
        self.sim = env.sim
        self.rl = env.supervisor.rl
        self.seed = seed
        self.total_step = 0
        self.num_episode = 0
        self.transitions = []       # (s, a, s_next, r) device tensors, per-agent views taken lazily

    def divide_states_for_agents(self, state):
        """{worker id: state[:, modes_chosen]} (train_rpc.py:418-427)."""
        import torch
        return {w: state[:, torch.as_tensor(np.asarray(idx, dtype=np.int64), device=state.device)]
                for w, idx in self.rl.modes_chosen.items()}

    def episode(self, steps=None, eval_mode=False, linear_control=False, on_transition=None):
        e = self.rl.env_rl
        steps = e["max_steps_per_episode"] if steps is None else steps
        self.env.set_sim_seed(self.seed)
        s = self.env.reset().clone() if self.env.n_env > 1 else self.sim.rows("STATE", self.rl.state_dim).clone()
        mdp = DelayedMDP(e["delayed_assignment"], e["modification_online"])
        r_total = 0.0
        for _ in range(steps):
            self.sim.step(mode=2 if linear_control else 0, eval_mode=eval_mode)
            a = self.sim.rows("ACTION", self.rl.action_dim).clone()
            r = self.sim.buffer("REWARD").view(self.env.n_env, self.rl.n_agents).clone()
            s_next = self.sim.rows("STATE", self.rl.state_dim).clone()
            if mdp.check_update_possibility():
                s0, a0, s2 = mdp.credit_assignment()
                if on_transition is not None:
                    on_transition(s0, a0, s2, r)
            mdp.save(s, a, s_next)
            r_total += float(r.sum(dim=1).mean())
            s = s_next
            self.total_step += 1
        self.num_episode += 1
        return r_total


class BatchedTrainer(BatchedRollout):
    """Episode loop with learning: TrainerRPC.episode + manage_memory + update_all_agents
    (train_rpc.py:503-553, 734-757, 556-560) for all agents and all environments at once.

    Every env-step contributes E transitions per agent to the learner's device replay (credit assignment through
    `DelayedMDP` exactly as the reference: oldest state/action of the window, newest next state, current reward,
    mask = 1 because episodes are time-limited, train_rpc.py:755); after the episode the learner runs
    `updates_per_episode` batched SAC updates (gradients all-reduced over the process group when there is one)
    and the new actors are uploaded into the simulator's tables.

    The window depth comes from env_rl["delayed_assignment"], a knob of its own as in the reference: it does not follow
    the controller delay (Simulator.set_delay / set_delay_env), and one depth serves every environment of the batch
    whatever their delays."""

    def __init__(self, env, learner, seed=1234, updates_per_episode=1000):
        super().__init__(env, seed=seed)
        import torch
        self.learner = learner
        self.updates_per_episode = int(updates_per_episode)
        dev = learner.device
        idx = torch.as_tensor(self.rl.agent_idx.astype(np.int64), device=dev)        # [A, IN], -1 = pad
        act = torch.as_tensor(self.rl.agent_act.astype(np.int64), device=dev)        # [A, ACT], -1 = pad
        self._idx, self._idx_ok = idx.clamp(min=0), (idx >= 0).float()
        self._act, self._act_ok = act.clamp(min=0), (act >= 0).float()

    def states_per_agent(self, state):
        """[E, state_dim] -> [A, E, IN] (zero padded; TrainerRPC.divide_states_for_agents, train_rpc.py:418-427)."""
        return state[:, self._idx].permute(1, 0, 2) * self._idx_ok[:, None, :]

    def actions_per_agent(self, action):
        """[E, action_dim] -> [A, E, ACT] (select_correct_modes_for_array, train_rpc.py:650-665)."""
        return action[:, self._act].permute(1, 0, 2) * self._act_ok[:, None, :]

    def _push(self, s0, a0, s2, r):
        import torch
        mem = self.learner.memory
        ctrl = self.sim.controller_env
        if ctrl is not None:
            # per-environment controllers: the learner trains slot 0; integrator rows carry no action and the other
            # slots' transitions are not the trained actor's
            i = torch.as_tensor(np.flatnonzero(ctrl == 0), device=r.device)
            if i.numel() == 0:
                return
            s0, a0, s2, r = s0[i], a0[i], s2[i], r[i]
        mem.push(self.states_per_agent(s0), self.actions_per_agent(a0), r.t().contiguous(),
                 self.states_per_agent(s2), torch.ones_like(r.t()))

    def train_episode(self, steps=None, updates=None):
        r_total = self.episode(steps=steps, on_transition=self._push)
        n = self.updates_per_episode if updates is None else int(updates)
        stats = None
        if len(self.learner.memory) > self.learner.batch_size:
            for _ in range(n):
                stats = self.learner.update()
            self.learner.upload_actors(self.sim)
        return r_total, stats


class StepLearner:
    """Config 5 without the gym wrapper: the simulator's fused step on the main stream, one batched SAC update of every
    agent per env-step on a second stream (the reference runs updates_per_episode_rpc = 1000 updates per 1000-step
    episode per agent, GlobalConfig.py:63, train_rpc.py:759-781, 1084-1133), gradients all-reduced over the process
    group when there is one.  Transitions go to the learner's device replay with the credit assignment window of
    `DelayedMDP` (oldest state / action, newest next state, current reward; train_rpc.py:734-757).  Its depth is
    env_rl["delayed_assignment"] (or `depth`), set by the user as in the reference and independent of the controller
    delay: per-environment delays (Simulator.set_delay_env) share the batch's one window."""

    def __init__(self, sim, rl, learner, depth=None):
        import torch
        self.torch = torch
        self.sim, self.rl, self.learner = sim, rl, learner
        dev = learner.device
        idx = torch.as_tensor(rl.agent_idx.astype(np.int64), device=dev)
        act = torch.as_tensor(rl.agent_act.astype(np.int64), device=dev)
        self._idx, self._idx_ok = idx.clamp(min=0), (idx >= 0).float()
        self._act, self._act_ok = act.clamp(min=0), (act >= 0).float()
        e = rl.env_rl
        self.mdp = DelayedMDP(e["delayed_assignment"], e["modification_online"]) if depth is None else DelayedMDP(depth, False)
        self.stream = torch.cuda.Stream()
        self.E = sim.n_env
        self._s = sim.rows("STATE", rl.state_dim).clone()
        # env-steps so far, and per environment the step that returned its s0 (0: the state at construction); a
        # transition of environment e is pushed only when the whole window lies after that step
        self._t = 0
        self._first = np.zeros(self.E, dtype=np.int64)
        self._ctrl = np.zeros(self.E, dtype=np.int32)      # controllers of the last step (Simulator.controller_env)

    def reset_envs(self, envs, seeds):
        """Autoreset of the environments `envs` with `seeds` (Simulator.reset_envs): their next step returns their s0, and
        from then on they push exactly what a StepLearner started after a full reset and linear step pushes.  No
        transition spans two episodes.  Set the new episode's conditions before the call."""
        self.sim.reset_envs(envs, seeds)
        self._first[np.asarray(envs, dtype=np.int64)] = self._t + 1

    def load_envs(self, envs, snap):
        """Resume the environments `envs` from records of Simulator.save_envs.  Their credit-assignment window restarts as
        after reset_envs: no transition spans the load."""
        self.sim.load_envs(envs, snap)
        self._first[np.asarray(envs, dtype=np.int64)] = self._t + 1

    def copy_envs(self, src, dst):
        """Environments `dst` continue as copies of environments `src`; their windows restart as in load_envs."""
        self.load_envs(dst, self.sim.save_envs(src))

    def states_per_agent(self, state):
        return state[:, self._idx].permute(1, 0, 2) * self._idx_ok[:, None, :]

    def actions_per_agent(self, action):
        return action[:, self._act].permute(1, 0, 2) * self._act_ok[:, None, :]

    def step(self, learn=True, overlap=True):
        """One env-step of the whole batch + (learn) one SAC update of all agents, the update on the second stream while
        the step runs (overlap) or after it."""
        torch = self.torch
        sim, rl, L = self.sim, self.rl, self.learner
        main = torch.cuda.current_stream()
        can_learn = learn and len(L.memory) > L.batch_size
        # per-environment controllers: only slot 0 (the trained actor) pushes, and an environment whose controller
        # changed restarts its window at the current state, so that no transition mixes two controllers
        ctrl = sim.controller_env
        ctrl = np.zeros(self.E, dtype=np.int32) if ctrl is None else ctrl
        changed = ctrl != self._ctrl
        self._first[changed] = np.maximum(self._first[changed], self._t)
        self._ctrl = ctrl
        if can_learn and overlap:
            self.stream.wait_stream(main)
            with torch.cuda.stream(self.stream):
                L.update()
        sim.step(mode=0)
        self._t += 1
        a = sim.rows("ACTION", rl.action_dim).clone()
        r = sim.buffer("REWARD").view(self.E, rl.n_agents).clone()
        s_next = sim.rows("STATE", rl.state_dim).clone()
        if can_learn and not overlap:
            L.update()
        if can_learn and overlap:
            main.wait_stream(self.stream)          # the replay is written below; the new actors are uploaded by the caller
        if self.mdp.check_update_possibility():
            s0, a0, s2 = self.mdp.credit_assignment()
            ok = (self._first <= self._t - self.mdp.depth - 1) & (ctrl == 0)   # the oldest state of the window is the episode's
            if not ok.all():
                i = torch.as_tensor(np.flatnonzero(ok), device=r.device)
                s0, a0, s2, r = s0[i], a0[i], s2[i], r[i]
            if ok.any():
                L.memory.push(self.states_per_agent(s0), self.actions_per_agent(a0), r.t().contiguous(),
                              self.states_per_agent(s2), torch.ones_like(r.t()))
        self.mdp.save(self._s, a, s_next)
        self._s = s_next
