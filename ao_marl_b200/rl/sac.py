"""Batched soft actor-critic learner: every agent of an experiment updated in one set of batched GEMMs.

The reference trains one `SAC` object per agent in its own RPC process (src/reinforcement_learning/
rpc_training/train_rpc.py:792-1161): twin Q networks `QNetwork` (algorithms_rpc/model_rpc.py:17-69), the
tanh-Gaussian `GaussianPolicy` (model_rpc.py:70-158), automatic entropy tuning with target entropy -|A|
(train_rpc.py:858-876), one Adam per network, `updates_per_episode_rpc` updates per episode on batches drawn
from a per-agent `ReplayMemory` (algorithms_rpc/replay_memory_rpc.py).  Here the A agents are stacked along a
leading dimension -- parameters `[A, out, in]`, zero-padded to the widest agent -- so one update of all agents
is a handful of `torch.baddbmm` calls with autograd; each agent keeps its own losses, its own Adam moments
(element-wise, so stacking changes nothing) and its own temperature.  Update order and formulas follow
`update_parameters_sac` (train_rpc.py:1084-1133): critic (1016-1037, Bellman backup 987-1002), actor
(1050-1062), temperature (1068-1082), soft target update (utils.py:22-24).

Experience is pooled over the batched environments: every env-step contributes E transitions per agent to a
device-resident ring (`DeviceReplay`).  With several GPUs each rank keeps the replay shard of its own
environments, and `BatchedSAC.update` all-reduces (averages) the flattened gradients of every optimiser step
over the process group (NCCL over NVLink on the GPU box, gloo in the CPU tests), so the replicated weights stay
bit-identical without a broadcast (SURVEY.md 8(e)).

PyTorch is the engine here by design (BASELINE.json north_star: "PyTorch only for tensors and the SAC
networks"); the stepping path consumes the actors through `pack_for_sim` + aom_actor_forward.
"""
import math

import numpy as np
import torch

LOG_SIG_MIN = -20.0
EPS = 1e-5          # model_rpc.py:13


def _xavier_(w, fan_in, fan_out, gen):
    bound = math.sqrt(6.0 / (fan_in + fan_out))
    w.uniform_(-bound, bound, generator=gen)


class DeviceReplay:
    """Per-agent transition ring on the device: state / action / reward / next state / mask, `[A, capacity, .]`."""

    def __init__(self, n_agents, capacity, state_dim, action_dim, device):
        self.A, self.capacity = n_agents, int(capacity)
        z = lambda *s: torch.zeros(s, device=device)
        self.s, self.s2 = z(n_agents, capacity, state_dim), z(n_agents, capacity, state_dim)
        self.a, self.r, self.m = z(n_agents, capacity, action_dim), z(n_agents, capacity), z(n_agents, capacity)
        self.position = 0
        self.size = 0

    def __len__(self):
        return self.size

    def reset(self):
        self.position = self.size = 0

    def push(self, s, a, r, s2, mask):
        """s, s2 [A, n, S]; a [A, n, U]; r, mask [A, n] -- n transitions per agent (one per environment)."""
        n = s.shape[1]
        if n > self.capacity:
            raise ValueError("Dimension mismatch: %d transitions pushed into a ring of %d" % (n, self.capacity))
        idx = (self.position + torch.arange(n, device=s.device)) % self.capacity
        self.s[:, idx], self.a[:, idx], self.r[:, idx], self.s2[:, idx], self.m[:, idx] = s, a, r, s2, mask
        self.position = (self.position + n) % self.capacity
        self.size = min(self.size + n, self.capacity)

    def sample(self, batch_size, generator=None):
        idx = torch.randint(0, self.size, (self.A, batch_size), device=self.s.device, generator=generator)
        return self.gather(idx)

    def gather(self, idx):
        ar = torch.arange(self.A, device=idx.device)[:, None]
        return self.s[ar, idx], self.a[ar, idx], self.r[ar, idx], self.s2[ar, idx], self.m[ar, idx]


class _Stack(torch.nn.Module):
    """A agents' MLPs as stacked parameters: layer i maps [A, B, d_i] -> [A, B, d_{i+1}] with baddbmm."""

    def __init__(self, n_agents, dims, gen, fan_in_first=None):
        super().__init__()
        self.W = torch.nn.ParameterList()
        self.b = torch.nn.ParameterList()
        for i in range(len(dims) - 1):
            w = torch.zeros(n_agents, dims[i + 1], dims[i])
            self.W.append(torch.nn.Parameter(w))
            self.b.append(torch.nn.Parameter(torch.zeros(n_agents, dims[i + 1])))
        self.dims = list(dims)

    def layer(self, i, x):
        return torch.baddbmm(self.b[i][:, None, :], x, self.W[i].transpose(1, 2))


class BatchedSAC:
    """All agents' critics, actors and temperatures; see the module docstring.

    in_dims / act_dims: per-agent true sizes (inputs beyond them are zero padding and stay inert because the
    corresponding weight columns start at zero and receive zero gradients; padded action columns are masked).
    """

    def __init__(self, in_dims, act_dims, sac, device="cuda", seed=0, dist=None, memory_size=None):
        self.cfg = s = dict(sac)
        self.device = torch.device(device)
        self.dist = dist
        self.A = len(in_dims)
        self.in_dims, self.act_dims = list(map(int, in_dims)), list(map(int, act_dims))
        self.IN, self.ACT = max(self.in_dims), max(self.act_dims)
        self.gamma, self.tau, self.lr = float(s["gamma"]), float(s["tau"]), float(s["lr"])
        self.batch_size = int(s["batch_size"])
        self.target_update_interval = int(s.get("target_update_interval", 1))
        self.auto_alpha = bool(s.get("automatic_entropy_tuning", True))
        self.log_sig_max = float(s.get("LOG_SIG_MAX", 2.0))
        self.action_scale, self.action_bias = float(s.get("gaussian_std", 1.0)), float(s.get("gaussian_mu", 0.0))
        H = int(s.get("hidden_size_actor", 256))
        La = int(s.get("num_layers_actor", 2))
        hc = s.get("hidden_size_critic", 256)
        # reference: a list gives len-1 hidden-to-hidden layers, a scalar gives num_layers_critic-1 (model_rpc.py:25-52)
        hc_dims = list(hc) if isinstance(hc, (list, tuple)) else [int(hc)] * int(s.get("num_layers_critic", 2))
        gen = torch.Generator().manual_seed(int(seed))
        A = self.A
        self.actor = _Stack(A, [self.IN] + [H] * La, gen)
        self.head = _Stack(A, [H, 2 * self.ACT], gen)              # mean rows then log-std rows
        self.q = torch.nn.ModuleList(_Stack(A, [self.IN + self.ACT] + hc_dims + [1], gen) for _ in range(2))
        self.q_target = torch.nn.ModuleList(_Stack(A, [self.IN + self.ACT] + hc_dims + [1], gen) for _ in range(2))
        with torch.no_grad():
            act_mask = torch.zeros(A, self.ACT)
            in_mask = torch.zeros(A, self.IN)
            for a in range(A):
                nin, nact = self.in_dims[a], self.act_dims[a]
                act_mask[a, :nact] = 1
                in_mask[a, :nin] = 1
                for i, W in enumerate(self.actor.W):
                    fi = nin if i == 0 else H
                    _xavier_(W[a, :, :fi], fi, H, gen)
                if not s.get("initialize_last_layer_0", True):
                    gain = 1e-4 if s.get("initialize_last_layer_near_0", False) else 1.0
                    for off in (0, self.ACT):
                        _xavier_(self.head.W[0][a, off:off + nact], H, nact, gen)
                        self.head.W[0][a, off:off + nact] *= gain
                for net in self.q:
                    for i, W in enumerate(net.W):
                        if i == 0:      # [state | pad | action | pad]: only the live columns are initialised
                            cols = torch.cat([torch.arange(nin), self.IN + torch.arange(nact)])
                            w = torch.empty(W.shape[1], nin + nact)
                            _xavier_(w, nin + nact, W.shape[1], gen)
                            W[a][:, cols] = w
                        else:
                            _xavier_(W[a], W.shape[2], W.shape[1], gen)
        self.act_mask, self.in_mask = act_mask.to(self.device), in_mask.to(self.device)
        for m in (self.actor, self.head, self.q, self.q_target):
            m.to(self.device)
        self.hard_update()
        self.log_alpha = torch.zeros(A, device=self.device, requires_grad=True)
        self.alpha_fixed = float(s.get("alpha", 0.2))
        self.target_entropy = -torch.tensor(self.act_dims, dtype=torch.float32, device=self.device)
        Adam = torch.optim.Adam
        wd = float(s.get("l2_norm_policy", -1))
        self.actor_params = list(self.actor.parameters()) + list(self.head.parameters())
        self.critic_params = list(self.q.parameters())
        self.policy_optim = Adam(self.actor_params, lr=self.lr, weight_decay=wd if wd > 0 else 0)
        self.critic_optim = Adam(self.critic_params, lr=self.lr)
        self.alpha_optim = Adam([self.log_alpha], lr=self.lr)
        cap = int(memory_size if memory_size is not None else s.get("memory_size", 1000000))
        self.memory = DeviceReplay(A, cap, self.IN, self.ACT, self.device)
        self.updates = 0
        self.sample_gen = torch.Generator(device=self.device).manual_seed(int(seed) + 1)

    # -- networks --------------------------------------------------------------------------------
    @property
    def alpha(self):
        return self.log_alpha.exp().detach() if self.auto_alpha else torch.full((self.A,), self.alpha_fixed,
                                                                                device=self.device)

    def policy_forward(self, state):
        x = state
        for i in range(len(self.actor.W)):
            x = torch.relu(self.actor.layer(i, x))
        out = self.head.layer(0, x)
        mean, log_std = out[..., :self.ACT], out[..., self.ACT:]
        return mean, torch.clamp(log_std, min=LOG_SIG_MIN, max=self.log_sig_max)

    def policy_sample(self, state, noise=None):
        """(action, log_prob [A, B], tanh-mean) as GaussianPolicy.sample (model_rpc.py:131-158), padded action
        columns masked out of the log-probability and zeroed in the action."""
        mean, log_std = self.policy_forward(state)
        std = log_std.exp()
        eps = torch.randn_like(mean) if noise is None else noise
        x_t = mean + std * eps
        y_t = torch.tanh(x_t)
        m = self.act_mask[:, None, :]
        action = (y_t * self.action_scale + self.action_bias) * m
        log_prob = -0.5 * eps.pow(2) - log_std - 0.5 * math.log(2 * math.pi)
        log_prob = log_prob - torch.log(self.action_scale * (1 - y_t.pow(2).clamp(min=0, max=1)) + EPS)
        log_prob = (log_prob * m).sum(-1)
        return action, log_prob, (torch.tanh(mean) * self.action_scale + self.action_bias) * m

    def q_forward(self, nets, state, action):
        x0 = torch.cat([state, action], -1)
        out = []
        for net in nets:
            x = x0
            n = len(net.W)
            for i in range(n):
                x = net.layer(i, x)
                if i < n - 1:
                    x = torch.relu(x)
            out.append(x[..., 0])
        return out

    def hard_update(self):
        with torch.no_grad():
            for t, s in zip(self.q_target.parameters(), self.q.parameters()):
                t.copy_(s)

    def soft_update(self):
        with torch.no_grad():
            for t, s in zip(self.q_target.parameters(), self.q.parameters()):
                t.mul_(1.0 - self.tau).add_(s, alpha=self.tau)

    # -- one update of every agent ---------------------------------------------------------------
    def _allreduce(self, params):
        d = self.dist
        if d is None or not d.is_initialized() or d.get_world_size() == 1:
            return
        flat = torch.cat([p.grad.reshape(-1) for p in params])
        d.all_reduce(flat, op=d.ReduceOp.SUM)
        flat /= d.get_world_size()
        off = 0
        for p in params:
            n = p.numel()
            p.grad.copy_(flat[off:off + n].view_as(p))
            off += n

    def update(self, batch=None, noise=None):
        """One SAC update of all agents (train_rpc.py:1110-1124).  batch: (s, a, r, s2, mask) stacked [A, B, .]
        (default: a fresh sample of the local replay shard); noise: optional (eps_next, eps_pi) N(0,1) draws."""
        s, a, r, s2, mask = batch if batch is not None else self.memory.sample(self.batch_size, self.sample_gen)
        n0, n1 = noise if noise is not None else (None, None)
        alpha = self.alpha
        with torch.no_grad():
            a2, logp2, _ = self.policy_sample(s2, n0)
            q1t, q2t = self.q_forward(self.q_target, s2, a2)
            target = r + mask * self.gamma * (torch.min(q1t, q2t) - alpha[:, None] * logp2)
        q1, q2 = self.q_forward(self.q, s, a)
        qf1 = (q1 - target).pow(2).mean(1)           # per agent: F.mse_loss over the batch
        qf2 = (q2 - target).pow(2).mean(1)
        for p in self.critic_params:
            p.grad = None
        (qf1 + qf2).sum().backward()
        self._allreduce(self.critic_params)
        self.critic_optim.step()

        pi, logp, _ = self.policy_sample(s, n1)
        q1p, q2p = self.q_forward(self.q, s, pi)
        policy_loss = (alpha[:, None] * logp - torch.min(q1p, q2p)).mean(1)
        for p in self.actor_params:
            p.grad = None
        policy_loss.sum().backward(inputs=self.actor_params)
        self._allreduce(self.actor_params)
        self.policy_optim.step()

        alpha_loss = torch.zeros(self.A, device=self.device)
        if self.auto_alpha:
            alpha_loss = -(self.log_alpha * (logp.detach() + self.target_entropy[:, None]).mean(1))
            self.log_alpha.grad = None
            alpha_loss.sum().backward()
            self._allreduce([self.log_alpha])
            self.alpha_optim.step()
        self.updates += 1
        if self.updates % self.target_update_interval == 0:
            self.soft_update()
        for p in self.critic_params:
            p.grad = None
        return dict(qf1=qf1.detach(), qf2=qf2.detach(), policy=policy_loss.detach(), alpha_loss=alpha_loss.detach(),
                    alpha=self.alpha)

    # -- exchange with the reference's per-agent modules and with the simulator -----------------------
    def actor_state_dict(self, a):
        """`GaussianPolicy.state_dict()` of agent a (reference parameter names, true sizes)."""
        nin, nact = self.in_dims[a], self.act_dims[a]
        sd = {"linear1.weight": self.actor.W[0][a, :, :nin], "linear1.bias": self.actor.b[0][a]}
        for i in range(1, len(self.actor.W)):
            sd["hidden.%d.weight" % (i - 1)] = self.actor.W[i][a]
            sd["hidden.%d.bias" % (i - 1)] = self.actor.b[i][a]
        sd["mean_linear.weight"] = self.head.W[0][a, :nact]
        sd["mean_linear.bias"] = self.head.b[0][a, :nact]
        sd["log_std_linear.weight"] = self.head.W[0][a, self.ACT:self.ACT + nact]
        sd["log_std_linear.bias"] = self.head.b[0][a, self.ACT:self.ACT + nact]
        return {k: v.detach().clone() for k, v in sd.items()}

    def load_actor_state_dict(self, a, sd):
        nin, nact = self.in_dims[a], self.act_dims[a]
        with torch.no_grad():
            self.actor.W[0][a].zero_()
            self.actor.W[0][a, :, :nin] = sd["linear1.weight"]
            self.actor.b[0][a] = sd["linear1.bias"]
            for i in range(1, len(self.actor.W)):
                self.actor.W[i][a] = sd["hidden.%d.weight" % (i - 1)]
                self.actor.b[i][a] = sd["hidden.%d.bias" % (i - 1)]
            self.head.W[0][a].zero_()
            self.head.b[0][a].zero_()
            self.head.W[0][a, :nact] = sd["mean_linear.weight"]
            self.head.b[0][a, :nact] = sd["mean_linear.bias"]
            self.head.W[0][a, self.ACT:self.ACT + nact] = sd["log_std_linear.weight"]
            self.head.b[0][a, self.ACT:self.ACT + nact] = sd["log_std_linear.bias"]

    def critic_state_dict(self, a, target=False):
        """`QNetwork.state_dict()` of agent a (reference names Q{1,2}_input / hidden_Q{1,2}.N / Q{1,2}_output)."""
        nin, nact = self.in_dims[a], self.act_dims[a]
        cols = torch.cat([torch.arange(nin), self.IN + torch.arange(nact)]).to(self.device)
        sd = {}
        for qi, net in enumerate(self.q_target if target else self.q, start=1):
            n = len(net.W)
            for i in range(n):
                name = "Q%d_input" % qi if i == 0 else ("Q%d_output" % qi if i == n - 1 else "hidden_Q%d.%d" % (qi, i - 1))
                sd[name + ".weight"] = net.W[i][a][:, cols] if i == 0 else net.W[i][a]
                sd[name + ".bias"] = net.b[i][a]
        return {k: v.detach().clone() for k, v in sd.items()}

    def load_critic_state_dict(self, a, sd):
        nin, nact = self.in_dims[a], self.act_dims[a]
        cols = torch.cat([torch.arange(nin), self.IN + torch.arange(nact)]).to(self.device)
        with torch.no_grad():
            for qi, (net, tnet) in enumerate(zip(self.q, self.q_target), start=1):
                n = len(net.W)
                for i in range(n):
                    name = "Q%d_input" % qi if i == 0 else ("Q%d_output" % qi if i == n - 1 else "hidden_Q%d.%d" % (qi, i - 1))
                    if i == 0:
                        net.W[i][a].zero_()
                        net.W[i][a][:, cols] = sd[name + ".weight"]
                    else:
                        net.W[i][a] = sd[name + ".weight"]
                    net.b[i][a] = sd[name + ".bias"]
                    tnet.W[i][a] = net.W[i][a]
                    tnet.b[i][a] = net.b[i][a]

    def checkpoint(self, a, worker_id, modes_controlled):
        """The reference's actor checkpoint dictionary (train_rpc.py:1155-1159)."""
        return {"worker_id": worker_id, "models_controlled": modes_controlled,
                "model_state_dict": {k: v.cpu() for k, v in self.actor_state_dict(a).items()}}

    def pack_for_sim(self):
        """Actor tables in the layout of include/aomarl.h (AOM_T_ACTOR_*), as host arrays for Simulator.set_table."""
        if len(self.actor.W) != 2:
            raise NotImplementedError("the batched actor kernel implements 2 hidden ReLU layers")
        ld = lambda n: (int(n) + 15) & ~15
        A, H = self.A, self.actor.dims[1]

        def pad(w, k):
            out = np.zeros(w.shape[:-1] + (ld(k),), np.float32)
            out[..., :w.shape[-1]] = w.detach().cpu().numpy()
            return out
        return dict(ACTOR_W1=pad(self.actor.W[0], self.IN), ACTOR_B1=self.actor.b[0].detach().cpu().numpy(),
                    ACTOR_W2=pad(self.actor.W[1], H), ACTOR_B2=self.actor.b[1].detach().cpu().numpy(),
                    ACTOR_WH=pad(self.head.W[0], H), ACTOR_BH=self.head.b[0].detach().cpu().numpy())

    def upload_actors(self, sim, slot=0):
        """Upload the current actors into policy slot `slot` of the simulator."""
        for name, arr in self.pack_for_sim().items():
            sim.set_table(name, np.ascontiguousarray(arr, dtype=np.float32), index=slot)

    @classmethod
    def from_layout(cls, rl, device="cuda", seed=0, dist=None, memory_size=None):
        """Learner for the agents of an `RLLayout`, starting from its actors."""
        wids = sorted(rl.agents)
        in_dims = [len(rl.modes_chosen[w]) for w in wids]
        act_dims = [rl.agents[w][1] - rl.agents[w][0] for w in wids]
        self = cls(in_dims, act_dims, rl.sac, device=device, seed=seed, dist=dist, memory_size=memory_size)
        for a, pol in enumerate(rl.policies):
            self.load_actor_state_dict(a, {k: v.to(self.device) for k, v in pol.state_dict().items()})
        return self
