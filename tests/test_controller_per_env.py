"""Per-environment controllers (aom_set_controller_env, Simulator.set_controller_env): several actor policies and the
integrator side by side in one batch.  Every environment computes bit for bit what it computes in a uniform batch with
its policy in slot 0, or stepped with mode 2 for the integrator: mixed batches, switches, copies, partial resets.  Every
comparison is exact, except the oracle's (1e-4 as in test_gpu_parity.py)."""
import copy
import types

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

STEPS = 10
CYCLE = np.array([1, 0, -1, 2, 0, 2, 1, -1])     # slots interleaved with the integrator, not contiguous
KEYS = ("ACTION", "ACTION_MEAN", "COM", "VOLTS", "SLOPES", "STATE", "REWARD")
SYSTEMS = {
    "10x10": ("production_sh_10x10_2m.py", 300, dict(n_zernike_start_end=[0, 80], n_reverse_filtered_from_cmat=5), 3),
    "40x40": ("production_sh_40x40_8m_3layers.py", 200,
              dict(n_zernike_start_end=[0, 1260], window_n_zernike=20, include_tip_tilt_windowed=True,
                   n_reverse_filtered_from_cmat=5, delayed_assignment=2), 44),
}


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def draw(rl, seed):
    """Policies of the layout's shapes with non-zero heads (the default last-layer init makes every policy alike)."""
    import torch
    g = torch.Generator().manual_seed(seed)
    pols = [copy.deepcopy(p) for p in rl.policies]
    with torch.no_grad():
        for p in pols:
            for w in p.parameters():
                w.copy_(torch.randn(tuple(w.shape), generator=g) * (0.05 if w.dim() > 1 else 0.1))
            p.log_std_linear.bias.fill_(-1.0)
    return pols


class System:
    def __init__(self, name, torch):
        from ao_marl_b200.system import build_system
        par, E, env_rl, ws = SYSTEMS[name]
        self.sim, self.t, self.rl = build_system(par, E, env_rl=env_rl, world_size=ws, seed=3)
        self.E, self.torch = E, torch
        self.sim.set_wfs_noise(0.0)                                   # photon noise: shared by both sides of a pair
        self.pols = {k: draw(self.rl, 100 + k) for k in range(3)}
        for k, p in self.pols.items():
            self.rl.upload_actors(self.sim, slot=k, policies=p)
        self.ctrl = CYCLE[np.arange(E) % CYCLE.size].astype(np.int32)
        self.seeds = 5000 + 7 * np.arange(E, dtype=np.int64)

    def uniform(self, k):
        """Every environment on slot 0, which holds policy k (k = -1: the integrator, stepped with mode 2)."""
        self.sim.set_controller_env(None)
        if k >= 0:
            self.rl.upload_actors(self.sim, slot=0, policies=self.pols[k])
        return 2 if k < 0 else 0

    def restore(self):
        self.sim.set_controller_env(None)
        self.rl.upload_actors(self.sim, slot=0, policies=self.pols[0])

    def rows(self):
        sim, t, rl, E = self.sim, self.t, self.rl, self.E
        n = dict(ACTION=rl.action_dim, ACTION_MEAN=rl.action_dim, COM=t.nactu, VOLTS=t.nactu, SLOPES=t.nslopes,
                 STATE=rl.state_dim)
        out = {k: sim.rows(k, v).cpu().numpy().copy() for k, v in n.items()}
        out["REWARD"] = sim.buffer("REWARD").view(E, rl.n_agents).cpu().numpy().copy()
        return out

    def run(self, steps, modes=0, eval_mode=False, before=None, seeds=None, linear=False):
        """reset (+ the linear step that follows one), then `steps` aom_step calls of modes[i]; before(i) ahead of step i.
        ACTION_MEAN (not cleared by a reset) starts at zero.  Rows after every step."""
        sim = self.sim
        sim.reset(self.seeds if seeds is None else seeds)
        sim.buffer("ACTION_MEAN").zero_()
        out = []
        if linear:
            sim.state_begin(); sim.move_atmos(); sim.comp_wfs_image(); sim.do_centroids(); sim.do_control(); sim.state_end()
            out.append(self.rows())
        for i in range(steps):
            if before is not None:
                before(i)
            sim.step(mode=modes if np.isscalar(modes) else modes[i], eval_mode=eval_mode)
            out.append(self.rows())
        sim.check_device()
        return out


@pytest.fixture(scope="module", params=list(SYSTEMS))
def system(request, torch):
    s = System(request.param, torch)
    yield s
    s.sim.close()


@pytest.fixture(scope="module")
def system10(torch):
    s = System("10x10", torch)
    yield s
    s.sim.close()


def same_rows(a, b, rows, what, keys=KEYS):
    assert rows.size > 0
    for i, (x, y) in enumerate(zip(a, b)):
        for k in keys:
            assert np.array_equal(x[k][rows], y[k][rows]), (what, i, k)


@pytest.mark.parametrize("eval_mode", [False, True])
def test_mixed_batch(system, eval_mode):
    """Slots 0, 1, 2 and the integrator interleaved over a ragged batch: each environment's rows of every step equal
    those of the uniform batch of its controller."""
    s = system
    try:
        s.sim.set_controller_env(s.ctrl)
        assert np.array_equal(s.sim.controller_env, s.ctrl)
        got = s.run(STEPS, eval_mode=eval_mode)
        refs = {}
        for k in (0, 1, 2, -1):
            refs[k] = s.run(STEPS, modes=s.uniform(k), eval_mode=eval_mode)
            same_rows(got, refs[k], np.flatnonzero(s.ctrl == k), ("controller", k))
        # the policies differ: a slot-1 environment does not act as slot 0 would, and integrator rows carry no action
        one = np.flatnonzero(s.ctrl == 1)
        assert not np.array_equal(got[-1]["ACTION"][one], refs[0][-1]["ACTION"][one])
        assert not (got[-1]["ACTION"][np.flatnonzero(s.ctrl == -1)]).any()
    finally:
        s.restore()


def test_switching(system):
    """A -> integrator -> B, four steps each (A = e % 3, B = (e + 1) % 3): each environment equals the uniform batch that
    ran A, then mode 2, then B uploaded into slot 0."""
    s = system
    E, n = s.E, 4
    a = (np.arange(E) % 3).astype(np.int32)
    b = ((np.arange(E) + 1) % 3).astype(np.int32)
    phases = {0: a, n: np.full(E, -1, np.int32), 2 * n: b}
    try:
        s.sim.set_controller_env(None)
        got = s.run(3 * n, before=lambda i: i in phases and s.sim.set_controller_env(phases[i]))
        for k in range(3):
            kb = (k + 1) % 3

            def switch(i, kb=kb):
                if i == 2 * n:
                    s.rl.upload_actors(s.sim, slot=0, policies=s.pols[kb])
            s.uniform(k)
            ref = s.run(3 * n, modes=[0] * n + [2] * n + [0] * n, before=switch)
            same_rows(got, ref, np.flatnonzero(a == k), ("A", k))
    finally:
        s.restore()


def test_copy_envs_across_controllers(system):
    """Environments copied into slots of other controllers: each branch equals a uniform context that loaded the same
    record and holds the destination's controller."""
    s = system
    E, at, after = s.E, 5, 5
    src = np.array([1, 2, 3, 4])
    want = {1: 1, 2: 0, 3: -1, 4: 2}                                # destination controller per source
    dst = np.array([np.flatnonzero((s.ctrl == want[e]) & (np.arange(E) > 150))[0] for e in src])
    assert (s.ctrl[src] != s.ctrl[dst]).all()
    rec = {}
    try:
        s.sim.set_controller_env(s.ctrl)

        def copy_at(i):
            if i == at:
                rec["r"] = s.sim.save_envs(src)
                s.sim.load_envs(dst, rec["r"])
        got = s.run(at + after, before=copy_at)[at:]
        assert np.array_equal(s.sim.controller_env, s.ctrl)           # the destination keeps its controller
        for k in (0, 1, 2, -1):
            rows = dst[s.ctrl[dst] == k]
            ref = s.run(after, modes=s.uniform(k), before=lambda i: i == 0 and s.sim.load_envs(dst, rec["r"]))
            same_rows(got, ref, rows, ("copy", k))
    finally:
        s.restore()


def test_reset_envs_in_mixed_batch(system):
    """reset_envs of environments on every controller: their fresh step gives the s0 of a freshly reset uniform batch of
    their controller, every later step equals that batch; the assignment persists."""
    s = system
    E, at, after = s.E, 4, 5
    envs = np.array([np.flatnonzero(s.ctrl == k)[3] for k in (0, 1, 2, -1)])
    new = 90000 + envs.astype(np.int64)
    seeds_c = s.seeds.copy()
    seeds_c[envs] = new
    try:
        s.sim.set_controller_env(s.ctrl)
        got = s.run(at + after, before=lambda i: i == at and s.sim.reset_envs(envs, new))[at:]
        assert np.array_equal(s.sim.controller_env, s.ctrl)
        for k in (0, 1, 2, -1):
            rows = envs[s.ctrl[envs] == k]
            ref = s.run(after - 1, modes=s.uniform(k), seeds=seeds_c, linear=True)
            same_rows(got[:1], ref[:1], rows, ("fresh", k), keys=("STATE", "COM", "SLOPES"))
            assert not got[0]["REWARD"][rows].any()
            same_rows(got[1:], ref[1:], rows, ("after", k))
    finally:
        s.restore()


def test_actions_against_oracle(system10):
    """10x10: each environment's actions equal the oracle's actors of its slot on the GPU's state (1e-4)."""
    from oracle import loop
    s = system10
    worst = 0.0
    try:
        s.sim.set_controller_env(s.ctrl)
        s.sim.reset(s.seeds)
        for i in range(4):
            st = s.sim.rows("STATE", s.rl.state_dim).cpu().numpy().copy()
            s.sim.step(mode=0)
            act = s.sim.rows("ACTION", s.rl.action_dim).cpu().numpy()
            for e in range(0, s.E, 7):
                if s.ctrl[e] < 0:
                    continue
                rl = copy.copy(s.rl)
                rl.policies = s.pols[int(s.ctrl[e])]
                o = types.SimpleNamespace(rl=rl, seed=int(s.seeds[e]), step_count=i)
                a, _ = loop.OracleEnv.actors(o, st[e])
                worst = max(worst, np.abs(act[e] - a).max() / max(np.abs(a).max(), 1e-30))
        s.sim.check_device()
    finally:
        s.restore()
    assert worst < 1e-4, worst


def test_errors_leave_the_assignment(system10, torch):
    s = system10
    sim = s.sim
    try:
        sim.set_controller_env(s.ctrl)
        for bad in (np.where(s.ctrl == 2, 8, s.ctrl), np.where(s.ctrl == 2, -2, s.ctrl), s.ctrl[:-1]):
            with pytest.raises(ValueError):
                sim.set_controller_env(bad)
            assert np.array_equal(sim.controller_env, s.ctrl)
        with pytest.raises(RuntimeError, match="slot 5"):
            sim.set_controller_env(np.where(s.ctrl == 2, 5, s.ctrl))
        assert np.array_equal(sim.controller_env, s.ctrl)
        sim.reset(s.seeds)
        sim.set_gemm_path("simt")
        try:
            with pytest.raises(RuntimeError, match="per-environment controllers"):
                sim.actor_forward()
            with pytest.raises(RuntimeError, match="per-environment controllers"):
                sim.step(mode=0)
        finally:
            sim.set_gemm_path("tcgen05")
        sim.set_controller_env(np.zeros(s.E, np.int32))              # slot 0 everywhere is the uniform state
        assert sim.controller_env is None
        sim.step(mode=0)
        sim.check_device()
    finally:
        s.restore()


def test_upload_into_slot_1_leaves_slot_0(system10):
    """Weights uploaded at index 1 do not change the actions of a uniform batch (they once replaced the pre-split copy
    of slot 0's weights)."""
    s = system10
    try:
        s.sim.set_controller_env(None)
        a = s.run(3)
        s.rl.upload_actors(s.sim, slot=1, policies=s.pols[2])
        b = s.run(3)
        same_rows(a, b, np.arange(s.E), "slot 1 upload", keys=("ACTION", "ACTION_MEAN", "COM"))
    finally:
        s.rl.upload_actors(s.sim, slot=1, policies=s.pols[1])
        s.restore()


def test_step_learner_pushes_slot_0_only(system10, torch):
    """StepLearner (learn=False) with mixed controllers: every push holds exactly the slot-0 environments, their rewards
    in order."""
    from ao_marl_b200.env.trainer import StepLearner
    from ao_marl_b200.rl.sac import BatchedSAC
    s = system10
    zero = np.flatnonzero(s.ctrl == 0)
    try:
        s.sim.set_controller_env(s.ctrl)
        s.sim.reset(s.seeds)
        L = BatchedSAC.from_layout(s.rl, device="cuda", seed=3, memory_size=4096)
        sl = StepLearner(s.sim, s.rl, L)
        pushes = 0
        for g in range(1, 9):
            pos = L.memory.position
            sl.step(learn=False)
            n = L.memory.position - pos
            assert n in (0, zero.size), (g, n)
            if n:
                pushes += 1
                r = s.sim.buffer("REWARD").view(s.E, s.rl.n_agents)[torch.as_tensor(zero, device="cuda")]
                assert torch.equal(L.memory.r[:, pos:pos + n], r.t()), g
        assert pushes > 0
        s.sim.check_device()
    finally:
        s.restore()
