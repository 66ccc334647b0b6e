"""The batched actor forward (aom_actor_forward: actor_gather_kernel, three gemm_tc_kernel launches over the pre-tiled
TF32 hi / lo weight planes with one bias per agent, actor_sample_kernel) against a float64 numpy reference of the same
operation, element by element, inside an error bound derived from the arithmetic rather than fitted to it.

Reference: the float32 arrays that were uploaded (pack_actors) and the STATE rows read back from the device, gathered
through agent_idx, relu(W1 x + b1), relu(W2 h + b2), the heads, the log-std clamped to [-20, LOG_SIG_MAX], the
exploration noise of oracle.rng.actor_noise, tanh, scale and bias, scattered through agent_act.

Bound per output element of a layer: gamma(K) sum_k |w_k| |x_k| + 2^-24 |b|, with gamma(K) = K_pad 2^-22 + 2^-17 on
the tensor cores (2^-17 covers the TF32 truncation of the lo parts and the dropped lo.lo product, K_pad 2^-22 the
truncating float32 accumulator, DESIGN.md) and (K_pad + 1) 2^-24 for the float32 FFMA kernel.  It is carried through
ReLU (1-Lipschitz) and then through |W| into the next layer, and through tanh as
scale sech^2 (bound_mu + |eps| exp(ls) bound_ls) plus a few ulps of expf / tanhf and of the float32 operations.

Shapes: the 10x10 layout (2 agents, 320 inputs, 160 head columns), the headline 40x40 layout (43 agents, 280 inputs, 60
head columns) and 14 agents + tip-tilt (520 inputs, 180 head columns: two column tiles; the tip-tilt agent's unused
slots are -1); hidden sizes 256, 200 (leading dimension 208: a partial second column tile and 13 k-blocks, not a
multiple of the three register sets in flight) and 64 (one partial tile); batches from 1 to 4097 environments, so
single rows, exact and ragged 128-row tiles and the headline 4096.  The largest error / bound ratio of every case is
printed at the end of the module (pytest -s shows it)."""
import json
import time

import numpy as np
import pytest

from oracle import rng as orng

F32, F64 = np.float32, np.float64
U = 2.0 ** -24
LOG_SIG_MIN = -20.0
PAR10 = "production_sh_10x10_2m.py"
PAR40 = "production_sh_40x40_8m_3layers.py"
ENV_RL_43 = dict(n_zernike_start_end=[0, 1260], window_n_zernike=20, include_tip_tilt_windowed=True,
                 n_reverse_filtered_from_cmat=5)
# layout name -> (parameter file, env_rl, world size)
LAYOUTS = {"10x10": (PAR10, dict(n_zernike_start_end=[0, 80], n_reverse_filtered_from_cmat=5), 3),
           "40x40_43": (PAR40, ENV_RL_43, 44),
           "40x40_14tt": (PAR40, ENV_RL_43, 16)}
UNMAPPED = (0, 1)            # (agent, output) whose action slot is taken away: that entry must keep its value
REPORT = {}
TIMES = {}


def record(case, key, value):
    REPORT.setdefault(case, {})[key] = max(value, REPORT.get(case, {}).get(key, 0.0))


@pytest.fixture(scope="module", autouse=True)
def _print_report():
    t0 = time.time()
    yield
    if REPORT:
        print("\nactor forward, largest error / bound per case:\n" + json.dumps(REPORT, indent=1, sort_keys=True))
    if TIMES:
        print("actor forward, wall time per test (s): %s; module %.1f s" % (json.dumps(TIMES, sort_keys=True),
                                                                          time.time() - t0))


def ld(n):
    return (int(n) + 15) & ~15


def gamma(path, K):
    """Relative error of one contraction over K (padded) terms, per unit of sum |w| |x|."""
    Kp = ld(K)
    return Kp * 2.0 ** -22 + 2.0 ** -17 if path == "tcgen05" else (Kp + 1) * U


# ----------------------------------------------------------------------------------------------------------------------
# data: actors with non-trivial heads, states with outliers

def make_layout(name, hidden, seed):
    """RLLayout of `name` with `hidden` units and actors whose biases, heads and log-std are all exercised: random
    biases on every layer (a wrong per-agent bias stride shows), mean weights N(0, 0.05), some means pushed into tanh
    saturation, log-std biases at +5 and -30 on some outputs (both clamps), one action slot unmapped."""
    from ao_marl_b200.rl.layout import RLLayout, load_normalization
    par, env, ws = LAYOUTS[name]
    nm = len(load_normalization(par)[1])
    rl = RLLayout(nm, dict(env, parameters_telescope=par), dict(hidden_size_actor=hidden), world_size=ws, seed=seed)
    perturb_actors(rl, np.random.default_rng(seed))
    a, j = UNMAPPED
    rl.agent_act = rl.agent_act.copy()
    rl.agent_act[a, j] = -1
    return rl


def probe_weights(r, shape):
    """Positive float32 weights 2^e (1 + 2^-10 - 2^-23), e in [-10, -7]: the largest part a TF32 truncation can drop
    (2^-10 of the value), all of the same sign, so that a lost product adds up over the whole contraction."""
    return np.ldexp(F32(1 + 2.0 ** -10 - 2.0 ** -23), r.integers(-10, -6, shape)).astype(F32)


def perturb_actors(rl, r):
    """Agent 0 is a coherent probe: positive W1, W2 and positive head rows for its first half of outputs, so that on a
    non-negative state row every product of every layer has the same sign and an error of the split cannot cancel
    (the bound is per unit of sum |w| |x|; random signs would hide a wrong split below it, see
    test_bound_separates_a_wrong_split).  Its other outputs and the other agents carry the saturation and clamps."""
    import torch
    for a, p in enumerate(rl.policies):
        nout = p.mean_linear.weight.shape[0]
        H, K = p.linear1.weight.shape
        mw, lw = r.normal(0, 0.05, (nout, H)), r.normal(0, 0.05, (nout, H))
        mb = r.normal(0, 0.3, nout)
        sat = r.choice(nout, size=max(1, nout // 6), replace=False)
        mb[sat] = r.choice([-7.0, 7.0], size=sat.size)               # tanh saturated
        lb = np.full(nout, -1.0)
        k = r.permutation(nout)
        lb[k[:max(1, nout // 8)]] = 5.0                              # clamped at LOG_SIG_MAX
        lb[k[max(1, nout // 8):max(2, nout // 4)]] = -30.0           # clamped at LOG_SIG_MIN
        new = {"linear1.bias": r.normal(0, 0.1, H), "hidden.0.bias": r.normal(0, 0.1, H)}
        if a == 0:
            c = nout // 2
            new = {"linear1.weight": probe_weights(r, (H, K)), "hidden.0.weight": probe_weights(r, (H, H)),
                   "linear1.bias": np.zeros(H), "hidden.0.bias": np.zeros(H)}
            mw[:c], lw[:c] = probe_weights(r, (c, H)), probe_weights(r, (c, H))
            mb[:c], lb[:c] = 0.0, -1.0
        new.update({"mean_linear.weight": mw, "mean_linear.bias": mb, "log_std_linear.weight": lw,
                    "log_std_linear.bias": lb})
        sd = p.state_dict()
        with torch.no_grad():
            for key, v in new.items():
                sd[key].copy_(torch.as_tensor(np.asarray(v, F32)))


def other_weights(rl, seed):
    """Weights B of the same shapes as the layout's (another draw of every parameter)."""
    import torch
    r = np.random.default_rng(seed)
    for p in rl.policies:
        with torch.no_grad():
            for name in ("linear1.weight", "hidden.0.weight"):
                w = p.state_dict()[name]
                w.copy_(torch.as_tensor(r.uniform(-1, 1, tuple(w.shape)).astype(F32) * float(w.abs().max())))
    perturb_actors(rl, r)


def probe_rows(E):
    """The first and last environment of every 128-row tile: their state rows are non-negative (coherent probe)."""
    return np.unique(np.concatenate([np.arange(0, E, 128), np.arange(127, E, 128), [E - 1]]))


def make_state(E, n, seed):
    """float32 [E, n] standard normals with a few entries near +-1e3 (as the degenerate modes produce); the probe
    rows are made non-negative."""
    r = np.random.default_rng(seed)
    S = r.standard_normal((E, n)).astype(F32)
    k = max(1, E * n // 500)
    S.reshape(-1)[r.choice(E * n, size=k, replace=False)] = (r.choice([-1.0, 1.0], k) * r.uniform(500, 1500, k)).astype(F32)
    p = probe_rows(E)
    S[p] = np.abs(S[p])
    return S


# ----------------------------------------------------------------------------------------------------------------------
# float64 reference and its bound

def tf32(x):
    """Truncation to TF32 (11 significant bits), as the tensor core reads a float32 register."""
    return (np.asarray(x, F32).view(np.uint32) & np.uint32(0xFFFFE000)).view(F32)


def contraction(x, W, mode):
    """x [E, K] . W[N, K]^T in float64 from float32 operands: 'exact', or an emulation of the tensor-core product
    ('3xtf32': hi.hi + hi.lo + lo.hi with hi = the leading 11 bits and lo = the TF32 truncation of the rest; '1xtf32':
    hi.hi only; 'no_hi_lo': without the hi(x).lo(W) product)."""
    x, W = np.asarray(x, F32), np.asarray(W, F32)
    if mode == "exact":
        return x.astype(F64) @ W.astype(F64).T
    xh, Wh = tf32(x), tf32(W)
    xl, Wl = tf32(x - xh), tf32(W - Wh)
    hh = xh.astype(F64) @ Wh.astype(F64).T
    if mode == "1xtf32":
        return hh
    lh = xl.astype(F64) @ Wh.astype(F64).T
    if mode == "no_hi_lo":
        return hh + lh
    return hh + xh.astype(F64) @ Wl.astype(F64).T + lh


def gather(state, idx):
    """X[a][e][i] = state[e][idx[a][i]] (0 where idx < 0), float32."""
    X = np.where(idx[:, None, :] >= 0, state[:, np.maximum(idx, 0)].transpose(1, 0, 2), F32(0))
    return X.astype(F32)


def heads_reference(P, X, actor_in, hidden, nout, paths=("tcgen05",), mode="exact"):
    """Per agent: mu and the raw log-std, float64 [A, E, nout], and per GEMM path the bounds (of mu, of the raw log-std).
    mode 'exact' is the reference; the emulation modes round every layer to float32 as the kernel's epilogue does."""
    A, E = X.shape[0], X.shape[1]
    mu, ls = np.empty((A, E, nout)), np.empty((A, E, nout))
    bounds = {path: (np.empty((A, E, nout)), np.empty((A, E, nout))) for path in paths}
    for a in range(A):
        x = X[a]
        W1, W2, WH = (P[k][a][:, :n] for k, n in (("ACTOR_W1", actor_in), ("ACTOR_W2", hidden), ("ACTOR_WH", hidden)))
        b1, b2, bh = (P[k][a].astype(F64) for k in ("ACTOR_B1", "ACTOR_B2", "ACTOR_BH"))
        if mode == "exact":
            h1 = np.maximum(contraction(x, W1, mode) + b1, 0)
            h2 = np.maximum(h1 @ W2.astype(F64).T + b2, 0)
            o = h2 @ WH.astype(F64).T + bh
            s1 = np.abs(x).astype(F64) @ np.abs(W1).astype(F64).T
            aW2, aWH = np.abs(W2).astype(F64), np.abs(WH).astype(F64)
            for path in paths:
                g1, g2 = gamma(path, actor_in), gamma(path, hidden)
                d1 = g1 * s1 + U * np.abs(b1)
                d2 = g2 * ((h1 + d1) @ aW2.T) + d1 @ aW2.T + U * np.abs(b2)
                d3 = g2 * ((h2 + d2) @ aWH.T) + d2 @ aWH.T + U * np.abs(bh)
                bounds[path][0][a], bounds[path][1][a] = d3[:, :nout], d3[:, nout:2 * nout]
        else:
            h1 = np.maximum((contraction(x, W1, mode) + b1).astype(F32), 0)
            h2 = np.maximum((contraction(h1, W2, mode) + b2).astype(F32), 0)
            o = (contraction(h2, WH, mode) + bh).astype(F32).astype(F64)
        mu[a], ls[a] = o[:, :nout], o[:, nout:2 * nout]
    return mu, ls, bounds


def noise(seeds, steps, A, nout):
    """eps [A, E, nout] of oracle.rng.actor_noise for environment seeds [E] at decision counters [E]."""
    k0, k1 = orng.seed_key(np.asarray(seeds, np.int64))
    nb = (nout + 3) // 4
    blk = np.arange(nb, dtype=np.uint32)[None, :]
    out = np.empty((A, len(seeds), nout), F32)
    for a in range(A):
        z = orng.normals4(blk, np.asarray(steps, np.uint32)[:, None], np.uint32(orng.TAG_ACTOR), np.uint32(a),
                          k0[:, None], k1[:, None])
        out[a] = np.stack(z, axis=2).reshape(len(seeds), -1)[:, :nout]
    return out


def sech2(x):
    return 1.0 / np.cosh(np.minimum(np.abs(x), 350.0)) ** 2


def actions_reference(mu, ls_raw, dmu, dls, eps, log_sig_max, scale, bias):
    """(sampled action, its bound, mean action, its bound), float64 [A, E, nout]."""
    ls = np.clip(ls_raw, LOG_SIG_MIN, log_sig_max)
    sig = np.exp(ls)
    e = np.abs(eps).astype(F64)
    x = mu + sig * eps
    # GPU's sigma is within exp(ls + dls) (the clamp is 1-Lipschitz), expf within 2 ulp, one product, one sum
    sig_hi = np.exp(np.minimum(ls + dls, log_sig_max))
    dx = dmu + e * sig_hi * (np.expm1(dls) + 4 * U) + (np.abs(x) + e * sig_hi + np.abs(mu)) * 2 * U
    y = np.tanh(x)
    # tanh moves by at most the largest sech^2 over [x - dx, x + dx]; tanhf within 2 ulp; scale, bias rounded twice
    dy = sech2(np.maximum(np.abs(x) - dx, 0)) * dx + (np.abs(y) + U) * 4 * U
    act = y * scale + bias
    dact = abs(scale) * dy + (np.abs(act) + abs(bias)) * 2 * U
    ym = np.tanh(mu)
    dym = sech2(np.maximum(np.abs(mu) - dmu, 0)) * dmu + (np.abs(ym) + U) * 4 * U
    mean = ym * scale + bias
    dmean = abs(scale) * dym + (np.abs(mean) + abs(bias)) * 2 * U
    return act, dact, mean, dmean


def scatter(v, act_slot, E, action_dim):
    """[A, E, nout] -> [E, action_dim] through agent_act (NaN where no agent writes), and the mask of written slots."""
    out = np.full((E, action_dim), np.nan)
    A, nout = act_slot.shape
    for a in range(A):
        ok = act_slot[a] >= 0
        out[:, act_slot[a][ok]] = v[a][:, ok]
    return out, ~np.isnan(out[0])


def owner(rl, slot):
    a, j = np.argwhere(rl.agent_act == slot)[0]
    return int(a), int(j)


def check_bound(got, ref, bound, mask, rl, what, case):
    """Every mapped element inside its bound; the worst one is reported with its coordinates."""
    g, r, b = got[:, mask].astype(F64), ref[:, mask], bound[:, mask]
    assert np.isfinite(g).all(), "%s: non-finite actions" % what
    ratio = np.abs(g - r) / b
    e, i = np.unravel_index(int(np.argmax(ratio)), ratio.shape)
    slot = int(np.flatnonzero(mask)[i])
    a, j = owner(rl, slot)
    worst = float(ratio[e, i])
    record(case, what, worst)
    assert worst <= 1.0, ("%s: worst element E=%d env %d agent %d output %d: value %.9g reference %.9g bound %.3g "
                          "(error / bound %.3g)" % (what, got.shape[0], e, a, j, g[e, i], r[e, i], b[e, i], worst))
    return worst


# ----------------------------------------------------------------------------------------------------------------------
# CPU: the bound is tight enough to see a wrong split

SENS_CASES = [("10x10", 256, 300), ("10x10", 64, 129), ("40x40_43", 200, 130)]


@pytest.mark.parametrize("name,hidden,E", SENS_CASES)
def test_bound_separates_a_wrong_split(name, hidden, E):
    """On the data of the GPU tests, a numpy emulation of the kernel's 3xTF32 product stays inside the bound, while a
    single TF32 pass and the split without the hi.lo product exceed it by 10x or more: the GPU tests would fail on a
    subtly wrong split."""
    from ao_marl_b200.rl.policy import pack_actors
    rl = make_layout(name, hidden, seed=11)
    P = pack_actors(rl.policies, rl.actor_in, rl.hidden, rl.actor_out)
    X = gather(make_state(E, rl.state_dim, 5), rl.agent_idx)
    nout = rl.actor_out
    seeds = np.arange(E, dtype=np.int64) + 100
    eps = noise(seeds, np.full(E, 3), rl.n_agents, nout)
    sc, bi, lmax = float(rl.sac["gaussian_std"]), float(rl.sac["gaussian_mu"]), float(rl.sac["LOG_SIG_MAX"])
    mu, ls, bounds = heads_reference(P, X, rl.actor_in, rl.hidden, nout)
    dmu, dls = bounds["tcgen05"]
    act, dact, mean, dmean = actions_reference(mu, ls, dmu, dls, eps, lmax, sc, bi)
    used = rl.agent_act >= 0
    ratios = {}
    for mode in ("3xtf32", "1xtf32", "no_hi_lo"):
        m2, l2, _ = heads_reference(P, X, rl.actor_in, rl.hidden, nout, (), mode)
        a2, _, e2, _ = actions_reference(m2, l2, dmu, dls, eps, lmax, sc, bi)
        ratios[mode] = max(float((np.abs(a2 - act) / dact).transpose(0, 2, 1)[used].max()),
                           float((np.abs(e2 - mean) / dmean).transpose(0, 2, 1)[used].max()))
    record("sensitivity[%s-H%d-E%d]" % (name, hidden, E), "emulation_error_over_bound", ratios["3xtf32"])
    REPORT["sensitivity[%s-H%d-E%d]" % (name, hidden, E)].update(
        {"1xtf32_error_over_bound": ratios["1xtf32"], "no_hi_lo_error_over_bound": ratios["no_hi_lo"]})
    assert ratios["3xtf32"] <= 1.0, ratios
    assert ratios["1xtf32"] >= 10.0, ratios
    assert ratios["no_hi_lo"] >= 10.0, ratios


# ----------------------------------------------------------------------------------------------------------------------
# GPU: aom_actor_forward against the reference

@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


@pytest.fixture(scope="module")
def static40():
    from ao_marl_b200 import tables
    from ao_marl_b200.config import load_config_from_file
    t = tables.build_static(load_config_from_file(PAR40))
    tables.build_basis(t)
    return t


class Case:
    """One context (Simulator without atmosphere) of a layout, hidden size and batch, its state rows written directly,
    and the float64 reference of its current weights and state."""

    def __init__(self, t, name, hidden, E, seed, torch):
        from ao_marl_b200.lib import Simulator
        self.name, self.E, self.torch = name, E, torch
        self.key = "%s-H%d-E%d" % (name, hidden, E)
        self.rl = rl = make_layout(name, hidden, seed)
        self.sim = Simulator(t, E, rl, atmosphere=False)
        self.seeds = np.arange(E, dtype=np.int64) * 3 + 1000 + seed
        self.sim.reset(self.seeds)
        self.steps = np.zeros(E, np.int64)            # each environment's decision counter
        self.state = make_state(E, rl.state_dim, seed + 1)
        self.write_state()
        self.refresh()

    def write_state(self):
        self.sim.rows("STATE", self.rl.state_dim).copy_(self.torch.as_tensor(self.state, device="cuda"))

    def refresh(self):
        """Reference of the weights in force (pack_actors of the layout's policies) on the state rows read back."""
        from ao_marl_b200.rl.policy import pack_actors
        rl = self.rl
        self.P = pack_actors(rl.policies, rl.actor_in, rl.hidden, rl.actor_out)
        st = self.sim.rows("STATE", rl.state_dim).cpu().numpy()
        assert np.array_equal(st, self.state)
        self.mu, self.ls, self.bounds = heads_reference(self.P, gather(st, rl.agent_idx), rl.actor_in, rl.hidden,
                                                        rl.actor_out, ("tcgen05", "simt"))

    def close(self):
        self.sim.close()

    def action_buffers(self):
        E, sim = self.E, self.sim
        return (sim.buffer("ACTION").view(E, -1).cpu().numpy(), sim.buffer("ACTION_MEAN").view(E, -1).cpu().numpy())

    def forward(self, path, eval_mode):
        """One aom_actor_forward on `path` from sentinel-filled action buffers; returns (ACTION, ACTION_MEAN, sentinels)
        as whole rows (pad columns included) and the counters the call used."""
        torch, sim = self.torch, self.sim
        g = torch.Generator(device="cuda").manual_seed(int(self.steps.sum()) + 7)
        for name in ("ACTION", "ACTION_MEAN"):
            b = sim.buffer(name)
            b.copy_(torch.rand(b.shape, device="cuda", generator=g) + 100.0)
        before = self.action_buffers()
        try:
            sim.set_gemm_path(path)
            sim.actor_forward(eval_mode=eval_mode)
        finally:
            sim.set_gemm_path("tcgen05")
        sim.check_device()
        return self.action_buffers(), before

    def check(self, path, eval_mode, steps=None, what=""):
        """One call: every mapped action inside its bound, ACTION == ACTION_MEAN in eval mode, every entry no agent
        maps (the unmapped slot, the pad columns) unchanged.  Counters advance as actor_sample_kernel documents."""
        rl, E = self.rl, self.E
        steps = self.steps.copy() if steps is None else steps
        (act_g, mean_g), (act_0, mean_0) = self.forward(path, eval_mode)
        eps = noise(self.seeds, steps, rl.n_agents, rl.actor_out)
        dmu, dls = self.bounds[path]
        sc, bi, lmax = float(self.sim.cfg.pol_act_scale), float(self.sim.cfg.pol_act_bias), float(self.sim.cfg.log_sig_max)
        act, dact, mean, dmean = actions_reference(self.mu, self.ls, dmu, dls, eps, lmax, sc, bi)
        A_ref, mask = scatter(act, rl.agent_act, E, rl.action_dim)
        dA, _ = scatter(dact, rl.agent_act, E, rl.action_dim)
        M_ref, _ = scatter(mean, rl.agent_act, E, rl.action_dim)
        dM, _ = scatter(dmean, rl.agent_act, E, rl.action_dim)
        n = rl.action_dim
        case = "%s[%s]" % (self.key, path)
        check_bound(mean_g[:, :n], M_ref, dM, mask, rl, "mean " + what, case)
        if eval_mode:
            assert np.array_equal(act_g[:, :n][:, mask], mean_g[:, :n][:, mask]), "eval mode: ACTION != ACTION_MEAN"
        else:
            check_bound(act_g[:, :n], A_ref, dA, mask, rl, "sampled " + what, case)
        keep = np.concatenate([~mask, np.ones(act_g.shape[1] - n, bool)])
        assert keep.sum() >= 1
        assert np.array_equal(act_g[:, keep], act_0[:, keep]), "%s: unmapped ACTION entries changed" % what
        assert np.array_equal(mean_g[:, keep], mean_0[:, keep]), "%s: unmapped ACTION_MEAN entries changed" % what
        return act_g, mean_g

    def run_modes(self, paths=("tcgen05", "simt"), what=""):
        """Per path: eval mode, then two sampled calls (the counter advances between them)."""
        for path in paths:
            for eval_mode in (True, False, False):
                self.check(path, eval_mode, what=what + ("eval" if eval_mode else "sampled"))
                self.steps += 1                                      # every call is one decision (lockstep batch)


@pytest.fixture(scope="module")
def case43(static40, torch):
    """The headline layout at E = 4096 (43 agents, 280 inputs, 256 hidden, 60 head columns): shared by the shape,
    reproducibility and reward tests."""
    c = Case(static40, "40x40_43", 256, 4096, 43, torch)
    yield c
    c.close()


SHAPES = [("10x10", 256, 4096), ("10x10", 256, 4097), ("10x10", 256, 1), ("10x10", 256, 128), ("10x10", 200, 129),
          ("10x10", 64, 127), ("40x40_43", 256, 300), ("40x40_43", 200, 129), ("40x40_43", 64, 1),
          ("40x40_14tt", 256, 4096), ("40x40_14tt", 256, 129), ("40x40_14tt", 200, 300), ("40x40_14tt", 64, 127)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,hidden,E", SHAPES)
def test_actor_forward_inside_bound(static10, static40, torch, name, hidden, E):
    """Eval mode and two sampled calls on both GEMM paths: every action inside its bound of the float64 reference,
    unmapped entries unchanged."""
    t0 = time.time()
    c = Case(static10 if name == "10x10" else static40, name, hidden, E, E + hidden, torch)
    try:
        c.run_modes()
    finally:
        c.close()
        TIMES["shape[%s]" % c.key] = round(time.time() - t0, 1)


@pytest.mark.gpu
def test_actor_forward_headline_E4096(case43):
    t0 = time.time()
    case43.run_modes()
    TIMES["shape[%s]" % case43.key] = round(time.time() - t0, 1)


@pytest.mark.gpu
def test_actor_forward_reproducible(case43):
    """Two identical eval-mode calls give bit-identical actions (one repetition: a race shows as a difference)."""
    (a1, m1), _ = case43.forward("tcgen05", True)
    (a2, m2), _ = case43.forward("tcgen05", True)
    case43.steps += 2
    assert np.array_equal(a1.view(np.uint32), a2.view(np.uint32))
    assert np.array_equal(m1.view(np.uint32), m2.view(np.uint32))


@pytest.mark.gpu
@pytest.mark.parametrize("name,hidden,E", [("10x10", 200, 300), ("40x40_14tt", 256, 129)])
def test_reupload_rebuilds_pretiled_weights(static10, static40, torch, name, hidden, E):
    """Weights A, forward, then weights B of the same shapes uploaded into the same context: both paths match
    reference B (the pre-tiled hi / lo planes were rebuilt, not kept from A)."""
    t0 = time.time()
    c = Case(static10 if name == "10x10" else static40, name, hidden, E, 5, torch)
    try:
        c.run_modes(what="A ")
        mu_a = c.mu.copy()
        other_weights(c.rl, 99)
        c.rl.upload_actors(c.sim)
        c.refresh()
        assert np.abs(c.mu - mu_a).max() > 0.1                    # B really differs from A
        c.run_modes(what="B ")
    finally:
        c.close()
        TIMES["reupload[%s]" % c.key] = round(time.time() - t0, 1)


@pytest.mark.gpu
def test_staggered_counters(static10, torch):
    """reset_envs on a subset with new seeds: every environment samples with its own key and counter.  A restarted
    environment's pending first step uses counter 0 and does not advance it; after state_end it counts from 0 while
    the others continue from the batch's count."""
    c = Case(static10, "10x10", 256, 300, 17, torch)
    try:
        c.run_modes(paths=("tcgen05",))                             # three lockstep decisions: counters at 3
        envs = np.array([0, 127, 128, 299], np.int64)
        new = np.array([77, 78, 79, 80], np.int64)
        c.sim.reset_envs(envs, new)
        c.seeds[envs] = new
        c.steps[envs] = 0
        c.write_state()                                             # reset_envs cleared those rows
        c.refresh()
        others = np.setdiff1d(np.arange(c.E), envs)
        # first step pending: the restarted environments draw with counter 0 and keep it
        c.check("tcgen05", False, what="first pending ")
        c.steps[others] += 1
        c.check("simt", False, what="first pending again ")
        c.steps[others] += 1
        c.sim.state_end()                                           # the linear half-step ends the first step
        c.write_state()
        c.refresh()
        for path in ("tcgen05", "simt"):
            c.check(path, False, what="staggered ")
            c.steps += 1
        assert c.steps[envs[0]] == 2 and c.steps[others[0]] == 7
    finally:
        c.close()


@pytest.mark.gpu
def test_reward_against_float64(case43, torch):
    """aom_reward: every (environment, agent) against float64 -factor mean(res^2) over the agent's mode range, to
    2 (n + 32) 2^-24 relative."""
    sim, rl, E = case43.sim, case43.rl, case43.E
    nm = int(sim.cfg.nmodes)
    r = np.random.default_rng(8)
    res = (r.standard_normal((E, nm)) * np.exp(r.uniform(-4, 4, (E, 1)))).astype(F32)
    res[1] = 0
    sim.rows("RES_MODES", nm).copy_(torch.as_tensor(res, device="cuda"))
    factor = 1000.0
    sim.reward(factor)
    got = sim.buffer("REWARD").view(E, rl.n_agents).cpu().numpy().astype(F64)
    sim.check_device()
    worst = 0.0
    for a, (a0, a1) in enumerate(rl.agent_reward):
        n = a1 - a0
        ref = -factor * (res[:, a0:a1].astype(F64) ** 2).mean(axis=1)
        tol = 2 * (n + 32) * U * np.abs(ref)
        ratio = np.abs(got[:, a] - ref) / np.where(tol > 0, tol, 1.0)
        assert np.array_equal(got[ref == 0, a], ref[ref == 0]), a
        e = int(np.argmax(ratio))
        worst = max(worst, float(ratio[e]))
        assert ratio[e] <= 1.0, ("agent %d env %d: reward %.9g reference %.9g tolerance %.3g"
                                 % (a, e, got[e, a], ref[e], tol[e]))
    record("reward[%s]" % case43.key, "error_over_tolerance", worst)
