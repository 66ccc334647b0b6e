"""C-ABI library: loads and exports every symbol declared in include/aomarl.h (no compute calls -- no GPU
here); host-side RL logic against the reference's golden vectors; world_size-2 gloo sharding."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_header_symbol():
    from ao_marl_b200 import lib as binding
    loaded = binding.load_library()
    header = open(os.path.join(ROOT, "include", "aomarl.h")).read()
    declared = set(re.findall(r"\b(aom_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations found"
    for name in declared:
        assert hasattr(loaded, name), "libaomarl.so does not export %s" % name
    assert declared == set(binding.EXPORTS)
    assert loaded.aom_config_size() == __import__("ctypes").sizeof(binding.AomConfig)


def test_table_and_buffer_enums_match_header():
    from ao_marl_b200 import lib as binding
    header = open(os.path.join(ROOT, "include", "aomarl.h")).read()
    tabs = re.findall(r"^\s*AOM_T_([A-Z0-9_]+)", header, flags=re.M)
    bufs = re.findall(r"^\s*AOM_B_([A-Z0-9_]+)", header, flags=re.M)
    assert [t for t in tabs if t != "COUNT"] == binding.TABLES
    assert [b for b in bufs if b != "COUNT"] == binding.BUFFERS
    opts = re.findall(r"^\s*AOM_OPT_([A-Z0-9_]+)", header, flags=re.M)
    assert [o for o in opts if o != "COUNT"] == binding.OPTIONS
    conds = re.findall(r"^\s*AOM_COND_([A-Z0-9_]+)", header, flags=re.M)
    assert [c for c in conds if c != "COUNT"] == binding.CONDITIONS


def test_no_cpu_path():
    import torch
    if torch.cuda.is_available():
        pytest.skip("only meaningful on a machine without a GPU")
    from ao_marl_b200.lib import Simulator
    with pytest.raises(RuntimeError):
        Simulator(None, 1)


def test_product_does_not_import_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "ao_marl_b200")):
        for f in files:
            if f.endswith(".py"):
                txt = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M), f


def test_state_split_tables(golden_rl):
    from ao_marl_b200.rl import helper_states as hs
    keys = ["dm_history_2", "dm_history_1", "dm_before_linear", "dm_residual"]

    def run(tag, total, start, end, nag, window, ttw, nf):
        d, ctrl, per = hs.agents_dictionary(total, start, end, nag + 2, True)
        ios, i0 = {}, 0
        for k in keys:
            ios[k] = [i0, i0 + (total if window > -1 else end - start + 2)]
            i0 = ios[k][1]
        env = dict(window_n_zernike=window, include_tip_tilt=True, include_tip_tilt_windowed=ttw)
        mc = hs.get_modes_chosen(d, ios, env, nf, total, ctrl, start)
        for w in mc:
            assert np.array_equal(mc[w], golden_rl["rl.%s.modes_chosen_%d" % (tag, w)])
        return mc

    assert len(run("10x10", 87, 0, 80, 1, -1, False, 5)) == 2
    assert len(run("40x40w20", 1283, 0, 1260, 42, 20, False, 5)) == 43
    assert len(run("40x40_14w20tt", 1283, 0, 1260, 14, 20, True, 5)) == 15


def test_delayed_mdp_slot_order(golden_rl):
    from ao_marl_b200.rl.delayed_mdp import DelayedMDP
    for delay, modif in ((1, False), (2, False), (0, False), (1, True)):
        m = DelayedMDP(delay, modif)
        rec = []
        for t in range(8):
            if m.check_update_possibility():
                rec.append((t,) + m.credit_assignment())
            m.save(100 + t, 200 + t, 300 + t)
        ref = golden_rl["rl.delayed_mdp_d%d_m%d" % (delay, int(modif))]
        assert np.array_equal(np.array(rec, dtype=np.int64).reshape(ref.shape), ref)


def test_policy_forward_matches_reference(golden_rl):
    import torch
    from ao_marl_b200.rl.policy import GaussianPolicy, pack_actors
    pol = GaussianPolicy(24, 6, hidden_dim=32, initialize_last_layer_zero=False)
    pol.load_state_dict({k[len("rl.policy."):]: torch.tensor(golden_rl[k]) for k in golden_rl.files
                         if k.startswith("rl.policy.") and k.split(".")[-1] in ("weight", "bias")})
    with torch.no_grad():
        m, l = pol.forward(torch.tensor(golden_rl["rl.policy.x"]))
    assert np.array_equal(m.numpy(), golden_rl["rl.policy.mean"])
    assert np.array_equal(l.numpy(), golden_rl["rl.policy.log_std"])
    packed = pack_actors([pol], 30, 32, 8)
    assert packed["ACTOR_W1"].shape == (1, 32, 32) and packed["ACTOR_WH"].shape == (1, 16, 32)
    assert np.array_equal(packed["ACTOR_WH"][0, 8:14, :32], golden_rl["rl.policy.log_std_linear.weight"])


def test_rl_layout_10x10():
    from ao_marl_b200.rl.layout import RLLayout
    rl = RLLayout(87, dict(parameters_telescope="production_sh_10x10_2m.py", n_zernike_start_end=[0, 80],
                           n_reverse_filtered_from_cmat=5), None, world_size=3)
    assert rl.action_dim == 82 and rl.state_dim == 328 and rl.n_agents == 2
    assert list(rl.action_map[-2:]) == [85, 86] and rl.actor_in == 320 and rl.actor_out == 80
    assert list(rl.agent_act[1, :3]) == [80, 81, -1] and list(rl.agent_reward[1]) == [85, 87]
    assert np.allclose(rl.freedom * 10, np.load(os.path.join(os.path.dirname(__file__), "..", "ao_marl_b200", "data",
                                                             "normalization", "production_sh_10x10_2m.npz"))["zn_norm"])


def test_env_sharding_gloo_world2(tmp_path):
    """N>1 path on CPU: two gloo ranks shard 10 environments, seeds are disjoint and the max-over-ranks
    timing reduction works (the step itself needs no collective)."""
    script = tmp_path / "w.py"
    script.write_text(
        "import os, sys, torch, torch.distributed as dist\n"
        "sys.path.insert(0, %r)\n"
        "from ao_marl_b200.parallel import shard_envs, reduce_max\n"
        "dist.init_process_group('gloo')\n"
        "r, w = dist.get_rank(), dist.get_world_size()\n"
        "lo, hi, seeds = shard_envs(10, r, w, base_seed=1234)\n"
        "allseeds = [None] * w\n"
        "dist.all_gather_object(allseeds, seeds.tolist())\n"
        "flat = sum(allseeds, [])\n"
        "assert sorted(flat) == list(range(1234, 1244)), flat\n"
        "t = reduce_max(float(r + 1), dist)\n"
        "assert t == float(w)\n"
        "dist.destroy_process_group()\n" % ROOT)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29533")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29533", str(script)], env=env,
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr


def test_rl_layout_40x40_agent_counts():
    """SURVEY note N1: the benchmarked layout is 43 agents (42 x 30 modes + tip-tilt, window 20 -> 280 / 168 inputs);
    the literal reading of the config name is 14 x 90 modes + tip-tilt (520 / 168 inputs).  Both are parameters of the
    same tables."""
    from ao_marl_b200.rl.layout import RLLayout
    env = dict(parameters_telescope="production_sh_40x40_8m_3layers.py", n_zernike_start_end=[0, 1260],
               window_n_zernike=20, include_tip_tilt_windowed=True, n_reverse_filtered_from_cmat=5)
    rl = RLLayout(1283, env, None, world_size=44)
    assert rl.n_agents == 43 and rl.action_dim == 1262 and rl.state_modes == 1283
    assert rl.actor_in == 280 and rl.actor_out == 30
    widths = (rl.agent_idx >= 0).sum(axis=1)
    assert sorted(set(widths.tolist())) == [168, 280] or int(widths.max()) == 280
    assert int((rl.agent_act >= 0).sum()) == rl.action_dim                       # every action slot owned once
    assert sorted(rl.agent_act[rl.agent_act >= 0].tolist()) == list(range(rl.action_dim))
    rl14 = RLLayout(1283, env, None, world_size=16)                             # 14 mode agents + tip-tilt + the trainer rank
    assert rl14.n_agents == 15 and rl14.actor_out == 90
    assert int((rl14.agent_idx >= 0).sum(axis=1).max()) == 520
    assert sorted(rl14.agent_act[rl14.agent_act >= 0].tolist()) == list(range(rl14.action_dim))
