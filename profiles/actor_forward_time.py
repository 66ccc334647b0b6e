"""Device time of aom_actor_forward alone on the headline layout (43 agents, 280 inputs, 256 hidden units, 60 head
columns, E = 4096), for one or more builds of the library, alternated round by round.

Each --tree is a checkout whose libaomarl.so is built.  Per round and tree a worker process builds the 40x40 tables and
layout, a context without atmosphere, random state rows (standard normals), then times `--calls` sampled-mode calls of
aom_actor_forward with CUDA events after `--warmup` untimed ones.  Prints the card and its power limit, one line per
round and tree, and a JSON summary with the median time per call and its floors:

  flop        useful 3xTF32 work: 3 x 2 x E x A x (AOM_LD(in) x H + H x H + H x heads), over the data-sheet TF32 rate
              (1,125 TFLOP/s dense, B200 at 1000 W)
  hbm bytes   each weight and state byte once (pre-split weight planes, state rows, actions), over 7.7 TB/s
  l2 stream   the pre-split weight bytes each 128-environment tile copies into shared memory (not a floor: no L2 rate
              is measured on this card; given as bytes and as the rate the measured time implies)

    python profiles/actor_forward_time.py [--tree LABEL=DIR ...] [--envs 4096] [--calls 200] [--warmup 20] [--rounds 3] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
PAR = "production_sh_40x40_8m_3layers.py"
ENV_RL = dict(n_zernike_start_end=[0, 1260], window_n_zernike=20, include_tip_tilt_windowed=True,
              n_reverse_filtered_from_cmat=5, delayed_assignment=2)
TF32_FLOPS = 1125e12
HBM_BPS = 7.7e12


def ld(n):
    return (int(n) + 15) & ~15


def worker(args):
    import numpy as np
    import torch
    from ao_marl_b200 import tables
    from ao_marl_b200.config import load_config_from_file
    from ao_marl_b200.lib import Simulator
    from ao_marl_b200.rl.layout import RLLayout, load_normalization
    E = args.envs
    t = tables.build_static(load_config_from_file(PAR))
    tables.build_basis(t)
    nm = len(load_normalization(PAR)[1])
    rl = RLLayout(nm, dict(ENV_RL, parameters_telescope=PAR), None, world_size=44, seed=1)
    sim = Simulator(t, E, rl, atmosphere=False)
    sim.reset(np.arange(E, dtype=np.int64) + 1234)
    g = torch.Generator(device="cuda").manual_seed(5)
    st = sim.rows("STATE", rl.state_dim)
    st.copy_(torch.randn(st.shape, device="cuda", generator=g))
    for _ in range(args.warmup):
        sim.actor_forward(eval_mode=False)
    torch.cuda.synchronize()
    l0 = sim.launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.calls):
        sim.actor_forward(eval_mode=False)
    e1.record()
    torch.cuda.synchronize()
    sim.check_device()
    ms = e0.elapsed_time(e1) / args.calls
    launches = (sim.launches() - l0) / args.calls
    A, K, H, heads = rl.n_agents, rl.actor_in, rl.hidden, 2 * rl.actor_out
    flop = 3 * 2 * E * A * (ld(K) * H + H * H + H * heads)
    # pre-split planes per agent: [128-column tiles][k blocks][hi, lo][128 x 16] floats
    planes = [-(-ld(H) // 128) * ld(K) * 2 * 128, -(-ld(H) // 128) * ld(H) * 2 * 128, -(-ld(heads) // 128) * ld(H) * 2 * 128]
    weight_bytes = 4 * A * sum(planes)
    hbm = weight_bytes + 4 * E * ld(rl.state_dim) + 2 * 4 * E * ld(rl.action_dim)
    tiles = -(-E // 128) * A
    l2 = 4 * tiles * (planes[0] + planes[1] + ld(heads) * ld(H) * 2)    # the heads copy only their rows
    sim.close()
    return {"ms_per_call": ms, "launches_per_call": launches, "E": E, "agents": A, "actor_in": K,
            "hidden": H, "heads": heads, "gflop": flop / 1e9, "tflops": flop / (ms * 1e-3) / 1e12,
            "flop_floor_ms": flop / TF32_FLOPS * 1e3, "hbm_bytes": hbm, "hbm_floor_ms": hbm / HBM_BPS * 1e3,
            "l2_weight_stream_bytes": l2, "l2_weight_stream_tbps": l2 / (ms * 1e-3) / 1e12}


def card():
    import torch
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        power = q.stdout.strip() or "unknown"
    except Exception as exc:  # the query is informative only
        power = "unknown (%s)" % exc
    return name, power


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--tree", action="append", default=None, metavar="LABEL=DIR",
                    help="checkout with a built library, and its label in the output (default: this one as 'tree')")
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON summary here")
    ap.add_argument("--worker", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the GPU and has no CPU fallback")
    if args.worker:
        print(json.dumps(worker(args)))
        return
    trees = dict(t.split("=", 1) if "=" in t else (os.path.basename(os.path.abspath(t)), t)
                 for t in (args.tree or ["tree=" + os.path.join(HERE, "..")]))
    name, power = card()
    print("card: %s, power limit %s" % (name, power), flush=True)
    runs = {label: [] for label in trees}
    for rnd in range(args.rounds):
        for label, tree in trees.items():
            tree = os.path.abspath(tree)
            cmd = [sys.executable, os.path.abspath(__file__), "--worker", "--envs", str(args.envs), "--calls",
                   str(args.calls), "--warmup", str(args.warmup)]
            env = dict(os.environ, PYTHONPATH=tree)
            r = subprocess.run(cmd, cwd=tree, env=env, capture_output=True, text=True)
            if r.returncode != 0:
                raise SystemExit("worker on %s failed:\n%s%s" % (label, r.stdout, r.stderr))
            res = json.loads(r.stdout.strip().splitlines()[-1])
            runs[label].append(res)
            print("round %d %s: %.4f ms per call, %.1f TFLOP/s, %.0f launches per call" %
                  (rnd, label, res["ms_per_call"], res["tflops"], res["launches_per_call"]), flush=True)
    summary = {"card": name, "power_limit": power, "envs": args.envs, "calls": args.calls, "rounds": args.rounds, "trees": {}}
    for label, rs in runs.items():
        ms = [r["ms_per_call"] for r in rs]
        s = dict(rs[0])
        s.update({"ms_per_call": statistics.median(ms), "ms_min": min(ms), "ms_max": max(ms),
                  "tflops": s["gflop"] * 1e9 / (statistics.median(ms) * 1e-3) / 1e12,
                  "l2_weight_stream_tbps": s["l2_weight_stream_bytes"] / (statistics.median(ms) * 1e-3) / 1e12})
        s["floor_ms"] = max(s["flop_floor_ms"], s["hbm_floor_ms"])
        s["bound"] = "tf32 rate" if s["flop_floor_ms"] >= s["hbm_floor_ms"] else "hbm"
        s["floor_over_time"] = s["floor_ms"] / s["ms_per_call"]
        summary["trees"][label] = s
    print(json.dumps(summary, indent=1))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(summary, f, indent=1)


if __name__ == "__main__":
    main()
