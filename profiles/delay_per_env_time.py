"""Cost of the three-row delay line on aom_step (production_sh_40x40_8m_3layers, 43 agents, E = 4096).

Times aom_step (mode 0: actors, controller, turbulence, sensor frame, state) in four variants, alternated block by block
in one session:

  parent     a checkout of the parent commit (--parent DIR): the two-row line, delay 1 of the parameter file
  uniform_1  this tree, delay 1 of the parameter file (the default path)
  uniform_2  this tree, common delay 2 (aom_set_delay)
  per_env    this tree, one delay per environment cycling through 0, 0.5, 1, 1.5, 2 (aom_set_delay_env)

Each tree runs in a worker process of its own (the two libraries export the same symbols) that keeps its context for the
whole session; the main process hands the variants to the workers in turn, so no two blocks overlap on the GPU.  Per
block: CUDA events around `--steps` steps after `--warmup` untimed ones.  Prints the card and its power limit, then one
line per block and a JSON summary.  Without --parent the parent variant is skipped.

    python profiles/delay_per_env_time.py [--parent DIR] [--envs 4096] [--steps 40] [--warmup 10] [--rounds 3] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
PAR = "production_sh_40x40_8m_3layers.py"
ENV_RL = dict(parameters_telescope=PAR, n_zernike_start_end=[0, 1260], window_n_zernike=20,
              include_tip_tilt_windowed=True, n_reverse_filtered_from_cmat=5, delayed_assignment=2)
MIX = [0.0, 0.5, 1.0, 1.5, 2.0]


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


def worker(args):
    """One context of the tree at --root: reads a variant name per line, answers with one "@@ "-prefixed JSON line per
    block."""
    sys.path.insert(0, args.root)
    import torch
    from ao_marl_b200.system import build_system
    E = args.envs
    sim, t, rl = build_system(PAR, E, env_rl=ENV_RL, world_size=44, seed=0)
    seeds = 1234 + np.arange(E, dtype=np.int64)
    mix = np.array([MIX[e % len(MIX)] for e in range(E)], np.float32)
    print("@@ " + json.dumps(dict(ready=True, agents=int(rl.n_agents))), flush=True)
    for line in sys.stdin:
        variant = line.strip()
        if not variant:
            break
        if variant != "parent":
            sim.set_delay_env(mix if variant == "per_env" else None)
            sim.set_delay(2.0 if variant == "uniform_2" else 1.0)
        sim.reset(seeds)
        sim.state_begin(); sim.move_atmos(); sim.comp_wfs_image(); sim.do_centroids(); sim.do_control(); sim.state_end()
        for _ in range(args.warmup):
            sim.step(mode=0)
        torch.cuda.synchronize()
        l0 = sim.launches()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            sim.step(mode=0)
        e1.record()
        torch.cuda.synchronize()
        launches = (sim.launches() - l0) // args.steps
        sim.check_device()
        print("@@ " + json.dumps(dict(variant=variant, ms_per_step=e0.elapsed_time(e1) / args.steps,
                                      launches_per_step=launches)), flush=True)
    sim.close()


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--parent", default=None, help="checkout of the parent commit (built, importable)")
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON summary here")
    ap.add_argument("--worker", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--root", default=ROOT, help=argparse.SUPPRESS)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the GPU and has no CPU fallback")
    if args.worker:
        return worker(args)
    name, power = card()
    print("card: %s, power limit %s" % (name, power), flush=True)

    def reply(p):
        """The next protocol line of a worker (lines of its own output are passed through)."""
        while True:
            line = p.stdout.readline()
            if not line:
                raise RuntimeError("worker exited (rc %s)" % p.poll())
            if line.startswith("@@ "):
                return json.loads(line[3:])
            sys.stdout.write(line)

    def spawn(root):
        p = subprocess.Popen([sys.executable, os.path.abspath(__file__), "--worker", "--root", root, "--envs",
                              str(args.envs), "--steps", str(args.steps), "--warmup", str(args.warmup)],
                             stdin=subprocess.PIPE, stdout=subprocess.PIPE, text=True, cwd=root)
        head = reply(p)
        assert head.get("ready"), head
        return p, head

    def ask(p, variant):
        p.stdin.write(variant + "\n")
        p.stdin.flush()
        return reply(p)

    workers = {}
    if args.parent:
        workers["parent"] = spawn(os.path.abspath(args.parent))
    workers["this"] = spawn(ROOT)
    agents = workers["this"][1]["agents"]
    variants = (["parent"] if args.parent else []) + ["uniform_1", "uniform_2", "per_env"]
    rows = []
    try:
        for rnd in range(args.rounds):
            for v in variants:
                b = ask(workers["parent" if v == "parent" else "this"][0], v)
                b["round"] = rnd
                rows.append(b)
                print("round %d %-10s %7.3f ms/step  %d launches/step" % (rnd, v, b["ms_per_step"], b["launches_per_step"]),
                      flush=True)
    finally:
        for p, _ in workers.values():
            p.stdin.close()
            p.wait(timeout=300)
    summary = dict(card=name, power_limit=power, workload=PAR, agents=agents, envs=args.envs, steps=args.steps,
                   warmup=args.warmup, mix=MIX, blocks=rows)
    for v in variants:
        ms = [b["ms_per_step"] for b in rows if b["variant"] == v]
        summary[v] = dict(ms_per_step_median=float(np.median(ms)), ms_per_step_min=float(np.min(ms)),
                          ms_per_step_max=float(np.max(ms)))
    print(json.dumps(summary))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(summary, f, indent=1)


if __name__ == "__main__":
    main()
