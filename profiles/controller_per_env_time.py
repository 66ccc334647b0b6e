"""Cost of per-environment controllers on aom_step and on aom_actor_forward (43 agents, E = 4096).

Four cases on one context (production_sh_40x40_8m_3layers, mode 0), alternated block by block in one process:

  uniform      every environment on slot 0 (the uniform actor kernel)
  slots2       two policy slots interleaved 50/50 (environment e on slot e % 2)
  slots4       four policy slots interleaved (e % 4)
  half_integ   every other environment on the integrator, the others on slot 0

Every slot holds its own weights (different draws of the same shapes), so that two slots stream two sets of pre-split
planes (about 60 MB each at this size) through the L2.  Per block: CUDA events around `--steps` steps after `--warmup`
untimed ones, and around `--steps` aom_actor_forward calls alone.  Prints the card and its power limit, then one line
per block and a JSON summary.

    python profiles/controller_per_env_time.py [--envs 4096] [--steps 40] [--warmup 10] [--rounds 3] [--out FILE]
"""
import argparse
import copy
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

ENV_RL = dict(n_zernike_start_end=[0, 1260], window_n_zernike=20, include_tip_tilt_windowed=True,
              n_reverse_filtered_from_cmat=5, delayed_assignment=2)


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


def draw(rl, seed):
    """Policies of the layout's shapes with non-zero heads."""
    import torch
    g = torch.Generator().manual_seed(seed)
    pols = [copy.deepcopy(p) for p in rl.policies]
    with torch.no_grad():
        for p in pols:
            for w in p.parameters():
                w.copy_(torch.randn(tuple(w.shape), generator=g) * (0.05 if w.dim() > 1 else 0.1))
            p.log_std_linear.bias.fill_(-1.0)
    return pols


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON summary here")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the GPU and has no CPU fallback")
    from ao_marl_b200.system import build_system
    name, power = card()
    print("card: %s, power limit %s" % (name, power), flush=True)
    E = args.envs
    par = "production_sh_40x40_8m_3layers.py"
    sim, t, rl = build_system(par, E, env_rl=dict(ENV_RL, parameters_telescope=par), world_size=44, seed=0)
    for k in range(4):
        rl.upload_actors(sim, slot=k, policies=draw(rl, 300 + k))
    e = np.arange(E)
    cases = {"uniform": None, "slots2": e % 2, "slots4": e % 4, "half_integ": np.where(e % 2 == 1, -1, 0)}
    seeds = 1234 + np.arange(E, dtype=np.int64)
    rows = []

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / args.steps

    for rnd in range(args.rounds):
        for case, ctrl in cases.items():
            sim.set_controller_env(ctrl)
            sim.reset(seeds)
            sim.state_begin(); sim.move_atmos(); sim.comp_wfs_image(); sim.do_centroids(); sim.do_control(); sim.state_end()
            for _ in range(args.warmup):
                sim.step(mode=0)
            torch.cuda.synchronize()
            step_ms = timed(lambda: sim.step(mode=0))
            actor_ms = timed(lambda: sim.actor_forward())
            sim.check_device()
            b = dict(case=case, round=rnd, ms_per_step=step_ms, actor_forward_ms=actor_ms)
            rows.append(b)
            print("round %d %-10s %7.3f ms/step  aom_actor_forward %6.3f ms" % (rnd, case, step_ms, actor_ms), flush=True)
    sim.set_controller_env(None)
    sim.close()
    summary = dict(card=name, power_limit=power, agents=int(rl.n_agents), envs=E, steps=args.steps, warmup=args.warmup,
                   blocks=rows)
    for case in cases:
        s = sorted(b["ms_per_step"] for b in rows if b["case"] == case)
        a = sorted(b["actor_forward_ms"] for b in rows if b["case"] == case)
        summary[case] = dict(ms_per_step_median=s[len(s) // 2], ms_per_step_min=s[0], ms_per_step_max=s[-1],
                             actor_forward_ms_median=a[len(a) // 2], actor_forward_ms_min=a[0], actor_forward_ms_max=a[-1])
    line = json.dumps(summary)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
