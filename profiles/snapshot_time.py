"""Cost of per-environment snapshots on the default workload (production_sh_40x40_8m_3layers, 43 agents, E = 4096).

aom_save_envs and aom_load_envs of K environments next to aom_reset_envs of the same K, for K = 1 .. 4096: host clock
around the call and a device synchronise (each call waits for the stream first), `--reps` repetitions each, alternating.
The records are loaded back into other slots of the same running batch (a copy).  Derived figures: bytes per
environment, and the achieved bandwidth of save and load (each environment's record read once and written once) against
the 7.7 TB/s of the B200's HBM3e.  Prints the card and its power limit, one line per measurement and a JSON summary.

    python profiles/snapshot_time.py [--envs 4096] [--ks 1,8,64,512,4096] [--reps 3] [--out FILE]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

from wind_per_env_time import ENV_RL, PAR, card  # noqa: E402  (same workload, same card query)

HBM_TBS = 7.7


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--ks", default="1,8,64,512,4096")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON summary here")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the GPU and has no CPU fallback")
    from ao_marl_b200.system import build_system
    name, power = card()
    print("card: %s, power limit %s" % (name, power), flush=True)
    E = args.envs
    sim, t, rl = build_system(PAR, E, env_rl=dict(ENV_RL), world_size=44, seed=0)
    seeds = 1234 + np.arange(E, dtype=np.int64)
    r = np.random.default_rng(11)
    sim.reset(seeds)
    for _ in range(3):
        sim.step(mode=0)
    nbytes = sim.env_state_bytes()
    print("record: %d bytes per environment" % nbytes, flush=True)

    def timed(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        return 1e3 * (time.perf_counter() - t0), out

    ks = [int(k) for k in args.ks.split(",") if int(k) <= E]
    for k in ks:                                     # untimed pass: every launch shape once
        envs = np.sort(r.choice(E, k, replace=False))
        sim.load_envs(r.permutation(envs), sim.save_envs(envs))
        sim.reset_envs(envs, 5000 + np.arange(k))
    res = {k: dict(save=[], load=[], reset_envs=[]) for k in ks}
    for rep in range(args.reps):
        for k in ks:
            envs = np.sort(r.choice(E, k, replace=False)).astype(np.int32)
            ms, snap = timed(lambda: sim.save_envs(envs))
            res[k]["save"].append(ms)
            ms, _ = timed(lambda: sim.load_envs(r.permutation(envs), snap))
            res[k]["load"].append(ms)
            del snap
            ms, _ = timed(lambda: sim.reset_envs(envs, 9000 + np.arange(k)))
            res[k]["reset_envs"].append(ms)
            print("rep %d K=%-5d save %9.3f ms  load %9.3f ms  reset_envs %9.2f ms" % (
                rep, k, res[k]["save"][-1], res[k]["load"][-1], res[k]["reset_envs"][-1]), flush=True)
    sim.check_device()
    summary = dict(card=name, power_limit=power, config=PAR, agents=int(rl.n_agents), envs=E, reps=args.reps,
                   bytes_per_env=nbytes, hbm_tb_s=HBM_TBS, timing="host clock around the call and a device synchronise")
    rows = {}
    for k in ks:
        row = {}
        for what in ("save", "load", "reset_envs"):
            v = res[k][what]
            row[what + "_ms"] = dict(median=float(np.median(v)), all=v)
        moved = 2.0 * k * nbytes                     # every record byte read once and written once
        for what in ("save", "load"):
            gbs = moved / (row[what + "_ms"]["median"] * 1e-3) / 1e9
            row[what + "_gb_s"] = gbs
            row[what + "_share_of_hbm"] = gbs / (HBM_TBS * 1e3)
        rows[str(k)] = row
        print("K=%-5d save %9.3f ms (%7.1f GB/s)  load %9.3f ms (%7.1f GB/s)  reset_envs %9.2f ms" % (
            k, row["save_ms"]["median"], row["save_gb_s"], row["load_ms"]["median"], row["load_gb_s"],
            row["reset_envs_ms"]["median"]), flush=True)
    summary["k"] = rows
    print(json.dumps(summary))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(summary, f, indent=1)
    sim.close()


if __name__ == "__main__":
    main()
