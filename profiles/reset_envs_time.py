"""Cost of per-environment resets on the default workload (production_sh_40x40_8m_3layers, 43 agents, E = 4096).

(i)  aom_reset_envs for K restarted environments against aom_reset of the whole batch: host clock around the call and a
     device synchronise (the call itself waits for the stream first), `--reps` repetitions each, alternating.
(ii) aom_step of a lockstep batch against a staggered one (half the environments restarted mid-run, common winds: the
     library runs its per-environment wind path while the accumulators of the two halves differ), alternating the two
     over `--rounds` rounds on the same context.  Per block: CUDA events around `--steps` steps after `--warmup` untimed
     ones, the sensor kernel's own time (AOM_OPT_TIME_WFS) and the extrusion passes per step from the library's
     accumulator arithmetic (oracle.aoframe.OracleAtmos.move; per layer and axis the largest count of the batch).
Prints the card and its power limit, one line per measurement and a JSON summary.

    python profiles/reset_envs_time.py [--envs 4096] [--ks 1,8,64,512,2048,4096] [--reps 2] [--steps 40] [--warmup 10]
                                       [--rounds 3] [--out FILE]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

from wind_per_env_time import ENV_RL, PAR, card  # noqa: E402  (same workload, same card query)


def group_counts(d, frames):
    """Whole-pixel counts of `frames` frames from a zeroed accumulator with step d (float32): the host's arithmetic."""
    a, out = 0.0, []
    for _ in range(frames):
        a += float(np.float32(d))
        n = float(np.trunc(a))
        a -= n
        out.append(int(n))
    return out


def passes(cdx, cdy, frames, restart=None):
    """Extrusion passes per frame for `frames` frames after a reset; restart: frame index at which half the batch was
    restarted (its accumulators from zero again), None for a lockstep batch."""
    out = []
    for f in range(frames):
        n = 0
        for dx, dy in zip(cdx, cdy):
            for d in (dx, dy):
                c = abs(group_counts(d, f + 1)[f])
                if restart is not None and f >= restart:
                    c = max(c, abs(group_counts(d, f + 1 - restart)[f - restart]))
                n += c
        out.append(n)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--ks", default="1,8,64,512,2048,4096")
    ap.add_argument("--reps", type=int, default=2)
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
    sim, t, rl = build_system(PAR, E, env_rl=dict(ENV_RL), world_size=44, seed=0)
    L = int(sim.cfg.n_layers)
    cdx = [float(sim.cfg.deltax[l]) for l in range(L)]
    cdy = [float(sim.cfg.deltay[l]) for l in range(L)]
    seeds = 1234 + np.arange(E, dtype=np.int64)
    r = np.random.default_rng(7)

    def linear_step():
        sim.state_begin(); sim.move_atmos(); sim.comp_wfs_image(); sim.do_centroids(); sim.do_control(); sim.state_end()

    def timed(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        return 1e3 * (time.perf_counter() - t0)

    # (i) start-up cost
    sim.reset(seeds)
    linear_step()
    ks = [int(k) for k in args.ks.split(",") if int(k) <= E]
    for k in ks:                                     # untimed pass: every launch shape once
        sim.reset_envs(np.sort(r.choice(E, k, replace=False)), 5000 + np.arange(k))
    reset_ms, envs_ms = [], {k: [] for k in ks}
    for rep in range(args.reps):
        reset_ms.append(timed(lambda: sim.reset(seeds)))
        print("rep %d aom_reset            %9.2f ms" % (rep, reset_ms[-1]), flush=True)
        for k in ks:
            envs = np.sort(r.choice(E, k, replace=False)).astype(np.int32)
            envs_ms[k].append(timed(lambda: sim.reset_envs(envs, 9000 + np.arange(k))))
            print("rep %d aom_reset_envs K=%-5d %9.2f ms" % (rep, k, envs_ms[k][-1]), flush=True)
    sim.check_device()

    # (ii) step time, lockstep against staggered
    half = np.arange(0, E, 2, dtype=np.int32)
    restart = 1 + args.warmup // 2                   # frames after the reset at which half the batch restarts

    def block(staggered):
        sim.reset(seeds)
        linear_step()
        for i in range(args.warmup):
            if staggered and i == args.warmup // 2:
                sim.reset_envs(half, 7000 + half.astype(np.int64))
            sim.step(mode=0)
        torch.cuda.synchronize()
        sim.time_wfs(True)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            sim.step(mode=0)
        e1.record()
        torch.cuda.synchronize()
        wfs_ms, n_wfs = sim.wfs_time_ms()
        sim.time_wfs(False)
        sim.check_device()
        frames = 1 + args.warmup + args.steps
        pp = passes(cdx, cdy, frames, restart if staggered else None)[1 + args.warmup:]
        return dict(batch="staggered" if staggered else "lockstep", ms_per_step=e0.elapsed_time(e1) / args.steps,
                    extrusion_passes_per_step=float(np.mean(pp)), time_wfs_ms=wfs_ms, wfs_timed_launches=n_wfs,
                    wfs_kernel=sim.wfs_kernel())

    rows = []
    for rnd in range(args.rounds):
        for staggered in (False, True):
            b = block(staggered)
            b["round"] = rnd
            rows.append(b)
            print("round %d %-9s  %7.3f ms/step  %5.2f extrusion passes/step  sensor kernel %6.3f ms (%s)" % (
                rnd, b["batch"], b["ms_per_step"], b["extrusion_passes_per_step"], b["time_wfs_ms"], b["wfs_kernel"]),
                flush=True)
    summary = dict(card=name, power_limit=power, config=PAR, agents=int(rl.n_agents), envs=E, reps=args.reps,
                   steps=args.steps, warmup=args.warmup,
                   reset_ms=dict(median=float(np.median(reset_ms)), all=reset_ms),
                   reset_envs_ms={str(k): dict(median=float(np.median(v)), all=v) for k, v in envs_ms.items()},
                   blocks=rows)
    for w in ("lockstep", "staggered"):
        sel = [b for b in rows if b["batch"] == w]
        summary[w] = dict(ms_per_step_median=float(np.median([b["ms_per_step"] for b in sel])),
                          ms_per_step_min=float(np.min([b["ms_per_step"] for b in sel])),
                          ms_per_step_max=float(np.max([b["ms_per_step"] for b in sel])),
                          time_wfs_ms_median=float(np.median([b["time_wfs_ms"] for b in sel])),
                          extrusion_passes_per_step=float(np.mean([b["extrusion_passes_per_step"] for b in sel])))
    print(json.dumps(summary))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(summary, f, indent=1)
    sim.close()


if __name__ == "__main__":
    main()
