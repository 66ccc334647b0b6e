"""Cost of per-environment winds on the default workload (production_sh_40x40_8m_3layers, 43 agents, E = 4096).

Times aom_step (mode 0: actors, controller, turbulence, sensor frame, state) with the configuration's common winds and
with one wind per environment and layer (speeds around the layer's own, all directions, seeded), alternating the two
in one process on the same context.  Per block: CUDA events around `--steps` steps after `--warmup` untimed ones, the
sensor kernel's own time from the library's event pairs (AOM_OPT_TIME_WFS), and the extrusion passes per step derived
from the winds with the library's accumulator arithmetic (oracle.aoframe.OracleAtmos.move: per layer |nx| + |ny|, with
per-environment winds the largest count of the batch on each axis).  Prints the card and its power limit, then one
line per block and a JSON summary.

    python profiles/wind_per_env_time.py [--envs 4096] [--steps 40] [--warmup 10] [--rounds 3] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

PAR = "production_sh_40x40_8m_3layers.py"
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


def passes(dx, dy, steps):
    """Extrusion passes of each of `steps` frames from zeroed accumulators: dx, dy float32 [L][E]."""
    L, E = dx.shape
    ax, ay = np.zeros((L, E)), np.zeros((L, E))
    out = []
    for _ in range(steps):
        n = 0
        ax += dx.astype(np.float64)
        ay += dy.astype(np.float64)
        nx, ny = np.trunc(ax), np.trunc(ay)
        ax -= nx
        ay -= ny
        n += int(np.abs(nx).max(axis=1).sum() + np.abs(ny).max(axis=1).sum())
        out.append(n)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--seed", type=int, default=2026)
    ap.add_argument("--spread", type=float, default=0.3, help="relative spread of the speeds around each layer's")
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
    cdx = np.array([sim.cfg.deltax[l] for l in range(L)], np.float32)
    cdy = np.array([sim.cfg.deltay[l] for l in range(L)], np.float32)
    r = np.random.default_rng(args.seed)
    speed = np.hypot(cdx.astype(np.float64), cdy.astype(np.float64))[:, None] * (1.0 + args.spread * r.uniform(-1, 1, (L, E)))
    ang = r.uniform(0.0, 2 * np.pi, (L, E))
    pdx, pdy = (speed * np.cos(ang)).astype(np.float32), (speed * np.sin(ang)).astype(np.float32)
    seeds = 1234 + np.arange(E, dtype=np.int64)

    def setup(per_env):
        for l in range(L):
            if per_env:
                sim.set_layer_wind(l, pdx[l], pdy[l])
            else:
                sim.set_layer_wind(l, None, None)
        sim.reset(seeds)                 # accumulators from zero: the pass counts below follow
        sim.state_begin(); sim.move_atmos(); sim.comp_wfs_image(); sim.do_centroids(); sim.do_control(); sim.state_end()
        torch.cuda.synchronize()

    def block(per_env):
        setup(per_env)
        for _ in range(args.warmup):
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
        d = (pdx, pdy) if per_env else (np.repeat(cdx[:, None], E, 1), np.repeat(cdy[:, None], E, 1))
        pp = passes(d[0], d[1], 1 + args.warmup + args.steps)[1 + args.warmup:]
        return dict(winds="per_env" if per_env else "common", ms_per_step=e0.elapsed_time(e1) / args.steps,
                    extrusion_passes_per_step=float(np.mean(pp)), time_wfs_ms=wfs_ms, wfs_timed_launches=n_wfs,
                    wfs_kernel=sim.wfs_kernel())

    rows = []
    for rnd in range(args.rounds):
        for per_env in (False, True):
            b = block(per_env)
            b["round"] = rnd
            rows.append(b)
            print("round %d %-7s  %7.3f ms/step  %5.2f extrusion passes/step  sensor kernel %6.3f ms (%s)" % (
                rnd, b["winds"], b["ms_per_step"], b["extrusion_passes_per_step"], b["time_wfs_ms"], b["wfs_kernel"]),
                flush=True)
    summary = dict(card=name, power_limit=power, config=PAR, agents=int(rl.n_agents), envs=E, steps=args.steps,
                   warmup=args.warmup, seed=args.seed, speed_spread=args.spread, blocks=rows)
    for w in ("common", "per_env"):
        sel = [b for b in rows if b["winds"] == w]
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
