"""Cost of per-environment guide star, sensor noise and integrator gain on aom_step (43 agents, E = 4096).

Times aom_step (mode 0: actors, controller, turbulence, sensor frame, state) in three pairs of variants, alternating
the variants of a pair block by block in one process on the same context:

  d1_noise   production_sh_40x40_8m_3layers_d1_noise with its common conditions (magnitude 9, 3 e- read noise, gain
             0.65) against one magnitude per environment (uniform over 4 .. 11), noise drawn from {0, 3, 5} e- and the
             gain of the parameter file that matches the magnitude (0.7 below 7, 0.65 up to 9, 0.3 above).  Controls:
             per-environment arrays that all hold the common values (the cost of the per-environment kernels alone),
             and the common conditions at magnitude 4 (the photon sampler's cost grows with the photon count)
  gains      production_sh_40x40_8m_3layers (noise-free) against one gain per environment drawn from the parameter
             files' gains {0.7, 0.6, 0.7, 0.3, 0.65}
  half_noisy production_sh_40x40_8m_3layers against every other environment with 3 e- read noise (the other half
             noise-free); control: every environment with 3 e- read noise (common value, uniform kernel)

Per block: CUDA events around `--steps` steps after `--warmup` untimed ones, and the sensor kernel's own time from the
library's event pairs (AOM_OPT_TIME_WFS).  Prints the card and its power limit, then one line per block and a JSON
summary.

    python profiles/noise_gain_per_env_time.py [--envs 4096] [--steps 40] [--warmup 10] [--rounds 3] [--out FILE]
"""
import argparse
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


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--seed", type=int, default=2026)
    ap.add_argument("--out", default=None, help="also write the JSON summary here")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the GPU and has no CPU fallback")
    from ao_marl_b200.init.geom import nphotons_for_mags
    from ao_marl_b200.system import build_system
    name, power = card()
    print("card: %s, power limit %s" % (name, power), flush=True)
    E = args.envs
    r = np.random.default_rng(args.seed)
    seeds = 1234 + np.arange(E, dtype=np.int64)
    rows = []

    def block(sim, pair, variant, apply):
        apply()
        sim.reset(seeds)
        sim.state_begin(); sim.move_atmos(); sim.comp_wfs_image(); sim.do_centroids(); sim.do_control(); sim.state_end()
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
        return dict(pair=pair, variant=variant, ms_per_step=e0.elapsed_time(e1) / args.steps, time_wfs_ms=wfs_ms,
                    wfs_timed_launches=n_wfs)

    def common(sim, nphotons=None):
        """The parameter file's conditions (with another common photon count if given)."""
        def f():
            sim.set_wfs_noise_env(None, None)
            sim.set_gain_env(None)
            sim.set_wfs_noise(float(sim.cfg.noise), float(sim.cfg.nphotons) if nphotons is None else nphotons)
        return f

    def run_pair(sim, pair, variants):
        for rnd in range(args.rounds):
            for v, fn in [("common", common(sim))] + variants:
                b = block(sim, pair, v, fn)
                b["round"] = rnd
                rows.append(b)
                print("round %d %-10s %-12s %7.3f ms/step  sensor kernel %6.3f ms" % (
                    rnd, pair, v, b["ms_per_step"], b["time_wfs_ms"]), flush=True)

    # 1. the _d1_noise file against a spread of magnitudes, noises and matching gains
    par = "production_sh_40x40_8m_3layers_d1_noise.py"
    sim, t, rl = build_system(par, E, env_rl=dict(ENV_RL, parameters_telescope=par), world_size=44, seed=0)
    c, w = t.config, t.p_wfs
    mags = r.uniform(4.0, 11.0, E)
    nph = nphotons_for_mags(c.p_loop.ittime, w.optthroughput, c.p_tel.diam, w.nxsub, w.zerop, mags)
    noise = r.choice(np.array([0.0, 3.0, 5.0], np.float32), E)
    gain = np.where(mags < 7.0, 0.7, np.where(mags <= 9.0, 0.65, 0.3)).astype(np.float32)

    nph0, noise0, gain0 = sim.wfs_nphotons, sim.wfs_noise, float(sim.cfg.gain)
    nph4 = float(nphotons_for_mags(c.p_loop.ittime, w.optthroughput, c.p_tel.diam, w.nxsub, w.zerop, 4.0))

    def mixed():
        sim.set_wfs_noise(noise0, nph0)
        sim.set_wfs_noise_env(noise=noise, nphotons=nph)
        sim.set_gain(gain)

    def equal():
        sim.set_wfs_noise(noise0, nph0)
        sim.set_wfs_noise_env(noise=np.full(E, noise0, np.float32), nphotons=np.full(E, nph0, np.float32))
        sim.set_gain(np.full(E, gain0, np.float32))
    run_pair(sim, "d1_noise", [("per_env", mixed), ("per_env_equal", equal), ("common_mag4", common(sim, nph4))])
    agents = int(rl.n_agents)
    sim.close()

    # 2 and 3. the noise-free default file
    par = "production_sh_40x40_8m_3layers.py"
    sim, t, rl = build_system(par, E, env_rl=dict(ENV_RL), world_size=44, seed=0)
    gains = r.choice(np.array([0.7, 0.6, 0.7, 0.3, 0.65], np.float32), E)
    half = np.where(np.arange(E) % 2 == 1, 3.0, -1.0).astype(np.float32)
    run_pair(sim, "gains", [("per_env_gain", lambda: sim.set_gain(gains))])

    def all_noisy():
        common(sim)()
        sim.set_wfs_noise(3.0)
    run_pair(sim, "half_noisy", [("half_noisy", lambda: sim.set_wfs_noise_env(noise=half)), ("all_noisy", all_noisy)])
    sim.close()

    summary = dict(card=name, power_limit=power, agents=agents, envs=E, steps=args.steps, warmup=args.warmup,
                   seed=args.seed, blocks=rows)
    for pair in ("d1_noise", "gains", "half_noisy"):
        for v in sorted({b["variant"] for b in rows if b["pair"] == pair}):
            sel = [b for b in rows if b["pair"] == pair and b["variant"] == v]
            summary["%s/%s" % (pair, v)] = dict(
                ms_per_step_median=float(np.median([b["ms_per_step"] for b in sel])),
                ms_per_step_min=float(np.min([b["ms_per_step"] for b in sel])),
                ms_per_step_max=float(np.max([b["ms_per_step"] for b in sel])),
                time_wfs_ms_median=float(np.median([b["time_wfs_ms"] for b in sel])))
    print(json.dumps(summary))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(summary, f, indent=1)


if __name__ == "__main__":
    main()
