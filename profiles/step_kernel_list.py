"""Kernel list of one env-step of the headline workload (bench.py's 40x40 workload, 43 agents, E = 4096) from
torch.profiler: every device kernel of one aom_step after a reset, the first linear step and warm-up steps, with its
device time.  Run on its own (tracing slows the host); the step time itself comes from bench.py.

    python profiles/step_kernel_list.py [--envs 4096] [--warmup 5] [--out FILE]
"""
import argparse
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the list here")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the GPU and has no CPU fallback")
    from torch.profiler import ProfilerActivity, profile
    import bench
    from ao_marl_b200.system import build_system
    wl = bench.WORKLOADS["40x40"]
    E = args.envs
    sim, t, rl = build_system(wl["par"], E, env_rl=dict(wl["env_rl"]), world_size=wl["world_size"], seed=0)
    sim.reset(1234 + np.arange(E, dtype=np.int64))
    sim.state_begin(); sim.move_atmos(); sim.comp_wfs_image(); sim.do_centroids(); sim.do_control(); sim.state_end()
    for _ in range(args.warmup):
        sim.step(mode=0)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        sim.step(mode=0)
        torch.cuda.synchronize()
    power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    rows = [(e.key, e.count, e.device_time_total) for e in prof.key_averages() if e.device_time_total > 0]
    rows.sort(key=lambda r: -r[2])
    lines = ["card: %s, power limit %s; one aom_step (mode 0), E = %d" % (torch.cuda.get_device_name(), power, E),
             "%10s %6s  %s" % ("device us", "calls", "kernel")]
    lines += ["%10.1f %6d  %s" % (us, n, key[:160]) for key, n, us in rows]
    lines.append("%10.1f         total" % sum(r[2] for r in rows))
    text = "\n".join(lines)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")
    sim.close()


if __name__ == "__main__":
    main()
