#!/usr/bin/env python
"""Benchmark of the batched closed-loop AO environment step (BASELINE.json metric).

    python bench.py --gpus 1 --steps K --warmup W            our arm (CUDA path through the C ABI)
    python bench.py --impl reference ...                     the reference's CPU path (numpy oracle on host cores)
    torchrun ... bench.py --gpus N ...                       one rank per GPU, environments sharded, no collective

A "step" is one env-step of every environment of the batch: all agents' actor forward, rl_control,
apply_control, reward, move_atmos, fused Shack-Hartmann frame, centroids, integrator, state assembly.
Workload: production_sh_40x40_8m_3layers (3 layers, 1200 subapertures, 1286 actuators, 43 windowed agents),
4096 environments per GPU, synthetic von-Karman turbulence from seeds.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

# CPU-baseline worker processes (spawned by cpu_baseline with AOM_BENCH_CPU_WORKER=1) re-import this file first: the
# BLAS / OpenMP pools must be limited BEFORE numpy / torch are imported, otherwise every "one core" worker runs a
# multi-threaded BLAS and N workers oversubscribe the box N times (round-1 finding).
if os.environ.get("AOM_BENCH_CPU_WORKER") == "1":
    for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS", "NUMEXPR_NUM_THREADS", "VECLIB_MAXIMUM_THREADS"):
        os.environ[_v] = "1"

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# DRAM bytes per environment per launch of the sensor kernel from `ncu --set full` (dram__bytes_read.sum +
# dram__bytes_write.sum of one launch at E = 1024, divided by 1024).  Used for roofline.traffic (scaled to the E of this run).
NCU_DRAM_BYTES_PER_ENV = {("40x40", "wfs_frame_ws_kernel"): (4.073935e9 + 14.962176e6) / 1024,      # profiles/r02_wfs_ws_v1_E1024_*
                          ("40x40_d0_noise", "wfs_frame_ws_kernel"): (4.072948e9 + 13.814528e6) / 1024,   # noisy frames run wfs_frame_umma_kernel
                          ("40x40_d0_noise", "wfs_frame_umma_kernel"): (4.072948e9 + 13.814528e6) / 1024,
                          ("40x40", "wfs_frame_umma_kernel"): (4.072948e9 + 13.814528e6) / 1024,   # profiles/r02_wfs_umma_v3_E1024_*
                          ("40x40", "wfs_frame_tma_kernel"): (4.108122e9 + 13.919744e6) / 1024,    # profiles/r01_wfs_tma_E1024_*
                          ("40x40", "wfs_frame_mma_kernel"): (4.062998e9 + 18.132992e6) / 1024}

ROOFLINE_NOTES = {
    "wfs_frame_ws_kernel": "both DFT stages on tcgen05 with the phases on specialised warps (8 field + 4 transform warps per CTA, 24 "
                           "warps per SM, UTCHMMA / LDTM / UTMALDG, packed FFMA2 arithmetic, ~915 warp instructions per subaperture): "
                           "issue slots 52 % busy, shared-memory wavefronts of the LSU at 56 % of their peak next to the tensor "
                           "core's operand fetch (21 % of cycles) and the TMA fills, tensor pipe 16 %, DRAM 24 %: bound by latency "
                           "and shared-memory bandwidth of the per-subaperture pipeline, neither by HBM nor by the tensor pipe; see "
                           "DESIGN.md section 4.1",
    "wfs_frame_umma_kernel": "both DFT stages on tcgen05 (UTCHMMA, no HMMA; tensor pipe 14 %, DRAM 21 %): bound by the CUDA-core "
                             "instruction stream around the tensor core (~1060 useful warp instructions per subaperture: bilinear "
                             "trace, mirrors, sincos, fp16 hi/lo splits of both operands, |.|^2, centroid) at ~0.5 IPC per scheduler "
                             "with 16 warps per SM; neither HBM nor tensor bound, see DESIGN.md section 4",
    "wfs_frame_tma_kernel": "round-1 kernel: bound by its instruction count (~1110 warp instructions per subaperture, 144 of them "
                            "mma.sync, at ~0.53 IPC per scheduler; HMMA pipe 50 %, DRAM 19 %)",
    "wfs_frame_kernel": "issue-bound on the FP32 pipe (SIMT pruned FFT), not on HBM",
}

WORKLOADS = {
    "40x40": dict(par="production_sh_40x40_8m_3layers.py", world_size=44,
                  env_rl=dict(n_zernike_start_end=[0, 1260], window_n_zernike=20, include_tip_tilt_windowed=True,
                              n_reverse_filtered_from_cmat=5, delayed_assignment=2),
                  name="production_sh_40x40_8m_3layers, 43 agents (42x30 modes + TT, window 20), delay 1"),
    # BASELINE.json config 4: its own parameter file (delay 0, magnitude 9 -> 241 photons per subaperture, 3 e- read
    # noise, gain 0.3) with the conv autoencoder denoiser in the state path (selected by --denoise)
    "40x40_d0_noise": dict(par="production_sh_40x40_8m_3layers_d0_noise.py", world_size=44,
                           env_rl=dict(n_zernike_start_end=[0, 1260], window_n_zernike=20, include_tip_tilt_windowed=True,
                                       n_reverse_filtered_from_cmat=5, delayed_assignment=1),
                           name="production_sh_40x40_8m_3layers_d0_noise, 43 agents, delay 0, photon + 3 e- read noise"),
    "10x10": dict(par="production_sh_10x10_2m.py", world_size=3,
                  env_rl=dict(n_zernike_start_end=[0, 80], n_reverse_filtered_from_cmat=5),
                  name="production_sh_10x10_2m, 2 agents (80 modes + TT), delay 1"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="env-steps in every timed section (headline, variants, end to end)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="40x40", choices=sorted(WORKLOADS))
    ap.add_argument("--envs", type=int, default=None, help="environments per GPU (default 4096 / 1024)")
    ap.add_argument("--cpu-seconds", type=float, default=20.0, help="budget of the bounded CPU baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--denoise", action="store_true",
                    help="run the fused per-subaperture denoiser inside every step (row a-6; the *_d0_noise files use it)")
    ap.add_argument("--geo", action="store_true",
                    help="also run the parameter file's geometric controller every step (SURVEY 8(f) rank 4; off by default)")
    ap.add_argument("--wfs-path", default=None,
                    choices=["umma_ws", "umma", "umma_fast", "simt", "tensor", "tensor_fast", "tensor_reg"],
                    help="Shack-Hartmann frame kernel (default: the library's product path)")
    ap.add_argument("--strehl-peak", action="store_true",
                    help="with --strehl: SE / LE from the fitted peak of the 3 x 3 PSF core instead of the on-axis pixel")
    ap.add_argument("--strehl", action="store_true",
                    help="evaluate the target Strehl inside every timed step, as the reference's next_part_two does by "
                         "default (compute_tar_psf=True, rlSupervisor.py:944-947); without the flag the figure is still "
                         "reported as a variant beside the headline")
    ap.add_argument("--no-variants", action="store_true", help="skip the extra sections (Strehl variant, learner, reset timing)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step left for its caller to DIR/<name>.npy (see dump_outputs)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.denoise and a.workload == "40x40":
        a.workload = "40x40_d0_noise"          # config 4 runs on its own parameter file
    return a


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=f,
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            with open(self.path) as f:
                for line in f:
                    p = [x.strip() for x in line.split(",")]
                    if len(p) < 9:
                        continue
                    try:
                        sm.append(float(p[1]))
                        mx.append(float(p[2]))
                    except ValueError:
                        continue
                    for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                                         p[5:9]):
                        if val.lower().startswith("active"):
                            reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out["sm_mhz"] = float(np.median(sm))
            out["sm_max_mhz"] = float(max(mx))
        out["reasons"] = sorted(reasons)
        return out


# ------------------------------------------------------------------------------------------------
def cpu_env_factory(workload_key, cmat_cache=None):
    """Builds the numpy oracle environment of a workload (CPU only: tables by the host builders, interaction
    matrix through the oracle's own Shack-Hartmann pipeline)."""
    from ao_marl_b200 import tables
    from ao_marl_b200.config import load_config_from_file
    from ao_marl_b200.init import rtc as rtc_b
    from ao_marl_b200.rl.layout import RLLayout
    from oracle import loop
    wl = WORKLOADS[workload_key]
    t = tables.build_static(load_config_from_file(wl["par"]))
    tables.build_basis(t)
    tab = t.as_oracle_dict()
    tab["wfs_index"] = t.wfs_index
    if cmat_cache is not None and os.path.exists(cmat_cache):
        cmat = np.load(cmat_cache)
    else:
        # the timing does not depend on the values of the command matrix: the geometric interaction matrix
        # (pre-filter columns dropped) stands in for the measured one to keep the start-up bounded
        D = rtc_b.imat_geom(t.p_wfs, [t.p_pzt, t.p_tt], t.config.p_geom)
        cmat = rtc_b.cmat_with_btt(D, t.Btt, 5)
    env_rl = dict(wl["env_rl"], parameters_telescope=wl["par"])
    rl = RLLayout(t.Btt.shape[1], env_rl, None, wl["world_size"], seed=0)
    return lambda seed: loop.OracleEnv(tab, cmat, t.Btt, t.P, rl, seed=seed), t, rl


def _host_cores():
    try:
        return sorted(os.sched_getaffinity(0))
    except Exception:
        return list(range(os.cpu_count() or 1))


def _cpu_worker(args):
    """One oracle environment on ONE pinned host core with single-threaded BLAS / torch."""
    blob_path, seed, seconds, min_steps, core = args
    import pickle
    if core is not None:
        try:
            os.sched_setaffinity(0, {core})
        except Exception:
            pass
    threads = {"omp_env": os.environ.get("OMP_NUM_THREADS")}
    try:
        import torch
        torch.set_num_threads(1)
        threads["torch"] = torch.get_num_threads()
    except Exception:
        pass
    try:
        from threadpoolctl import threadpool_info, threadpool_limits
        threadpool_limits(1)
        threads["blas"] = max([int(x.get("num_threads", 1)) for x in threadpool_info()] or [1])
    except Exception:
        pass
    from oracle import loop
    with open(blob_path, "rb") as f:
        d = pickle.load(f)
    env = loop.OracleEnv(d["tab"], d["cmat"], d["Btt"], d["P"], d["rl"], seed=seed)
    # no 2N-extrusion reset inside the sample: start from a short warm-up of the screens
    for l in range(env.atm.nl):
        for _ in range(8):
            env.atm._one(l, 0, 1)
    state = env.linear_step()
    t0 = time.perf_counter()
    n = 0
    while True:
        a, _ = env.actors(state)
        state, _ = env.env_step(a)
        n += 1
        el = time.perf_counter() - t0
        if (el >= seconds and n >= min_steps) or n >= 100000:
            break
    return n, el, threads


_BLOBS = {}


def cpu_baseline(workload_key, seconds, procs=1):
    """env-steps/s of the oracle on `procs` host processes (one environment, one pinned core, one BLAS thread each),
    bounded sample.  The static tables are built once in this process and handed to the workers through a pickle;
    the workers are always spawned so that their thread pools are limited before numpy / torch load."""
    import multiprocessing as mp
    import pickle
    t0 = time.perf_counter()
    if workload_key not in _BLOBS:
        make, t, rl = cpu_env_factory(workload_key)
        cells = dict(zip(make.__code__.co_freevars, (c.cell_contents for c in make.__closure__)))
        _BLOBS[workload_key] = dict(tab=cells["tab"], cmat=cells["cmat"], Btt=cells["t"].Btt, P=cells["t"].P, rl=cells["rl"])
    blob = _BLOBS[workload_key]
    with tempfile.NamedTemporaryFile("wb", suffix=".pkl", delete=False) as f:
        pickle.dump(blob, f, protocol=pickle.HIGHEST_PROTOCOL)
        path = f.name
    cores = _host_cores()
    procs = max(1, min(int(procs), len(cores)))
    saved = {k: os.environ.get(k) for k in ("AOM_BENCH_CPU_WORKER",)}
    os.environ["AOM_BENCH_CPU_WORKER"] = "1"
    try:
        ctx = mp.get_context("spawn")
        with ctx.Pool(procs) as pool:
            res = pool.map(_cpu_worker, [(path, 1234 + i, seconds, 2, cores[i % len(cores)]) for i in range(procs)])
    finally:
        os.unlink(path)
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    rate = sum(n / el for n, el, _ in res)
    steps = sum(n for n, _, _ in res)
    el_max = max(el for _, el, _ in res)
    return dict(value=rate, unit="env-steps/s", cores=procs, per_core=rate / procs, host_cores=len(cores),
                os_cpu_count=os.cpu_count(), threads_per_process=res[0][2], kind="port",
                sample="%d env-steps of 1 environment per process on %d pinned single-thread process(es), %.1f s of "
                       "stepping (oracle/loop.py: numpy frame + CPU torch actors), start-up %.0f s excluded"
                       % (steps, procs, el_max, time.perf_counter() - t0 - el_max))


# ------------------------------------------------------------------------------------------------
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = WORKLOADS[args.workload]
    procs = len(_host_cores())
    per_step = max(2.0, args.cpu_seconds / max(1, args.steps + args.warmup))
    t0 = time.perf_counter()
    base = cpu_baseline(args.workload, per_step * (args.steps + args.warmup), procs)
    one = cpu_baseline(args.workload, min(10.0, args.cpu_seconds), 1)      # BASELINE.md section 3: all cores and 1 core
    base["one_core"] = {"value": one["value"], "unit": one["unit"], "sample": one["sample"]}
    line = {
        "impl": "reference", "metric": "AO env-steps/s (batched closed-loop step + actor forward)",
        "value": base["value"], "unit": "env-steps/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 / base["value"] if base["value"] else None, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl["name"], "envs_per_process": 1, "processes": procs,
                   "note": "reference CPU path = numpy restatement of the sutra frame (the compiled simulator is not "
                           "in the reference repo) + reference-architecture actors on CPU torch"},
        "cpu_baseline": base,
        "e2e": {"value": base["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": time.perf_counter() - t0,
    }
    print(json.dumps(line))


def measure_variants(args, sim, t, rl, E, dist, barrier, ev):
    """Extra timed sections of the same run (device times in ms, max over ranks taken by the caller):
    strehl_ms   one env-step with the target Strehl evaluated every frame (the reference's default compute_tar_psf=True)
    learn_*     config 5: one batched SAC update of all agents per env-step, gradients all-reduced over NCCL"""
    import torch
    out = {}
    k = args.steps
    if not args.strehl:
        sim.step_with_strehl(True, 1.65)
        for _ in range(2):
            sim.step(mode=0)
        barrier()
        a, b = ev(enable_timing=True), ev(enable_timing=True)
        a.record()
        for _ in range(k):
            sim.step(mode=0)
        b.record()
        barrier()
        out["strehl_ms"] = a.elapsed_time(b) / k
        sim.strehl_from_peak(True)                  # fitted PSF-core peak (comp_strehl(do_fit=True)) instead of the on-axis pixel
        sim.step(mode=0)
        barrier()
        a, b = ev(enable_timing=True), ev(enable_timing=True)
        a.record()
        for _ in range(k):
            sim.step(mode=0)
        b.record()
        barrier()
        out["strehl_peak_ms"] = a.elapsed_time(b) / k
        sim.strehl_from_peak(False)
        sim.step_with_strehl(False)
    if rl.n_agents:
        from ao_marl_b200.env.trainer import StepLearner
        from ao_marl_b200.rl.sac import BatchedSAC
        learner = BatchedSAC.from_layout(rl, device="cuda", seed=3, dist=dist, memory_size=4 * E)
        sl = StepLearner(sim, rl, learner)
        for _ in range(sl.mdp.depth + 2):           # fill the credit-assignment window and the replay
            sl.step(learn=False)
        for _ in range(2):                          # warm-up of the update (autograd graphs, optimiser state)
            sl.step(learn=True, overlap=True)
        barrier()
        times = {}
        for name, kw in (("learn_step_ms", dict(learn=True, overlap=True)), ("learn_serial_ms", dict(learn=True, overlap=False)),
                         ("learn_env_only_ms", dict(learn=False))):
            a, b = ev(enable_timing=True), ev(enable_timing=True)
            a.record()
            for _ in range(k):
                sl.step(**kw)
            b.record()
            barrier()
            times[name] = a.elapsed_time(b) / k
        out.update(times)
        # the update alone, and its gradient all-reduces alone (three buckets: critics, actors, temperatures)
        a, b = ev(enable_timing=True), ev(enable_timing=True)
        a.record()
        for _ in range(k):
            learner.update()
        b.record()
        barrier()
        out["learn_update_ms"] = a.elapsed_time(b) / k
        buckets = [learner.critic_params, learner.actor_params, [learner.log_alpha]]
        out["allreduce_bytes"] = int(sum(p.numel() for bk in buckets for p in bk) * 4)
        out["allreduce_ms"] = 0.0
        if dist is not None:
            for bk in buckets:
                for p in bk:
                    if p.grad is None:
                        p.grad = torch.zeros_like(p)
            a, b = ev(enable_timing=True), ev(enable_timing=True)
            a.record()
            for _ in range(k):
                for bk in buckets:
                    learner._allreduce(bk)
            b.record()
            barrier()
            out["allreduce_ms"] = a.elapsed_time(b) / k
        out["learn_agents"] = int(rl.n_agents)
        out["learn_batch"] = int(learner.batch_size)
        del sl, learner
        torch.cuda.empty_cache()
    return out


def format_variants(v, args, E, world, ms):
    out = {}
    if "strehl_ms" in v:
        out["with_strehl_every_frame"] = {
            "ms_per_step": v["strehl_ms"], "value": E * world / (v["strehl_ms"] * 1e-3), "unit": "env-steps/s",
            "note": "aom_step with AOM_OPT_STREHL: target Strehl (pupil sums, no focal-plane image) evaluated after "
                    "apply_control on every frame, as the reference's default next_part_two does (rlSupervisor.py:944-947); "
                    "the turbulence update then cannot run beside the actor GEMMs"}
    if "strehl_peak_ms" in v:
        out["with_peak_strehl_every_frame"] = {
            "ms_per_step": v["strehl_peak_ms"], "value": E * world / (v["strehl_peak_ms"] * 1e-3), "unit": "env-steps/s",
            "note": "the same with the 3 x 3 PSF core of the reference's focal grid summed in the sweep and the fitted "
                    "peak as SE / LE (comp_strehl(do_fit=True), targetCompass.py:139-196)"}
    if "learn_step_ms" in v:
        out["learn"] = {
            "config": "config 5: %d agents, batch %d, one SAC update of every agent per env-step, gradients "
                      "all-reduced over %d rank(s)" % (v.get("learn_agents", 0), v.get("learn_batch", 0), world),
            "ms_per_step_overlapped": v["learn_step_ms"], "ms_per_step_serial": v["learn_serial_ms"],
            "ms_per_step_env_only": v["learn_env_only_ms"], "ms_per_update_alone": v["learn_update_ms"],
            "env_steps_per_s": E * world / (v["learn_step_ms"] * 1e-3), "updates_per_s": 1e3 / v["learn_step_ms"],
            "agent_updates_per_s": v.get("learn_agents", 0) * 1e3 / v["learn_step_ms"],
            "allreduce_bytes_per_update": v.get("allreduce_bytes", 0), "allreduce_ms_per_update": v.get("allreduce_ms", 0.0),
            "overlap": "update on a second stream beside aom_step: hidden fraction = %.2f"
                       % max(0.0, min(1.0, (v["learn_serial_ms"] - v["learn_step_ms"]) / max(v["learn_update_ms"], 1e-9))),
            "note": "env-only includes the replay pushes (state / action gathers per agent); reference semantics "
                    "train_rpc.py:759-781, 1084-1133"}
    return out


DUMP_MAX_ENVS = 512
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(path, sim, t, rl, E, args):
    """Writes what the last timed step left for its caller -- state, rewards, actions, slopes and commands, plus the
    Strehl figures / geometric commands when the step computes them -- as float32 `path/<name>.npy`, [n, width] rows of
    a fixed seeded sample of n <= 512 environments (their indices in env_index.npy), at most 64 MB in all.  The inputs
    of a run depend only on its arguments, so two builds run with the same arguments can be compared file for file."""
    import torch
    outs = [("state", "STATE", rl.state_dim), ("reward", "REWARD", rl.n_agents), ("action", "ACTION", rl.action_dim),
            ("slopes", "SLOPES", t.nslopes), ("commands", "COM", t.nactu)]
    if args.strehl:
        outs.append(("strehl", "STREHL", 4))
    if args.geo:
        outs.append(("geo_commands", "GEO_COM", t.nactu))
    per_env = 8 + 4 * sum(width for _, _, width in outs)
    n = min(E, DUMP_MAX_ENVS, DUMP_MAX_BYTES // per_env)
    idx = np.sort(np.random.default_rng(0).choice(E, n, replace=False))
    sel = torch.as_tensor(idx, device="cuda")
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "env_index.npy"), idx.astype(np.float64))
    for name, buf, width in outs:
        np.save(os.path.join(path, name + ".npy"), sim.rows(buf, width).index_select(0, sel).cpu().numpy())


def run_ours(args):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py (our arm) needs a CUDA device: there is no CPU path")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from ao_marl_b200.system import build_system
    wl = WORKLOADS[args.workload]
    E = args.envs or (4096 if args.workload.startswith("40x40") else 1024)
    t_build = time.perf_counter()
    sim, t, rl = build_system(wl["par"], E, env_rl=dict(wl["env_rl"]), world_size=wl["world_size"], seed=0)
    if args.wfs_path:
        sim.set_wfs_path(args.wfs_path)
    if args.strehl:
        sim.step_with_strehl(True, 1.65)
        sim.strehl_from_peak(bool(args.strehl_peak))
    if args.denoise:
        from ao_marl_b200.denoiser import Autoencoder
        Autoencoder(dict(type="cnn_single_subaperture", path="autoencoder_M9_rms_3"), device="cuda", sim=sim)
        sim.step_with_denoiser(True)
    if args.geo:
        from ao_marl_b200.init import geo as geo_b
        sim.set_geo(*geo_b.build_geo(t))
        sim.step_with_geo(True)
    wfs_kernel_name = sim.wfs_kernel()
    seeds = 1234 + rank * E + np.arange(E, dtype=np.int64)
    torch.cuda.synchronize()
    r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l_reset = sim.launches()
    r0.record()
    sim.reset(seeds)                  # RlSupervisor.reset: 2N extrusions per layer (SURVEY 3.3), timed on its own
    r1.record()
    torch.cuda.synchronize()
    reset_ms = r0.elapsed_time(r1)
    l_reset = sim.launches() - l_reset
    # first frame of the episode (AoEnv.reset ends with one linear step)
    sim.state_begin(); sim.move_atmos(); sim.comp_wfs_image(); sim.do_centroids(); sim.do_control(); sim.state_end()
    torch.cuda.synchronize()
    t_build = time.perf_counter() - t_build

    ev = torch.cuda.Event

    def one_step():
        # TrainerRPC.episode body (train_rpc.py:503-553): one aom_step = actors, rl_control, apply_control, reward,
        # move_atmos (on the library's second stream, next to the actor GEMMs), sensor frame, centroids, control, state
        sim.step(mode=0)

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        one_step()
    sampler = ClockSampler(local_rank)
    barrier()
    sim.time_wfs(True)                # CUDA events around the sensor-kernel launches, on the launching stream
    sampler.start()
    l0 = sim.launches()
    torch.cuda.profiler.start()      # ncu --profile-from-start off captures the timed region only
    e0, e1 = ev(enable_timing=True), ev(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        one_step()
    e1.record()
    barrier()
    torch.cuda.profiler.stop()
    clocks = sampler.stop()
    launches = sim.launches() - l0
    ms = e0.elapsed_time(e1)
    wfs_ms, _ = sim.wfs_time_ms()
    sim.time_wfs(False)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, sim, t, rl, E, args)

    variants = {}
    if not args.no_variants:
        variants = measure_variants(args, sim, t, rl, E, dist, barrier, ev)

    # end to end through host buffers: the actions of every step come from pinned host memory (H2D) and go back to
    # it (D2H) -- the host is in the action loop, as in the reference's env.step -- and the step's state and rewards
    # are read back to pinned host memory too.  State / rewards are not fed back, so their D2H runs on a copy stream
    # from a device-side snapshot while the next step computes (double buffered; the host sees them one step late);
    # every copy is inside the timed region and complete before it ends.
    act_h = torch.zeros((E, rl.action_dim), dtype=torch.float32).pin_memory()
    st_h = [torch.zeros((E, rl.state_dim), dtype=torch.float32).pin_memory() for _ in range(2)]
    rw_h = [torch.zeros((E, rl.n_agents), dtype=torch.float32).pin_memory() for _ in range(2)]
    act_d = sim.rows("ACTION", rl.action_dim)
    st_d = sim.rows("STATE", rl.state_dim)
    rw_d = sim.buffer("REWARD").view(E, rl.n_agents)
    st_snap = [torch.empty((E, rl.state_dim), device="cuda") for _ in range(2)]
    rw_snap = [torch.empty((E, rl.n_agents), device="cuda") for _ in range(2)]
    copy_stream = torch.cuda.Stream()
    snap_ready = [ev() for _ in range(2)]
    snap_copied = [ev() for _ in range(2)]
    main = torch.cuda.current_stream()
    act_h.copy_(act_d)
    k_e2e = args.steps                            # the same K as the device-timed loop
    barrier()
    f0, f1 = ev(enable_timing=True), ev(enable_timing=True)
    f0.record()
    atmos_stream = torch.cuda.Stream()
    frame_done = ev()
    for i in range(k_e2e):
        b = i & 1
        act_d.copy_(act_h, non_blocking=True)       # H2D: this step's actions
        main.wait_stream(atmos_stream)              # the turbulence of this step was advanced during the last round trip
        sim.step(mode=1, atmos_done=(i > 0 and not args.strehl))   # rl half-step + reward + linear half-step
        if i + 1 < k_e2e and not args.strehl:
            # the next step's turbulence does not depend on the actions: it runs on a second stream while the
            # actions make their round trip through the host (the GPU would idle on PCIe and the host sync)
            frame_done.record(main)
            atmos_stream.wait_event(frame_done)
            with torch.cuda.stream(atmos_stream):
                sim.move_atmos()
        sim.actor_forward(False)                    # next actions from the new state
        act_h.copy_(act_d, non_blocking=True)       # D2H: next actions
        if i >= 2:
            main.wait_event(snap_copied[b])         # the snapshot of step i-2 has left the device
        st_snap[b].copy_(st_d, non_blocking=True)
        rw_snap[b].copy_(rw_d, non_blocking=True)
        snap_ready[b].record(main)
        copy_stream.wait_event(snap_ready[b])
        with torch.cuda.stream(copy_stream):
            st_h[b].copy_(st_snap[b], non_blocking=True)    # D2H: state, rewards (overlaps the next step)
            rw_h[b].copy_(rw_snap[b], non_blocking=True)
            snap_copied[b].record(copy_stream)
        main.synchronize()                          # the host owns the actions before the next step
    main.wait_stream(copy_stream)
    f1.record()
    barrier()
    ms_e2e = f0.elapsed_time(f1)

    vkeys = sorted(k for k, v in variants.items() if isinstance(v, float))
    t_all = torch.tensor([ms, ms_e2e, wfs_ms, reset_ms] + [variants[k] for k in vkeys], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(t_all, op=dist.ReduceOp.MAX)
    vals = [float(x) for x in t_all.cpu()]
    ms, ms_e2e, wfs_ms, reset_ms = vals[:4]
    for k, v in zip(vkeys, vals[4:]):
        variants[k] = v
    if rank == 0:
        peaks = {}
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                peaks = json.load(f)
        except Exception:
            pass
        hbm = float(peaks.get("hbm_gbs", 6650.0))
        w = t.p_wfs
        bytes_per_frame = w._nvalid * (w._pdiam ** 2 * 4 + w.npix ** 2 * 4 + 2 * 4)      # SURVEY 8(d)
        achieved = bytes_per_frame * E / (wfs_ms * 1e-3) / 1e9
        flops_per_frame = w._nvalid * 8.0 * (32 * 16 * 16 + 32 * 16 * 32)                # pruned DFT-as-GEMM count
        total_steps = args.steps * E * world
        line = {
            "metric": "AO env-steps/s (batched closed-loop step + actor forward)",
            "value": total_steps / (ms * 1e-3), "unit": "env-steps/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["name"], "envs_per_gpu": E, "total_envs": E * world,
                       "strehl_every_frame": bool(args.strehl),
                       "parallelism": "env-sharded x%d, no collective on the step path" % world, "wfs_path": args.wfs_path,
                       "geo_controller": bool(args.geo), "denoiser": bool(args.denoise),
                       "l2": "inputs larger than L2 (%.1f GB of screens per GPU)" % (
                           sum(int(n) ** 2 for n in t.dim_screens) * 4 * E / 1e9),
                       "us_per_frame": ms / args.steps / E * 1e3, "build_s": t_build},
            "roofline": {"kernel": wfs_kernel_name, "bound": "hbm", "achieved": achieved, "peak": hbm,
                         "unit": "GB/s", "frac": achieved / hbm,
                         "traffic": (NCU_DRAM_BYTES_PER_ENV[(args.workload, wfs_kernel_name)] * E
                                     if (args.workload, wfs_kernel_name) in NCU_DRAM_BYTES_PER_ENV else None),
                         "traffic_source": "ncu dram bytes per env at E=1024 (profiles/) x E",
                         "algorithmic_bytes": bytes_per_frame * E,
                         "peak_source": "measured" if peaks else "fallback",
                         "ms_per_launch": wfs_ms, "share_of_step": wfs_ms / (ms / args.steps),
                         "fp32_tflops_algorithmic": flops_per_frame * E / (wfs_ms * 1e-3) / 1e12,
                         "note": ROOFLINE_NOTES.get(wfs_kernel_name, "see DESIGN.md section 4")},
            "e2e": {"value": k_e2e * E * world / (ms_e2e * 1e-3), "unit": "env-steps/s",
                    "h2d_bytes_per_step": int(E * rl.action_dim * 4),
                    "d2h_bytes_per_step": int(E * (rl.action_dim + rl.state_dim + rl.n_agents) * 4), "steps": k_e2e,
                    "note": "actions H2D + D2H synchronously every step (host in the loop); state and rewards D2H from a "
                            "device snapshot on a copy stream, overlapped with the next step; the next step's turbulence "
                            "update (independent of the actions) runs on a second stream during the round trip"},
            "gpu_launches": int(launches), "clocks": clocks,
            "reset": {"ms": reset_ms, "gpu_launches": int(l_reset),
                      "extrusions": int(sum(2 * int(n) for n in t.dim_screens)),
                      "ms_per_step_amortised_over_1000": reset_ms / 1000.0,
                      "value_with_reset_per_1000_steps": total_steps / ((ms + args.steps * reset_ms / 1000.0) * 1e-3),
                      "note": "RlSupervisor.reset (rlSupervisor.py:236-246): 2N sequential extrusions per layer, once per "
                              "1000-step episode; not inside the timed steps"},
        }
        line.update(format_variants(variants, args, E, world, ms))
        if not args.no_cpu_baseline and world == 1:
            try:
                line["cpu_baseline"] = cpu_baseline(args.workload, args.cpu_seconds, 1)
            except Exception as exc:   # the baseline is reported, never allowed to sink the GPU number
                line["cpu_baseline"] = {"value": None, "unit": "env-steps/s", "cores": 1, "kind": "port",
                                        "sample": "failed: %r" % (exc,)}
        print(json.dumps(line))
    sim.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
