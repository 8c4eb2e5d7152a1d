#!/usr/bin/env python
"""bench.py -- audio-seconds/sec of the AERO generator forward (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 4-16|12-48|11-44|train] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one forward over one batch of synthetic white-noise clips per GPU; clips are independent, so ranks shard
the batch with no data-path collective ("weak" scaling: the per-GPU batch is fixed).  Rank 0 prints ONE JSON line.

  --config 4-16  (default) BASELINE.json configs[1]: aero_4-16_512_64, 32 x 2 s clips per GPU
  --config 12-48           configs[2]: aero_12-48_512_128, 16 x 2 s clips per GPU (T = 751)
  --config 11-44           configs[4]: aero_11-44_512_64 stereo, 2 x 10 s clips per GPU (8 clips on 4 GPUs; T = 6892)
  --config train           configs[3]: one training step (generator fwd + MR-STFT loss + bwd + Adam), 8 clips per GPU

  value    : device-timed (CUDA events, max over ranks), inputs resident in HBM, on the path a caller gets: the
             CUDA-graph replay `Aero.forward` uses for a steady-state shape.
  e2e      : same metric through the public API with pinned-host input, H2D and D2H of the waveform inside the timed
             region; median of the per-step times (mean also given).
  roofline : dominant kernel family = the decoder's 3x3 rewrite tap-GEMMs, timed with CUDA events on the launch stream
             in a separate eager pass of the same K steps; fraction of the measured burst AND sustained cuBLAS bf16 rates.
  step     : whole-step achieved TFLOP/s against the same peaks, and the step time against the sum of its launches' own
             rooflines (tools/traffic_model.py: algorithmic bytes / FLOPs per launch).
  --dump-outputs DIR : after the timed steps, DIR/out.npy (float32) holds the waveform the last timed step returned on rank 0.
             Inputs and weights are seeded, so two builds run with the same arguments can be compared output for output.
  cpu_baseline / --impl reference : the oracle port (oracle/aero_oracle.py, the same torch library calls the reference
             makes) on the host cores, BASELINE.md section 3 protocol.  The reference is a Python package and cannot travel
             to the GPU box; oracle/ is its pinned restatement.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

import torch  # noqa: E402

SEED = 2036
# workload table: experiment file, clips per GPU, low-rate samples per clip, clip seconds, reference-equivalent GFLOP per clip
# (SURVEY.md 8d) and the GFLOP actually required (decoder-0's structural zeros skipped)
CONFIGS = {
    "4-16": dict(exp="aero_4-16_512_64", batch=32, length=8000, seconds=2.0, gflop=124.16, gflop_req=102.9,
                 name="aero_4-16_512_64 inference forward, 2 s white-noise clips 4->16 kHz (BASELINE configs[1])"),
    "12-48": dict(exp="aero_12-48_512_128", batch=16, length=24000, seconds=2.0, gflop=185.6, gflop_req=None,
                  name="aero_12-48_512_128 inference forward, 2 s white-noise clips 12->48 kHz (BASELINE configs[2])"),
    "11-44": dict(exp="aero_11-44_512_64", batch=2, length=110250, seconds=10.0, gflop=1989.0, gflop_req=None,
                  name="aero_11-44_512_64 inference forward, 10 s stereo white-noise clips 11.025->44.1 kHz (BASELINE configs[4]: "
                       "8 clips on 4 GPUs = 2 per GPU)"),
}
# dram__bytes_read.sum + dram__bytes_write.sum of the largest launch of the roofline family (decoder.0 rewrite, B=32) from the
# `ncu --set full` capture summarised in profiles/
TRAFFIC_NCU = {1: {"kernel": "tapgemm_tc_kernel<0,0,1,tf32> decoder.0.rw B=32", "bytes_per_launch": 473.8e6, "algorithmic_bytes": 513.7e6,
                   "tensor_pipe_pct": 80.8, "source": "profiles/r1_dec0rw_tc_ncu.md"},
               2: {"kernel": "tapgemm_tc_kernel<0,0,1,f16,f16> decoder.0.rw B=32", "bytes_per_launch": 208.2e6, "algorithmic_bytes": 256.9e6,
                   "tensor_pipe_pct": 89.5, "source": "profiles/r2_dec0rw_f16_ncu.md"}}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops_sustained"], "bf16_tflops_burst": d["bf16_tflops"],
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1400.0, "bf16_tflops_burst": 1650.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag, self.period, self.paused = index, [], False, 0.02, False

    def run(self):
        try:                                   # NVML in-process: millisecond polls, no fork on the launching host
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            bits = [(0x8, 2), (0x40, 3), (0x20, 4), (0x4, 5)]      # hw_slowdown, hw_thermal, sw_thermal, sw_power_cap
            while not self.stop_flag:
                if self.paused:
                    time.sleep(0.01)
                    continue
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                row = [str(sm), str(mx), "", "", "", ""]
                for bit, col in bits:
                    row[col] = "Active" if r & bit else "Not Active"
                self.rows.append(row)
                time.sleep(self.period)
            return
        except Exception:
            pass
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag:
            if self.paused:
                time.sleep(0.01)
                continue
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": int(self.rows[0][1]) if self.rows[0][1].isdigit() else None,
                "reasons": reasons, "samples": len(self.rows)}


def pin_to_gpu_numa(index):
    """Run this process on the cores of the GPU's NUMA node (pinned buffers and the launch thread then sit next to the
    PCIe root the GPU hangs off).  Returns the core count, or None if NVML cannot tell."""
    try:
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(index)
        n = os.cpu_count() or 1
        words = nv.nvmlDeviceGetCpuAffinity(h, (n + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def physical_cores():
    try:
        import psutil
        n = psutil.cpu_count(logical=False)
        if n:
            return int(n)
    except Exception:
        pass
    return max(1, (os.cpu_count() or 2) // 2)


def build_model(cfg):
    from util import trained_like_
    from aero_b200 import Aero, aero_kwargs
    torch.manual_seed(SEED)
    m = Aero(**aero_kwargs(cfg["exp"])).eval()
    m.load_state_dict(trained_like_(m.state_dict()))
    return m


def cpu_forward_times(cfg, batch, threads, repeats, warmup):
    """Per-forward wall times of the oracle port (library-call form == what the reference executes) on the host."""
    from oracle import aero_oracle as O
    torch.set_num_threads(threads)
    model = build_model(cfg)
    sd = {k: v.cpu() for k, v in model.state_dict().items()}
    x = torch.randn(batch, model.in_channels, cfg["length"], generator=torch.Generator().manual_seed(SEED))
    times = []
    with torch.no_grad():
        for i in range(warmup + repeats):
            t0 = time.perf_counter()
            O.aero_forward(sd, model.geom, x)
            if i >= warmup:
                times.append(time.perf_counter() - t0)
    return times


def _probe(cfg_key, threads, batch, repeats, warmup, timeout):
    """Run the oracle port in a child process on ALL host cores' affinity (a hung / oversubscribed BLAS cannot stall the
    bench).  Returns the list of per-forward times or None."""
    cmd = [sys.executable, os.path.abspath(__file__), "--config", cfg_key, "--_cpu_probe", f"{threads},{batch},{repeats},{warmup}"]
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout).stdout.strip().splitlines()
        return json.loads(out[-1]) if out else None
    except Exception:
        return None


def median(v):
    v = sorted(v)
    return v[len(v) // 2] if len(v) % 2 else 0.5 * (v[len(v) // 2 - 1] + v[len(v) // 2])


def pick_cpu_threads(cfg_key):
    """Thread count that gives the reference's CPU path its BEST throughput on this host.  BASELINE.md section 3 asks for
    all physical cores; on this pool's 64-core / 2-NUMA hosts that is slower than 16-32 threads (measured: 1.9 vs 3.3-3.7
    audio-s/s at B=32), so the arm uses the best of {all physical, 32, 16} by a B=4 probe and reports which.
    Returns (best, {threads: seconds per probe forward})."""
    env = os.environ.get("AERO_CPU_THREADS")
    if env:
        return int(env), {}
    n = physical_cores()
    seen = {}
    for c in sorted({n, min(n, 32), min(n, 16)}, reverse=True):
        t = _probe(cfg_key, c, 4, 1, 1, 90)
        if t:
            seen[c] = t[0]
    if not seen:
        return min(n, 16), {}
    return min(seen, key=seen.get), seen


def run_reference(args, cfg, rank, world):
    """--impl reference: the reference's CPU implementation of the path (oracle port), host cores only, the SAME batch
    as the GPU arm's per-GPU workload."""
    if rank != 0:
        return
    os.sched_setaffinity(0, range(os.cpu_count() or 1))
    threads, probes = pick_cpu_threads(args.config)
    batch = cfg["batch"]
    per_clip = (probes[threads] / 4) if threads in probes else 1.0
    # keep the workload's own batch; only if (steps + warmup) forwards of it would run past ~4 minutes, shrink the sample (the whole arm,
    # thread probes and the single-thread B=1 line included, then ends in about 6 minutes on this pool's hosts)
    if per_clip * batch * (args.steps + args.warmup) > 240.0:
        batch = max(1, int(240.0 / (per_clip * (args.steps + args.warmup))))
    times = cpu_forward_times(cfg, batch, threads, args.steps, args.warmup)
    dt = sum(times) / len(times)
    val = batch * cfg["seconds"] / dt
    one = _probe(args.config, 1, 1, 3, 1, 120)
    line = {"impl": "reference", "metric": "audio-seconds/sec forward", "value": val, "unit": "audio-s/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "ms_per_step_median": median(times) * 1e3,
            "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": cfg["name"], "batch_per_step": batch, "same_batch_as_gpu_arm": batch == cfg["batch"]},
            "cpu_baseline": {"value": val, "unit": "audio-s/s", "cores": threads, "kind": "port",
                             "host_cores": {"logical": os.cpu_count(), "physical": physical_cores()},
                             "thread_probe_audio_s_per_s": {str(c): 4 * cfg["seconds"] / t for c, t in probes.items()},
                             "single_thread_b1": ({"value": cfg["seconds"] / median(one), "unit": "audio-s/s", "cores": 1,
                                                   "sample": "B=1, 1 warm-up, median of 3 (torch.set_num_threads(1), as reference enhance.py:12)"}
                                                  if one else None),
                             "sample": f"{args.steps} forwards of a {batch}-clip batch after {args.warmup} warm-ups on {threads} threads "
                                       f"(the best of all-physical-cores / 32 / 16 by a B=4 probe), oracle library-call form"},
            "e2e": {"value": val, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(path, out):
    """Write `out` as <path>/out.npy in float32.  Beyond DUMP_MAX_BYTES it is a fixed seeded sample of 4 M flattened
    positions instead, listed in out_index.npy (float64 holds them exactly)."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    flat = out.detach().float().cpu().reshape(-1)
    if flat.numel() * 4 <= DUMP_MAX_BYTES:
        np.save(os.path.join(path, "out.npy"), flat.view(out.shape).numpy())
        return
    idx = torch.randint(0, flat.numel(), (4 << 20,), generator=torch.Generator().manual_seed(SEED)).sort().values
    np.save(os.path.join(path, "out.npy"), flat[idx].numpy())
    np.save(os.path.join(path, "out_index.npy"), idx.double().numpy())


def timed_steps(fn, steps, barrier):
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(steps):
        fn()
    ev1.record()
    barrier()
    return ev0.elapsed_time(ev1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="4-16", choices=sorted(CONFIGS) + ["train"])
    ap.add_argument("--batch", type=int, default=None, help="clips per GPU (default: the BASELINE config's)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the precision sub-lines and the strong-scaling sample")
    ap.add_argument("--precision", type=int, default=None,
                    help="engine precision: 2 (default) FP16-stored activations / kind::f16 tcgen05, 1 fp32 storage / kind::tf32, "
                         "0 every kernel in exact fp32")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the output of the last timed step (rank 0) to DIR/out.npy, float32")
    ap.add_argument("--_cpu_probe", default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.config == "train" or args.impl != "ours"):
        ap.error("--dump-outputs applies to the GPU inference configurations (--impl ours, --config other than train)")
    if args.config == "train":
        import bench_train
        return bench_train.main(args)
    cfg = dict(CONFIGS[args.config])
    if args._cpu_probe:
        th, b, rep, wu = (int(v) for v in args._cpu_probe.split(","))
        os.sched_setaffinity(0, range(os.cpu_count() or 1))
        print(json.dumps(cpu_forward_times(cfg, b, th, rep, wu)), flush=True)
        return
    if args.batch:
        cfg["batch"] = args.batch
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, cfg, rank, world)
        return

    import torch.distributed as dist
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa_cores = pin_to_gpu_numa(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from aero_b200 import cabi
    lib = cabi.load()
    model = build_model(cfg).to(dev)
    eng = model._engine()
    if args.precision is not None:
        eng.precision = args.precision
    B, L, Cin = cfg["batch"], cfg["length"], model.in_channels
    gen = torch.Generator().manual_seed(SEED + rank)
    host_in = torch.randn(B, Cin, L, generator=gen).pin_memory()
    x_dev = host_in.to(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up: packs weights, allocates workspaces, and captures this shape's CUDA graph (the path a steady-state
    #      caller is on from its third call; forced here so that any --warmup reaches it)
    eng.use_graph = True
    out = None
    for _ in range(args.warmup):
        out = model(x_dev)
    eng.use_graph = "auto"
    host_out = torch.empty(out.shape, dtype=out.dtype).pin_memory()
    barrier()
    assert len(eng._graphs) >= 1

    # ---- device-resident timing on the graph path
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    last = []

    def graph_step():
        last[:] = [model(x_dev)]
    ms_dev = timed_steps(graph_step, args.steps, barrier)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last[0])
    del last[:]

    # ---- the same K steps launched eagerly with CUDA events around the roofline kernel family
    fam = ("decoder.0.rw", "decoder.1.rw", "decoder.2.rw", "decoder.3.rw")      # tags = packed-weight names
    eng.start_profile(fam)
    launches0 = lib.aero_launch_count()
    ms_eager = timed_steps(lambda: model(x_dev), args.steps, barrier)
    launches_per_step = (lib.aero_launch_count() - launches0) // args.steps
    prof = eng.stop_profile()

    # ---- end to end through the public API with host buffers.  NVML queries contend with CUDA API calls for driver locks
    #      (measured: +3-4 ms per synchronised step): the clocks were sampled during the device-timed regions above, stop here.
    sampler.paused = True
    barrier()
    stream = torch.cuda.current_stream()
    marks = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    marks[0].record()
    for i in range(args.steps):
        xin = host_in.to(dev, non_blocking=True)
        out = model(xin)
        host_out.copy_(out, non_blocking=True)
        marks[i + 1].record()
        stream.synchronize()                      # the caller reads the result every step
    barrier()
    per_step = [marks[i].elapsed_time(marks[i + 1]) for i in range(args.steps)]
    ms_e2e_mean, ms_e2e_med = sum(per_step) / len(per_step), median(per_step)
    sampler.stop_flag = True

    extras = {}
    if not args.no_extras:
        # other engine precisions on the same workload (eager launches, 3 steps each after one warm-up)
        keep = eng.precision
        for prec in (1, 0):
            if prec == keep:
                continue
            eng.precision = prec
            eng.use_graph = False
            model(x_dev)
            extras[f"precision_{prec}"] = {"ms_per_step": timed_steps(lambda: model(x_dev), 3, barrier),
                                           "what": {1: "fp32 storage rounded to TF32 / tcgen05 kind::tf32", 0: "every kernel in exact fp32 (SIMT)"}[prec]}
        eng.precision, eng.use_graph = keep, "auto"
        if world > 1 and B % world == 0:
            # strong scaling sample: the ONE-GPU workload (B clips in total) split over the ranks
            xs = x_dev[: B // world].contiguous()
            eng.use_graph = True
            for _ in range(3):
                model(xs)
            eng.use_graph = "auto"
            extras["strong"] = {"ms_per_step": timed_steps(lambda: model(xs), args.steps, barrier), "global_batch": B}

    from aero_b200.parallel import reduce_max
    ms_dev, ms_eager, ms_e2e_mean, ms_e2e_med = (reduce_max(v, dev) for v in (ms_dev, ms_eager, ms_e2e_mean, ms_e2e_med))
    for v in extras.values():
        v["ms_per_step"] = reduce_max(v["ms_per_step"], dev)

    if rank == 0:
        pk = peaks()
        total_clips = B * world
        secs = cfg["seconds"]
        value = total_clips * secs / (ms_dev * 1e-3)
        e2e = total_clips * secs / (ms_e2e_med * 1e-3)
        # roofline of the dominant kernel family
        flops = sum(v["flops"] for v in prof.values())
        ms_k = sum(v["ms"] for v in prof.values())
        n_l = sum(v["launches"] for v in prof.values())
        prec = eng.precision
        tf32 = prec == 1
        # kind::f16 runs at the bf16 rate the driver measured with cuBLAS; kind::tf32 at half of it (no TF32 figure is measured)
        div = 2 if tf32 else 1
        peak_s, peak_b = pk["bf16_tflops"] / div, pk["bf16_tflops_burst"] / div
        clk = sampler.summary()
        pipe = (4096 if tf32 else 8192) * 148 * (clk.get("sm_mhz") or 1965) * 1e6 / 1e12     # tcgen05 flop/clk/SM (ncu pipe rate)
        ach = flops / (ms_k * 1e-3) / 1e12 if ms_k > 0 else 0.0
        roof = {"bound": "tensor", "kernel": "tap-GEMM, decoder 3x3 rewrite convs (4 launches/step)",
                "achieved": ach, "peak": peak_b, "unit": "TFLOP/s", "frac": ach / peak_b,
                "frac_burst": ach / peak_b, "frac_sustained": ach / peak_s, "peak_sustained": peak_s,
                "peak_source": pk["source"] + ": cuBLAS bf16 8192^3 best-of-10 (burst; the family is a ~16 % duty cycle of a step at max "
                               "clock, so burst is the denominator of `frac`) and back-to-back for 4 s (sustained)" +
                               ("; TF32 dense peak taken as half the bf16 figure" if tf32 else "; cuBLAS bf16 = the kind::f16 rate") +
                               "; frac_tensor_pipe is the stricter fraction of the tensor pipe's own rate at the sampled clock",
                "peak_tensor_pipe": pipe, "frac_tensor_pipe": ach / pipe,
                "precision": {2: "f16 operands tcgen05 (kind::f16), fp32 accumulate", 1: "tf32 tcgen05", 0: "fp32 SIMT (no tensor pipe)"}[prec],
                "ms_per_step_in_kernel": ms_k / args.steps, "share_of_step": (ms_k / args.steps) / ms_eager,
                "timed_in": "eager pass of the same K steps (CUDA events on the launch stream around each launch of the family)",
                "launches_timed": n_l,
                "per_layer_tflops": {k: (v["flops"] / (v["ms"] * 1e-3) / 1e12 if v["ms"] > 0 else 0.0) for k, v in sorted(prof.items())},
                "traffic": TRAFFIC_NCU.get(prec) if args.config == "4-16" else None}
        gflop_req = cfg["gflop_req"] or cfg["gflop"]
        step_tflops = B * gflop_req * 1e9 / (ms_dev * 1e-3) / 1e12
        step = {"tflops": step_tflops, "frac_sustained": step_tflops / peak_s, "frac_burst": step_tflops / peak_b,
                "gflop_per_clip_counted": gflop_req}
        try:
            import traffic_model
            sr = traffic_model.step_roofline(cfg["exp"], B, L, prec, p_tensor=peak_s * 1e12)
            step.update({"sum_of_launch_rooflines_ms": sr["sum_roofline_ms"], "frac_of_sum_of_rooflines": sr["sum_roofline_ms"] / ms_dev,
                         "algorithmic_hbm_gb_per_step": sr["hbm_gb"], "avg_hbm_tbs": sr["hbm_gb"] / ms_dev,
                         "how": "tools/traffic_model.py: per launch max(read/5.55, write/3.88, (r+w)/6.49 TB/s, FLOP/sustained peak), summed"})
        except Exception as e:          # the model is tooling; the bench line does not depend on it
            step["sum_of_launch_rooflines_ms"] = None
            step["traffic_model_error"] = str(e)[:200]
        line = {"metric": "audio-seconds/sec forward", "value": value, "unit": "audio-s/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_dev, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": {2: "f16 tensor-core operands and activation storage (10-bit mantissa = tf32), fp32 accumulate / norm inputs / cell state",
                          1: "f32 (tf32 tensor-core operands, fp32 accumulate)", 0: "f32"}[prec], "data": "synthetic",
                "config": {"workload": f"{cfg['name']}, batch {B}/GPU", "config_key": args.config,
                           "global_batch": total_clips, "parallelism": f"batch-sharded x{world}, no collective",
                           "l2": "activations (>700 MB/step) exceed the 126 MB L2; no explicit flush",
                           "gflop_per_clip": cfg["gflop"], "gflop_per_clip_required": gflop_req,
                           "timed_path": "CUDA-graph replay (what Aero.forward does for a steady-state shape)",
                           "host_numa_cores": numa_cores},
                "ms_per_step_eager": ms_eager,
                "model_tflops": total_clips * gflop_req * 1e9 / (ms_dev * 1e-3) / 1e12,
                "e2e": {"value": e2e, "unit": "audio-s/s", "ms_per_step": ms_e2e_med, "ms_per_step_mean": ms_e2e_mean,
                        "statistic": "median of per-step device times (H2D + forward + D2H, one stream sync per step)",
                        "h2d_bytes_per_step": host_in.numel() * 4 * world, "d2h_bytes_per_step": host_out.numel() * 4 * world},
                "gpu_launches": int(launches_per_step * args.steps),
                "gpu_launches_note": f"{launches_per_step} kernels per forward x {args.steps} steps; the timed steps replay them from a "
                                     "CUDA graph (counted on the eager pass of the same steps)",
                "clocks": clk, "roofline": roof, "step": step}
        for k, v in extras.items():
            if k == "strong":
                v["value"] = v["global_batch"] * secs / (v["ms_per_step"] * 1e-3)
                v["what"] = (f"strong scaling sample: {v['global_batch']} clips in total split over {world} GPUs ({v['global_batch'] // world} per GPU); "
                             "limited by the LSTM's 200 dependent steps per window and by per-launch latency at small batch")
            else:
                v["value"] = total_clips * secs / (v["ms_per_step"] * 1e-3)
            line[k] = v
        if not args.no_cpu_baseline and world == 1:
            os.sched_setaffinity(0, range(os.cpu_count() or 1))
            threads, probes = pick_cpu_threads(args.config)
            # bounded sample of the BASELINE.md section 3 protocol (the full one -- 2 warm-ups, median of >= 5 -- is what
            # `--impl reference` runs): the workload's own batch, all physical cores, 1 warm-up, median of 3
            cb = B if args.config == "4-16" else max(1, B // 4)
            ts = _probe(args.config, threads, cb, 3, 1, 600)
            one = _probe(args.config, 1, 1, 3, 1, 120) if args.config == "4-16" else None
            line["cpu_baseline"] = {"value": (cb * secs / median(ts)) if ts else None, "unit": "audio-s/s", "cores": threads,
                                    "kind": "port",
                                    "host_cores": {"logical": os.cpu_count(), "physical": physical_cores()},
                                    "thread_probe_audio_s_per_s": {str(c): 4 * secs / t for c, t in probes.items()},
                                    "single_thread_b1": ({"value": secs / median(one), "unit": "audio-s/s", "cores": 1,
                                                          "sample": "B=1 (BASELINE configs[0]), 1 warm-up, median of 3"} if one else None),
                                    "sample": f"median of 3 forwards of {cb} clips (the GPU arm's per-GPU batch is {B}) after 1 warm-up; oracle port "
                                              f"(same torch library calls as the reference) on {threads} threads = the best of all-physical-cores / 32 / 16 (B=4 probe)"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
