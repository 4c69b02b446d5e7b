"""Benchmark of the per-frame arm-pose estimation hot path (BASELINE.json's metric: MC-sampled arm-pose
estimates/sec at 1/2/4/8 B200 vs the reference CPU path, and % of roofline).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Workload (configs[2] of BASELINE.json, the largest single-GPU configuration and the one the throughput metric
is quoted on): watch+phone upper-arm estimator (I38 H128 L3 T6 O12) with quaternion FK, 1024 concurrent streams
x 100 MC samples PER GPU (weak scaling: streams are sharded, no collective), synthetic IMU rows, seeded
random-init weights.  One step = one frame of every stream = 1024 estimates per GPU.

  value      estimates/s, whole job, inputs resident in HBM, CUDA events, max over ranks
  e2e        the same metric through BatchedEstimator.step() with HOST rows: pinned H2D of the raw rows and D2H
             of messages + std + per-sample positions inside the timed region, every step
  roofline   the dominant kernel (the launch that carries the LSTM layers >= 1): algorithmic flops / its device time
             (events recorded by the library around each launch, timed alone after a pause), against MEASURED_PEAKS.json
             (burst peak); `in_pipeline` = the whole step's algorithmic flops / ms_per_step
  sustained  the same step back to back for >= 2 s (the board settles at its power cap), against the SUSTAINED peak
  fp32_exact the exact fp32 FFMA kernel on the same workload, against a MEASURED fp32 FMA peak (ape_selftest_ffma_peak)
  relabel    BASELINE configs[3] (offline relabelling of recordings, watch-only model, host rows in / host messages out)
  cpu_baseline / --impl reference: the oracle's restatement of the reference CPU path (torch.nn.LSTM on the CPU +
             numpy FK, exactly the arithmetic the reference executes) timed on this box's host cores: all cores
             (one single-stream process per core) and a single process with torch's default threads.

--dump-outputs DIR writes what the last timed step of the device-resident leg returned (msg, std, samples, status of rank 0's
streams) as DIR/<name>.npy in float32: inputs, weights and Philox seed are fixed, so two builds can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

WORKLOADS = {
    # name: (kind, streams per GPU, MC samples, smooth)
    "uarm_1024x100": (2, 1024, 100, 1),
    "pocket_1x100": (1, 1, 100, 1),
    "watch_only_1024x100": (0, 1024, 100, 1),
    "pocket_1024x100": (1, 1024, 100, 1),
}
WORKLOAD_TEXT = {
    "uarm_1024x100": "watch+phone upper-arm estimator with quaternion FK, 1024 concurrent streams x 100 MC samples on 1 B200 (BASELINE configs[2])",
    "pocket_1x100": "watch+phone pocket LSTM estimator, 1 stream x 100 MC samples (BASELINE configs[1])",
    "watch_only_1024x100": "watch-only LSTM estimator (the model of BASELINE configs[0] / [3]), 1024 concurrent streams x 100 MC samples",
    "pocket_1024x100": "watch+phone pocket LSTM estimator (the model of BASELINE configs[1]), 1024 concurrent streams x 100 MC samples",
}
METRIC, UNIT = "mc_sampled_arm_pose_estimates_per_sec", "estimates/s"
DEBUG_STEPS = os.environ.get("APE_BENCH_DEBUG", "0") == "1"


def tc_kernel_name(H, pair=False):
    if pair:
        return ("lstm_pair_tcw_kernel (layers 1 + 2 of one 256-row tile as a wavefront in ONE launch; tcgen05 cta_group::2, fp16 operands, fp32 "
                "accumulate, weights streamed with cp.async.bulk, h_t in TMEM, bias added by the tensor pipe)")
    if H == 256:
        return ("lstm_layer_tcs_kernel<256> (one layer >= 1 launch; tcgen05 cta_group::2, fp16 operands, fp32 accumulate, weights streamed "
                "with cp.async.bulk, h_t in TMEM)")
    return f"lstm_layer_tc_kernel<{H}> (one layer >= 1 launch; tcgen05 cta_group::2, fp16 operands, fp32 accumulate, weights resident in shared memory)"


def ncu_traffic(kernel_key):
    """DRAM bytes per launch of a kernel from the committed `ncu --set full` capture (profiles/r2_ncu_traffic.json, written from
    the capture by tools/ncu_summary.py --traffic); None when that kernel / shape was not captured."""
    p = ROOT / "profiles" / "r2_ncu_traffic.json"
    if not p.exists():
        return None
    ent = json.loads(p.read_text()).get(kernel_key)
    if not ent:
        return None
    return {"bytes_per_launch": ent["dram_bytes_read"] + ent["dram_bytes_write"], "dram_bytes_read": ent["dram_bytes_read"],
            "dram_bytes_write": ent["dram_bytes_write"], "source": ent["source"], "shape": ent.get("shape")}


def cpu_model():
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                return ln.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def bind_rank_to_cores(local_rank, world):
    """One contiguous slice of the host cores per rank: eight Python ranks otherwise migrate over each other's cores while they
    enqueue (the 1 -> 8 curve of round 1 lost 5 % to launch jitter inside a 7 ms timed window)."""
    try:
        cores = sorted(os.sched_getaffinity(0))
        per = len(cores) // max(1, world)
        if world > 1 and per >= 1:
            os.sched_setaffinity(0, cores[local_rank * per:(local_rank + 1) * per])
            return per
    except (AttributeError, OSError):
        pass
    return None


def algorithmic_flops_per_estimate(I, H, L, T, O, n):
    """F(n) of SURVEY.md §8d: layer 0 once per estimate, layers >= 1 per MC sample, output layer on the last step."""
    return T * 2 * 4 * H * (I + H) + n * (L - 1) * T * 2 * 4 * H * (2 * H) + n * 2 * H * O


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "sm_max_mhz": 1965.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md's clocks line).  ONE poller per job
    (rank 0 samples the GPUs of every rank): a poller per rank at 20 ms was itself part of the 8-GPU launch jitter."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, indices=(0,), period_ms=25, enabled=True):
        self.indices, self.period_ms, self.enabled, self.proc, self.lines = list(indices), period_ms, enabled, None, []

    def __enter__(self):
        if not self.enabled:
            return self
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", ",".join(str(i) for i in self.indices), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", str(self.period_ms)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def __exit__(self, *exc):
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()

    def wait_first_sample(self, timeout=10.0):
        t0 = time.time()
        while self.enabled and self.proc is not None and not self.lines and time.time() - t0 < timeout:
            time.sleep(0.05)                                  # nvidia-smi start-up must not land in the timed region

    def summary(self):
        sm, smax, power, reasons = [], 0.0, 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                smax = max(smax, float(parts[1]))
                power = max(power, float(parts[2]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax or None, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": power or None, "gpus_sampled": len(self.indices)}


# ---- the reference CPU path (oracle port), used by cpu_baseline and --impl reference --------------------------------
_W = {}


def _cpu_worker_init(kind, n, smooth, threads):
    """Per-process set-up: one single-stream oracle estimator (torch CPU LSTM + numpy FK) and its synthetic rows."""
    import torch
    torch.set_num_threads(threads)
    from arm_pose_estimation_b200 import synthetic as syn
    from oracle import estimator as OE
    spec = syn.kind_spec(kind)
    state = syn.synth_state_dict(spec["I"], spec["H"], spec["L"], spec["O"], 1234 + kind)
    _W["orc"] = OE.OracleEstimator(syn.KIND_NAMES[kind], spec["lookup"], state, spec["stats"], spec["y_targets"].name,
                                   spec["T"], smooth, n, None, spec["p"], mask_source="torch")
    _W["rows"] = syn.synth_rows(kind, 1, 256, config_id=3, first_stream=os.getpid() % 1000)[0]
    _W["pos"] = 0
    for r in _W["rows"][:3]:
        _W["orc"].step(r)                                     # warm-up frames


def _cpu_worker_frames(n_frames):
    orc, rows = _W["orc"], _W["rows"]
    t0 = time.perf_counter()
    for _ in range(n_frames):
        orc.step(rows[_W["pos"] % len(rows)])                 # the three calls of estimator.py:174-176
        _W["pos"] += 1
    return n_frames, time.perf_counter() - t0


class CpuReference:
    """The reference CPU path on `workers` independent single-stream processes (the reference is single-stream by
    construction, nn_models.py:201-202): `rate(frames)` = summed estimates/s over one bounded sample."""

    def __init__(self, kind, n, smooth, workers, threads_per_worker=1):
        import multiprocessing as mp
        self.workers = workers
        self.pool = mp.get_context("spawn").Pool(workers, initializer=_cpu_worker_init,
                                                 initargs=(kind, n, smooth, threads_per_worker))

    def rate(self, frames_per_worker):
        t0 = time.perf_counter()
        res = self.pool.map(_cpu_worker_frames, [frames_per_worker] * self.workers, chunksize=1)
        wall = time.perf_counter() - t0
        return sum(f for f, _ in res) / max(dt for _, dt in res), wall

    def close(self):
        self.pool.close()
        self.pool.join()


def cpu_single_process(kind, n, smooth, frames):
    """The reference CPU estimator as its own scripts run it: ONE process, torch's default thread count (BASELINE.md §3's
    denominator of the >= 1000x target; the loop of estimator.py:174-176)."""
    import torch
    threads = torch.get_num_threads()
    ref = CpuReference(kind, n, smooth, 1, threads_per_worker=threads)
    ref.rate(3)
    rate, wall = ref.rate(frames)
    ref.close()
    return {"value": rate, "unit": UNIT, "processes": 1, "torch_threads": threads,
            "sample": f"one process, torch default threads ({threads}), {frames} frames; {wall:.1f} s of CPU work"}


def run_reference(args, rank, world):
    if rank != 0:
        return
    kind, B, n, smooth = WORKLOADS[args.workload]
    workers = max(1, min(os.cpu_count() or 1, 64))
    ref = CpuReference(kind, n, smooth, workers)
    for _ in range(args.warmup):
        ref.rate(2)
    rates, t_all = [], time.perf_counter()
    for _ in range(args.steps):
        rates.append(ref.rate(args.ref_frames)[0])
    wall = time.perf_counter() - t_all
    ref.close()
    value = float(np.mean(rates))
    sample = (f"{workers} single-stream worker processes (1 thread each) x {args.ref_frames} frames per step of the {args.workload} "
              f"workload (n={n} MC samples, smooth={smooth}); torch.nn.LSTM on CPU + numpy FK (oracle port of the reference path)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000.0 * wall / max(1, args.steps), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": args.workload, "streams_per_gpu": B, "mc_samples": n, "smooth": smooth},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": workers, "kind": "port", "sample": sample, "cpu_model": cpu_model(),
                         "single_process": cpu_single_process(kind, n, smooth, 60)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---- our arm -----------------------------------------------------------------------------------------------------------
def make_estimator(BatchedEstimator, N, syn, kind, count, n, smooth, lstm, first=0, frames_per_call=1, emit_samples=True, seed=2026):
    spec = syn.kind_spec(kind)
    state = syn.synth_state_dict(spec["I"], spec["H"], spec["L"], spec["O"], 1234 + kind)
    be = BatchedEstimator(kind=kind, layout=spec["layout"], state=state, seq_len=spec["T"], y_targets=spec["y_targets"],
                          stats=spec["stats"], n_streams=count, mc_samples=n, smooth=smooth, dropout=spec["p"],
                          frames_per_call=frames_per_call, mask_mode=N.MASK_PHILOX, philox_seed=seed, first_stream=first,
                          emit_samples=emit_samples, lstm_variant=lstm)
    return be, spec


def layer_times(be, frames, reps, L):
    """Per-launch device time of the LSTM stage (events recorded by the library around every launch), after a pause: the
    launches are timed ALONE against the burst peak, and a launch timed right behind a loaded leg measures 10-15 % longer."""
    import torch
    time.sleep(0.5)
    layer_ms, acc = np.zeros(L, np.float32), np.zeros(L, np.float64)
    for f in range(reps):
        be.step_device(frames[f % len(frames)], layer_ms=layer_ms)
        acc += layer_ms
    torch.cuda.synchronize()
    return acc / reps


def dominant_launch(be, acc, rows_mc, T, H, L):
    """(flops, ms, pair?) of the launch that carries the layers >= 1: the two-layer wavefront launch when the library pairs
    layers 1 + 2 (layer_ms then holds the pair's time in entry 1 and ~0 in entry 2), else a middle layer (L = 2: the last)."""
    per_layer = rows_mc * T * 2 * 4 * H * (2 * H)
    pair = be.lstm_variant == "tc" and L >= 3 and be._lstm_launches(be._lstm_args(1, 0, None, None)[0]) < L
    if pair:
        return 2 * per_layer, float(acc[1]), True
    return per_layer, (float(np.mean(acc[1:-1])) if L > 2 else float(acc[-1])), False


def sustained_leg(be, frames, seconds, flops_per_step, peaks, sampler_indices):
    """The step back to back for >= `seconds` (device-resident inputs): the board settles at its power cap, so this is the
    throughput a long job sees; reported against the SUSTAINED tensor peak of MEASURED_PEAKS.json with its clock record."""
    import torch
    be.reset()
    for f in range(5):
        be.step_device(frames[f % len(frames)], raw_ready=True)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    steps, t0 = 0, time.perf_counter()
    with ClockSampler(sampler_indices, period_ms=100, enabled=bool(sampler_indices)) as clk:
        clk.wait_first_sample()
        e0.record()
        while True:
            for _ in range(200):
                be.step_device(frames[steps % len(frames)], raw_ready=True)
                steps += 1
            torch.cuda.current_stream().synchronize()
            if time.perf_counter() - t0 >= seconds:
                break
        e1.record()
        torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    tf = flops_per_step * steps / (ms * 1e-3) / 1e12
    return {"value": be.B * steps / (ms * 1e-3), "unit": UNIT, "steps": steps, "seconds": ms * 1e-3, "ms_per_step": ms / steps,
            "achieved_tflops": tf, "peak": peaks.get("bf16_tflops_sustained"), "frac_of_sustained_peak": tf / peaks["bf16_tflops_sustained"]
            if peaks.get("bf16_tflops_sustained") else None, "clocks": clk.summary(),
            "note": "whole-step algorithmic flops (SURVEY.md §8d F(n)) / wall device time of a >= 2 s back-to-back run; per GPU"}


def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from arm_pose_estimation_b200 import _native as N, synthetic as syn
    from arm_pose_estimation_b200.estimate.batched import BatchedEstimator, shard_streams

    cores_per_rank = bind_rank_to_cores(local_rank, world)
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    kind, B, n, smooth = WORKLOADS[args.workload]
    first, count = shard_streams(B * world, world, rank)      # weak scaling: B streams per GPU, global stream ids
    be, spec = make_estimator(BatchedEstimator, N, syn, kind, count, n, smooth, args.lstm, first=first)
    I, H, L, T, O = (spec[k] for k in "IHLTO")
    K, W = args.steps, args.warmup
    # synthetic rows: 64 distinct seeded streams tiled over the shard (generation cost only), K+W frames
    base = syn.synth_rows(kind, min(64, count), K + W, config_id=3, first_stream=first)
    rows = np.ascontiguousarray(np.tile(base, (-(-count // base.shape[0]), 1, 1))[:count])
    rows_dev = torch.from_numpy(rows).cuda()
    frames_dev = [rows_dev[:, f:f + 1].contiguous() for f in range(K + W)]
    frames_host = [np.ascontiguousarray(rows[:, f:f + 1]) for f in range(K + W)]
    sampler_gpus = list(range(world)) if rank == 0 else []

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident throughput ("value") ----
    be.reset()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(sampler_gpus, enabled=rank == 0) as clk:
        clk.wait_first_sample()
        for f in range(W):
            be.step_device(frames_dev[f], raw_ready=True)
        barrier()
        launches0 = be.launches
        step_ev = []
        ev0.record()
        for f in range(W, W + K):
            last = be.step_device(frames_dev[f], raw_ready=True)     # inputs resident in HBM before the timed region
            if DEBUG_STEPS:
                step_ev.append(torch.cuda.Event(enable_timing=True))
                step_ev[-1].record()
        ev1.record()
        barrier()
    # (copied now: the legs below reuse the estimator's output buffers)
    dumped = last.host() if args.dump_outputs and rank == 0 else None
    if DEBUG_STEPS:                                           # APE_BENCH_DEBUG=1: completion time of every step of the timed region, per rank
        print(f"rank {rank}: total {ev0.elapsed_time(ev1):.3f} ms; step completions (ms): "
              + " ".join(f"{ev0.elapsed_time(e):.3f}" for e in step_ev), file=sys.stderr, flush=True)
    dev_ms = max_over_ranks(ev0.elapsed_time(ev1))
    launches = be.launches - launches0
    clocks = clk.summary()

    # ---- end to end through the public host-facing call ----
    # (after a pause: the leg above leaves the board at its power cap, and the two legs are to be compared under the same
    # conditions - the sustained leg below is the one that reports the power-capped state)
    time.sleep(0.5)
    be.reset()
    with ClockSampler(sampler_gpus, enabled=rank == 0) as clk_e2e:
        clk_e2e.wait_first_sample()
        for f in range(W):
            be.step(frames_host[f])
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        checksum, pending = 0.0, []
        for f in range(W, W + K):
            pending.append(be.submit(frames_host[f]))         # pinned H2D -> 3 stages -> pinned D2H, enqueued
            if len(pending) >= be.N_SLOTS - 1:                # (the estimator has N_SLOTS staging slots)
                checksum += float(pending.pop(0).result().msg[0, 0, 4])   # host read of an earlier step's result
        for p in pending:
            checksum += float(p.result().msg[0, 0, 4])
        e1.record()
        barrier()
    e2e_ms = max_over_ranks(e0.elapsed_time(e1))

    # ---- roofline leg: per-launch device time of the LSTM stage (events recorded by the library) ----
    acc = layer_times(be, frames_dev[W:], max(3, min(K, 10)), L)
    peaks, peak_src = measured_peaks()
    rows_mc = count * n
    dom_flops, dom_ms, pair = dominant_launch(be, acc, rows_mc, T, H, L)
    achieved = dom_flops / (dom_ms * 1e-3) / 1e12
    total_est = count * K * world
    tensor = be.lstm_variant == "tc"
    step_flops = count * algorithmic_flops_per_estimate(I, H, L, T, O, n)        # per GPU and step
    if tensor:
        roofline = {"bound": "tensor", "kernel": tc_kernel_name(H, pair),
                    "achieved": achieved, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s", "frac": achieved / peaks["bf16_tflops"],
                    "peak_source": f"MEASURED_PEAKS.json bf16_tflops (burst) [{peak_src}]; fp16 and bf16 tcgen05.mma run at the same rate"}
        traffic = ncu_traffic("lstm_pair_tcw_kernel" if pair else f"lstm_layer_tc{'s' if H == 256 else ''}_kernel") \
            if (count, n) == (1024, 100) else None
    else:
        roofline = {"bound": "fp32_ffma", "kernel": "lstm_layer_fma_kernel (one layer >= 1 launch)", "achieved": achieved,
                    "unit": "TFLOP/s", "frac_of_bf16_tensor_peak": achieved / peaks["bf16_tflops"]}
        roofline.update(ffma_peak_fields(N, torch, achieved))
        traffic = None
    in_pipe = step_flops / (dev_ms / K * 1e-3) / 1e12
    roofline.update({"flops_per_launch": dom_flops, "ms_per_launch": dom_ms, "layer_ms": [float(v) for v in acc],
                     "layers_per_launch": 2 if pair else 1,
                     "traffic": traffic["bytes_per_launch"] if traffic else None, "traffic_detail": traffic,
                     "in_pipeline": {"achieved": in_pipe, "frac": in_pipe / peaks["bf16_tflops"] if tensor else None,
                                     "note": "whole-step algorithmic flops F(n) x estimates / ms_per_step of the device-resident leg "
                                             "(consecutive calls overlap on two lanes, so the tail of one launch is filled by the next)"}})

    line = {
        "metric": METRIC, "value": total_est / (dev_ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": ("f16 operands, f32 accumulate/state" if tensor else "f32"), "data": "synthetic",
        "config": {"workload": args.workload, "baseline_config": WORKLOAD_TEXT[args.workload],
                   "model": {"I": I, "H": H, "L": L, "T": T, "O": O, "dropout": spec["p"]}, "streams_per_gpu": count,
                   "mc_samples": n, "smooth": smooth, "frames_per_step": 1, "estimates_per_step_per_gpu": count,
                   "lstm_variant": ("tcgen05_fp16_operands_fp32_accumulate" if tensor else "fp32_ffma"),
                   "tc_probe_error_m": be.tc_probe_error_m, "parity_tolerance_m": 1e-4, "rng": "philox4x32-10",
                   "host_path": "ape_pipeline_submit (one C call per step)" if be._pipe is not None else "python streams/events",
                   "cores_per_rank": cores_per_rank,
                   "l2": f"per-step working set ({count * n * T * H * 2 / 1e6:.0f} MB of fp16 layer-0 / inter-layer sequences, "
                         f"{2.6 * count / 1024:.1f} MB of results) is produced and consumed once per step; inputs differ every step"},
        "e2e": {"value": total_est / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": be.h2d_bytes_per_frame,
                "d2h_bytes_per_step": be.d2h_bytes_per_frame, "ms_per_step": e2e_ms / K, "clocks": clk_e2e.summary()},
        "gpu_launches": launches,
        "clocks": clocks,
        "roofline": roofline,
        "checksum": checksum,
    }
    # ---- sustained leg (every N: the 1 -> 8 curve of a long job) ----
    if not args.no_sustained:
        sus = sustained_leg(be, frames_dev, args.sustained_seconds, step_flops, peaks, sampler_gpus if rank == 0 else [])
        ms_all = max_over_ranks(sus["ms_per_step"])
        sus.update({"ms_per_step_max_over_ranks": ms_all, "value_all_gpus": count * world / (ms_all * 1e-3)})
        line["sustained"] = sus
    # ---- BASELINE configs[3]: offline relabelling, every N (recordings sharded, no collective) ----
    if not args.no_relabel:
        line["relabel"] = relabel_leg(BatchedEstimator, N, syn, torch, dist, rank, world, args.lstm, max_over_ranks, barrier)
    if rank == 0 and world == 1 and not args.no_other_models and args.workload == "uarm_1024x100":
        del be                                                # free its buffers before the other models are set up
        line["fp32_exact"] = fp32_exact_leg(BatchedEstimator, N, syn, torch, kind, B, n, smooth)
        line["tc_split"] = tc_split_leg(BatchedEstimator, N, syn, torch, kind, B, n, smooth)
        line["ff"] = ff_leg(N, torch)
        line["other_models"] = {w: quick_throughput(w, args.lstm, BatchedEstimator, N, syn, torch, sustained_seconds=0 if args.no_sustained else 2.0)
                                for w in ("watch_only_1024x100", "pocket_1024x100")}
    if rank == 0 and world == 1 and not args.no_realtime:
        line["realtime"] = realtime_latency(BatchedEstimator, N, syn)
    if rank == 0 and world == 1 and not args.no_other_models:
        line["fk_roofline"] = fk_standalone(N, syn, torch, kind, n, measured_peaks()[0])
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        workers = max(1, min(os.cpu_count() or 1, 64))
        ref = CpuReference(kind, n, smooth, workers)
        ref.rate(2)
        rate, wall = ref.rate(args.cpu_frames)
        ref.close()
        line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": workers, "kind": "port", "cpu_model": cpu_model(),
                                "sample": f"{workers} single-stream worker processes (1 thread each) x {args.cpu_frames} frames of the "
                                          f"{args.workload} workload (n={n}); torch.nn.LSTM on CPU + numpy FK; {wall:.1f} s of CPU work",
                                "single_process": cpu_single_process(kind, n, smooth, 100)}
    if dumped is not None:
        dump_outputs(Path(args.dump_outputs), dumped)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir, res):
    """The arrays of one EstimateBatch as <name>.npy, float32 (status: 0 / 1 flags)."""
    arrays = {"msg": res.msg, "std": res.std, "samples": res.samples, "status": res.status}
    assert sum(a.size * 4 for a in arrays.values()) <= 64 << 20, "outputs exceed 64 MB"
    out_dir.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(out_dir / f"{name}.npy", np.ascontiguousarray(a, dtype=np.float32))


def ffma_peak_fields(N, torch, achieved):
    """Measured fp32 FMA peak of this GPU (ape_selftest_ffma_peak: unrolled register-only FFMA microkernel, best of 5)."""
    import ctypes
    scratch = torch.zeros(1024, dtype=torch.float32, device="cuda")
    tf = ctypes.c_float(0.0)
    N.check(N.load().ape_selftest_ffma_peak(N.ptr(scratch), 4096, 5, ctypes.byref(tf), N.current_stream_ptr()), "ape_selftest_ffma_peak")
    return {"peak": float(tf.value), "frac": achieved / float(tf.value),
            "peak_source": "measured in this run: ape_selftest_ffma_peak (2 x 148 CTAs x 1024 threads, 8 independent FFMA chains per thread, "
                           "best of 5 launches); MEASURED_PEAKS.json has no fp32 figure"}


def fp32_exact_leg(BatchedEstimator, N, syn, torch, kind, B, n, smooth, steps=6):
    """The exact path: the fp32 FFMA LSTM kernel on the headline workload (what a model that fails the tensor-core precision
    probes falls back to), device-resident, with its roofline against the measured fp32 FMA peak."""
    be, spec = make_estimator(BatchedEstimator, N, syn, kind, B, n, smooth, "fp32")
    I, H, L, T, O = (spec[k] for k in "IHLTO")
    base = syn.synth_rows(kind, 64, steps + 2, config_id=3)
    rows_dev = torch.from_numpy(np.ascontiguousarray(np.tile(base, (B // 64, 1, 1)))).cuda()
    frames = [rows_dev[:, f:f + 1].contiguous() for f in range(steps + 2)]
    for f in range(2):
        be.step_device(frames[f], raw_ready=True)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for f in range(2, 2 + steps):
        be.step_device(frames[f], raw_ready=True)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    acc = layer_times(be, frames, 3, L)
    flops, dom_ms, _ = dominant_launch(be, acc, B * n, T, H, L)
    achieved = flops / (dom_ms * 1e-3) / 1e12
    out = {"value": B * steps / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / steps, "steps": steps, "lstm_variant": be.lstm_variant,
           "roofline": {"bound": "fp32_ffma", "kernel": "lstm_layer_fma_kernel (one layer >= 1 launch)", "achieved": achieved, "unit": "TFLOP/s",
                        "flops_per_launch": flops, "ms_per_launch": dom_ms, "layer_ms": [float(v) for v in acc]}}
    out["roofline"].update(ffma_peak_fields(N, torch, achieved))
    return out


def tc_split_leg(BatchedEstimator, N, syn, torch, kind, B, n, smooth, steps=40, warmup=5):
    """The split-precision tensor-core kernel (csrc/ape_lstm_tcx.cu: fp16 pairs hi + lo, three tcgen05 passes per product, ex2 / rcp
    cell update) forced on the headline workload: what `auto` runs for an H = 128 model whose weights fail the single-pass probe,
    instead of the fp32 FFMA kernel.  Device-resident and end to end; roofline = ALGORITHMIC flops of a layer >= 1 launch (the
    kernel executes three times as many) against the burst tensor peak."""
    be, spec = make_estimator(BatchedEstimator, N, syn, kind, B, n, smooth, "tcx")
    I, H, L, T, O = (spec[k] for k in "IHLTO")
    base = syn.synth_rows(kind, 64, steps + warmup, config_id=3)
    rows = np.ascontiguousarray(np.tile(base, (B // 64, 1, 1)))
    rows_dev = torch.from_numpy(rows).cuda()
    frames = [rows_dev[:, f:f + 1].contiguous() for f in range(steps + warmup)]
    time.sleep(0.5)
    for f in range(warmup):
        be.step_device(frames[f], raw_ready=True)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for f in range(warmup, warmup + steps):
        be.step_device(frames[f], raw_ready=True)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    acc = layer_times(be, frames[warmup:], 3, L)
    time.sleep(0.5)
    be.reset()
    for f in range(warmup):
        be.step(rows[:, f:f + 1])
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record()
    pending, checksum = [], 0.0
    for f in range(warmup, warmup + steps):
        pending.append(be.submit(rows[:, f:f + 1]))
        if len(pending) >= be.N_SLOTS - 1:
            checksum += float(pending.pop(0).result().msg[0, 0, 4])
    for p in pending:
        checksum += float(p.result().msg[0, 0, 4])
    g1.record()
    torch.cuda.synchronize()
    e2e_ms = g0.elapsed_time(g1)
    peaks, _ = measured_peaks()
    flops = B * n * T * 2 * 4 * H * (2 * H)
    dom_ms = float(np.mean(acc[1:]))
    achieved = flops / (dom_ms * 1e-3) / 1e12
    return {"value": B * steps / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / steps, "steps": steps,
            "lstm_variant": "tcgen05_split_precision_fp16_pairs_3_passes", "probe_error_m": be.tcx_probe_error_m,
            "e2e": {"value": B * steps / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms / steps, "checksum": checksum},
            "roofline": {"bound": "tensor", "kernel": "lstm_layer_tcx_kernel (one layer >= 1 launch)", "achieved": achieved,
                         "peak": peaks["bf16_tflops"], "unit": "TFLOP/s", "frac": achieved / peaks["bf16_tflops"],
                         "executed_frac": 3.0 * achieved / peaks["bf16_tflops"], "flops_per_launch": flops, "ms_per_launch": dom_ms,
                         "layer_ms": [float(v) for v in acc],
                         "note": "frac counts ALGORITHMIC flops (SURVEY.md §8d); the three passes per product execute 3x (+ the bias K step)"}}


def ff_leg(N, torch, rows=1024, n=100, I=110, H=128, Lh=2, O=14, reps=20):
    """The MC-dropout feed-forward regressor (DropoutFF2D of the reference, nn_models.py:317-370; SURVEY.md §8 f.2 - no deployed model uses
    it): 1024 rows (streams) x 100 MC samples per launch of `ape_mc_ff`; algorithmic flops = hidden stack once per row + the output
    layer per (row, sample), against the fp32 FMA peak measured in this run.  (8 rows per CTA: W^T streamed through shared memory once per
    CTA, thread = one (row, sample) pair in the output layer; the round-1 kernel - one CTA per row - took 0.252 ms for this launch.)"""
    import ctypes
    g = torch.Generator(device="cuda").manual_seed(5)
    floats = I * H + H + Lh * (H * H + H) + O * H + O
    blob = torch.randn(floats, generator=g, device="cuda") * 0.05
    x = torch.randn((rows, I), generator=g, device="cuda")
    preds = torch.empty((rows, n, O), device="cuda")
    lib, st = N.load(), N.current_stream_ptr()

    def run():
        N.check(lib.ape_mc_ff(N.ptr(blob), I, H, Lh, O, 0.2, N.ptr(x), rows, n, N.MASK_PHILOX, None, 7, 0, 0, N.ptr(preds), st), "ape_mc_ff")
    for _ in range(3):
        run()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        run()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    flops = rows * 2 * (I * H + Lh * H * H) + rows * n * 2 * H * O
    tf = flops / (ms * 1e-3) / 1e12
    out = {"kernel": "mc_ff_kernel", "model": {"I": I, "H": H, "hidden_layers": Lh, "O": O}, "rows": rows, "mc_samples": n, "ms_per_launch": ms,
           "value": rows / (ms * 1e-3), "unit": "rows x 100 MC samples per s", "achieved": tf, "flops_per_launch": flops}
    out.update(ffma_peak_fields(N, torch, tf))
    return out


def relabel_leg(BatchedEstimator, N, syn, torch, dist, rank, world, lstm, max_over_ranks, barrier, R=1024, F=128, fpc=4):
    """BASELINE configs[3] on a bounded sample: R synthetic recordings per GPU x F frames (the job is 10 000 recordings x 3600 frames;
    recordings are independent, so it shards by recording with no collective) through record/replay.py::relabel_recordings -
    watch-only model, 100 MC samples, HOST rows in and HOST messages + std out, every call inside the timed region."""
    from arm_pose_estimation_b200.record.replay import relabel_recordings
    kind = syn.KIND_WATCH_ONLY
    spec = syn.kind_spec(kind)
    state = syn.synth_state_dict(spec["I"], spec["H"], spec["L"], spec["O"], 1234 + kind)
    base = syn.synth_rows(kind, 16, F, config_id=4, first_stream=rank * R)
    rows = np.ascontiguousarray(np.tile(base, (-(-R // 16), 1, 1))[:R])

    built = {}

    def make(n_streams, frames_per_call):
        # the estimator (weight packing, buffers, the precision probe) is built once, by the warm-up call: the 10 000-recording job builds
        # it once per GPU for 36 M estimates, the bounded sample would otherwise charge it to 131 072
        key = (n_streams, frames_per_call)
        if key not in built:
            built[key] = BatchedEstimator(kind=kind, layout=spec["layout"], state=state, seq_len=spec["T"], y_targets=spec["y_targets"],
                                          stats=spec["stats"], n_streams=n_streams, mc_samples=100, smooth=1, dropout=spec["p"],
                                          frames_per_call=frames_per_call, mask_mode=N.MASK_PHILOX, philox_seed=4, first_stream=rank * R,
                                          emit_samples=False, lstm_variant=lstm)
        return built[key]

    relabel_recordings(rows[:, :16], make, frames_per_call=fpc)      # warm-up (allocations, probe)
    time.sleep(0.5)
    barrier()
    t0 = time.perf_counter()
    res = relabel_recordings(rows, make, frames_per_call=fpc)
    torch.cuda.synchronize()
    dt = max_over_ranks((time.perf_counter() - t0) * 1e3) * 1e-3
    est = R * F * world
    return {"workload": f"BASELINE configs[3] sample: {R} recordings per GPU x {F} frames (of 10 000 x 3600), watch-only model I20 H256 L2 T8, "
                        f"100 MC samples, {fpc} frames per call, host rows in / host messages out", "n_gpus": world,
            "estimates": est, "seconds": dt, "value": est / dt, "unit": UNIT, "scaling": "weak (recordings per GPU fixed)",
            "full_job_seconds_at_this_rate": 10000 * 3600 / (est / dt), "timing": "host wall clock of relabel_recordings() incl. the final synchronize, max over ranks (the estimator object is built by the warm-up call)",
            "finite": bool(np.isfinite(res[0]["msg"]).all())}


def fk_standalone(N, syn, torch, kind, n, peaks, E=32768, reps=20):
    """Stage 3 on its own (SURVEY.md §8d: judged separately against the HBM roofline): `ape_fk_reduce` over E estimates x n MC rows
    of random network targets - 157 MB of predictions in, messages + std + per-sample positions out, far beyond the 126 MB L2.
    Algorithmic bytes per estimate: 4 S O in + 100 (message) + 24 (std) + 24 S (sample positions)."""
    spec = syn.kind_spec(kind)
    O, tgt = spec["O"], {12: N.TARGET_ORI_CAL_LARM_UARM, 14: N.TARGET_ORI_CAL_LARM_UARM_HIPS}[spec["O"]]
    g = torch.Generator(device="cuda").manual_seed(3)
    preds = torch.randn((E, 1, n, O), generator=g, device="cuda", dtype=torch.float32)
    yy_m = torch.as_tensor(np.asarray(spec["stats"]["yy_m"], np.float32)).cuda()
    yy_s = torch.as_tensor(np.asarray(spec["stats"]["yy_s"], np.float32)).cuda()
    from arm_pose_estimation_b200.data_types.bone_map import body_measurements_row
    body = torch.as_tensor(body_measurements_row(None).astype(np.float32).ravel()).cuda()
    msg = torch.empty((E, 25), device="cuda"); std = torch.empty((E, 6), device="cuda")
    samples = torch.empty((E, n, 6), device="cuda"); status = torch.zeros(E, dtype=torch.int32, device="cuda")
    lib, st = N.load(), N.current_stream_ptr()

    def run():
        N.check(lib.ape_fk_reduce(N.ptr(preds), 1, N.ptr(yy_m), N.ptr(yy_s), N.ptr(body), tgt, O, E, 1, 0, None, n, 1,
                                  N.ptr(msg), N.ptr(samples), N.ptr(std), None, N.ptr(status), st), "ape_fk_reduce")
    for _ in range(3):
        run()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        run()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    bytes_per_est = 4 * n * O + 100 + 24 + 24 * n
    gbs = E * bytes_per_est / (ms * 1e-3) / 1e9
    return {"kernel": "fk_reduce_kernel (stage 3 standalone)", "estimates": E, "mc_rows": n, "ms_per_launch": ms,
            "bytes_per_estimate": bytes_per_est, "bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
            "frac": gbs / peaks["hbm_gbs"], "estimates_per_s": E / (ms * 1e-3),
            # DRAM bytes of one launch from the committed ncu capture (part of the 83 MB of results is still in the L2 when the kernel
            # ends); only for the captured shape
            "traffic": (lambda t: t["bytes_per_launch"] if t else None)(ncu_traffic("fk_reduce_kernel") if (E == 32768 and n == 100 and O == 12) else None),
            "traffic_detail": ncu_traffic("fk_reduce_kernel") if (E == 32768 and n == 100 and O == 12) else None,
            "l2": f"{E * bytes_per_est / 1e6:.0f} MB per launch: larger than the 126 MB L2"}


def quick_throughput(workload, lstm, BatchedEstimator, N, syn, torch, steps=50, warmup=5, sustained_seconds=2.0):
    """Device-resident throughput, end-to-end throughput, roofline of the dominant kernel and the sustained leg for the other two
    deployed models (both H = 256), same shape as the headline workload: 1024 streams x 100 MC samples, one frame per step."""
    kind, B, n, smooth = WORKLOADS[workload]
    be, spec = make_estimator(BatchedEstimator, N, syn, kind, B, n, smooth, lstm)
    I, H, L, T, O = (spec[k] for k in "IHLTO")
    base = syn.synth_rows(kind, 64, steps + warmup, config_id=3)
    rows_dev = torch.from_numpy(np.ascontiguousarray(np.tile(base, (B // 64, 1, 1)))).cuda()
    frames = [rows_dev[:, f:f + 1].contiguous() for f in range(steps + warmup)]
    time.sleep(0.5)
    for f in range(warmup):
        be.step_device(frames[f], raw_ready=True)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for f in range(warmup, warmup + steps):
        be.step_device(frames[f], raw_ready=True)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    acc = layer_times(be, frames[warmup:], 5, L)
    # end to end: host rows in (pinned H2D), host results out (pinned D2H), every step inside the timed region
    host_frames = [np.ascontiguousarray(np.tile(base[:, f:f + 1], (B // 64, 1, 1))) for f in range(steps + warmup)]
    time.sleep(0.5)
    be.reset()
    for f in range(warmup):
        be.step(host_frames[f])
    torch.cuda.synchronize()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record()
    pending, checksum = [], 0.0
    for f in range(warmup, warmup + steps):
        pending.append(be.submit(host_frames[f]))
        if len(pending) >= be.N_SLOTS - 1:
            checksum += float(pending.pop(0).result().msg[0, 0, 4])
    for p in pending:
        checksum += float(p.result().msg[0, 0, 4])
    g1.record()
    torch.cuda.synchronize()
    e2e_ms = g0.elapsed_time(g1)
    peaks, _ = measured_peaks()
    flops, dom_ms, pair = dominant_launch(be, acc, B * n, T, H, L)
    tensor = be.lstm_variant == "tc"
    achieved = flops / (dom_ms * 1e-3) / 1e12
    roof = {"bound": "tensor" if tensor else "fp32_ffma", "kernel": tc_kernel_name(H, pair) if tensor else "lstm_layer_fma_kernel",
            "achieved": achieved, "unit": "TFLOP/s", "flops_per_launch": flops, "ms_per_launch": dom_ms, "layer_ms": [float(v) for v in acc]}
    if tensor:
        roof.update({"peak": peaks["bf16_tflops"], "frac": achieved / peaks["bf16_tflops"]})
        t = ncu_traffic("lstm_layer_tcs_kernel" if H == 256 else "lstm_layer_tc_kernel") if workload == "watch_only_1024x100" else None
        roof.update({"traffic": t["bytes_per_launch"] if t else None, "traffic_detail": t})
    else:
        roof.update(ffma_peak_fields(N, torch, achieved))
    out = {"config": WORKLOAD_TEXT[workload], "model": {"I": I, "H": H, "L": L, "T": T, "O": O}, "value": B * steps / (ms * 1e-3), "unit": UNIT,
           "ms_per_step": ms / steps, "steps": steps, "lstm_variant": be.lstm_variant, "tc_probe_error_m": be.tc_probe_error_m,
           "e2e": {"value": B * steps / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms / steps, "h2d_bytes_per_step": be.h2d_bytes_per_frame,
                   "d2h_bytes_per_step": be.d2h_bytes_per_frame, "checksum": checksum},
           "roofline": roof}
    if sustained_seconds > 0:
        out["sustained"] = sustained_leg(be, frames, sustained_seconds, B * algorithmic_flops_per_estimate(I, H, L, T, O, n), peaks, [0])
    return out


def realtime_latency(BatchedEstimator, N, syn, frames=300):
    """BASELINE configs[1]: watch+phone pocket LSTM estimator, 1 stream x 100 MC samples, per-frame latency through the
    host-facing call (one 55-float row in pinned memory -> message + std + 100 sample positions back on the host)."""
    kind = syn.KIND_POCKET
    spec = syn.kind_spec(kind)
    state = syn.synth_state_dict(spec["I"], spec["H"], spec["L"], spec["O"], 1234 + kind)
    be = BatchedEstimator(kind=kind, layout=spec["layout"], state=state, seq_len=spec["T"], y_targets=spec["y_targets"],
                          stats=spec["stats"], n_streams=1, mc_samples=100, smooth=1, dropout=spec["p"], frames_per_call=1,
                          mask_mode=N.MASK_PHILOX, philox_seed=7)
    rows = syn.synth_rows(kind, 1, frames + 20, config_id=2)
    out = {"workload": "watch+phone pocket LSTM estimator (I22 H256 L2 T6 O14), 1 stream x 100 MC samples, frame by frame",
           "lstm_variant": be.lstm_variant, "frames": frames,
           "lstm_kernel": "lstm_small_kernel<256> (all layers in one launch of one 8-CTA cluster, hidden units split across it)" if be.small_batch
           else "one launch per layer on one CTA pair"}
    for key, fn, what in (("", be.step_graph, "BatchedEstimator.step_graph (one CUDA-graph launch of 4 nodes: one pinned H2D copy of frame counter + row, the 3 stages, stage 3 writing its results straight into mapped pinned host memory; then sync)"),
                          ("eager_", be.step, "BatchedEstimator.step (H2D + 3 stages + D2H enqueued call by call, then sync)")):
        be.reset()
        lat = []
        for f in range(frames + 20):
            t0 = time.perf_counter()
            fn(rows[:, f:f + 1])
            lat.append(time.perf_counter() - t0)
        lat = np.asarray(lat[20:]) * 1e3
        out.update({key + "p50_ms": float(np.percentile(lat, 50)), key + "p99_ms": float(np.percentile(lat, 99)),
                    key + "timing": "host wall clock around " + what})
    # device time of the LSTM stage alone, and the same frame through the layer kernels (one CTA pair per layer) for comparison
    import torch
    lm = np.zeros(spec["L"], np.float32)
    dev = torch.from_numpy(np.ascontiguousarray(rows[:, :1])).cuda()
    for _ in range(3):
        be.step_device(dev, layer_ms=lm)
    out["lstm_device_ms"] = float(lm.sum())
    ref = BatchedEstimator(kind=kind, layout=spec["layout"], state=state, seq_len=spec["T"], y_targets=spec["y_targets"],
                           stats=spec["stats"], n_streams=1, mc_samples=100, smooth=1, dropout=spec["p"], frames_per_call=1,
                           mask_mode=N.MASK_PHILOX, philox_seed=7, small_batch_kernel=False)
    lat = []
    for f in range(frames + 20):
        t0 = time.perf_counter()
        ref.step_graph(rows[:, f:f + 1])
        lat.append(time.perf_counter() - t0)
    out["layer_kernels_p50_ms"] = float(np.percentile(np.asarray(lat[20:]) * 1e3, 50))
    for _ in range(3):
        ref.step_device(dev, layer_ms=lm)
    out["layer_kernels_lstm_device_ms"] = float(lm.sum())
    # the multi-stream real-time front-end's tick (SURVEY.md section 8 f.3): 16 streams x 100 MC samples per graph launch - one cluster per 128 rows
    # of the call in the same launch of the small-batch kernel, against the layer kernels (one CTA pair per 256-row tile)
    ms = {}
    for key, kw in (("p50_ms", {}), ("layer_kernels_p50_ms", {"small_batch_kernel": False})):
        eng = BatchedEstimator(kind=kind, layout=spec["layout"], state=state, seq_len=spec["T"], y_targets=spec["y_targets"], stats=spec["stats"],
                               n_streams=16, mc_samples=100, smooth=1, dropout=spec["p"], frames_per_call=1, mask_mode=N.MASK_PHILOX,
                               philox_seed=7, **kw)
        rows16 = syn.synth_rows(kind, 16, 220, config_id=2)
        lat = []
        for f in range(220):
            t0 = time.perf_counter()
            eng.step_graph(rows16[:, f:f + 1])
            lat.append(time.perf_counter() - t0)
        lat = np.asarray(lat[20:]) * 1e3
        ms[key] = float(np.percentile(lat, 50))
        if not kw:
            ms["p99_ms"], ms["clusters"] = float(np.percentile(lat, 99)), (16 * 100 + 127) // 128 if eng.small_batch else 0
    out["multi_stream_16x100"] = ms
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="uarm_1024x100", choices=sorted(WORKLOADS))
    ap.add_argument("--cpu-frames", type=int, default=400, help="frames per worker of the bounded cpu_baseline sample")
    ap.add_argument("--ref-frames", type=int, default=50, help="--impl reference: frames per worker per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-realtime", action="store_true", help="skip the configs[1] single-stream latency leg")
    ap.add_argument("--no-other-models", action="store_true", help="skip the fp32 leg, the legs of the two H = 256 models and the stage-3 leg")
    ap.add_argument("--no-sustained", action="store_true", help="skip the >= 2 s back-to-back legs")
    ap.add_argument("--sustained-seconds", type=float, default=2.0)
    ap.add_argument("--no-relabel", action="store_true", help="skip the BASELINE configs[3] relabelling leg")
    ap.add_argument("--lstm", default="auto", choices=["auto", "fp32", "tc"], help="LSTM kernel variant (auto: probe-gated tensor cores)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's results as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's results: not with --impl reference")
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries the ONE JSON line and nothing else: whatever libraries write to file descriptor 1 (NCCL prints its
    # version banner there) goes to stderr instead
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(json_fd, "w")
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        if world != args.gpus and world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N > 1")
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
