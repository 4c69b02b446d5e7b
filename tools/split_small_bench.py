"""Real-time latency of a split-precision model (weights x4 + forget-gate bias: the single-pass probe fails) on the split-precision
small-batch kernel (tc_flags = 5) against the split layer kernels (tc_flags = 3), with the single-pass cluster kernel on the unscaled
weights (tc_flags = 4) as the floor.  --kind uarm (I38 H128 L3 T6, the default): csrc/ape_lstm_tcxl.cu; --kind pocket (I22 H256 L2 T6)
and / or watch_only (I20 H256 L2 T8): csrc/ape_lstm_tcxsl.cu (ape_mc_lstm_tcxsl), with the number of its 16-CTA clusters the device
holds at once.

  * workloads: 1, 4 and 16 streams x 100 MC samples, one frame per call, Philox masks;
  * per eager call (``step``: H2D of the rows, three stages, D2H of the results, host clock around a synchronised call) and per
    ``step_graph`` frame (one CUDA-graph replay), p50 and p99; the LSTM stage's device time (the library's layer_ms events);
  * the variants alternate inside every round, every shape is warmed up first;
  * crossover against the split layer kernels from 128 to 8192 rows (n = 128): one call at a time (device events around the call) and
    back to back;
  * the outputs of the two split paths are compared bitwise in the same run; the GPU name, power limit and maximum SM clock are read
    in the same run.

    python tools/split_small_bench.py [--kind uarm | pocket watch_only] [--out profiles/split_small_bench.json] [--rounds 3]

The bitwise comparison and the latencies run the new kernel on every shape listed, above the estimator's row bound too (this tool
measures the kernels, not the routing).
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from arm_pose_estimation_b200 import _native as N, synthetic as syn  # noqa: E402
from arm_pose_estimation_b200.estimate.batched import BatchedEstimator  # noqa: E402

NS = 100
KINDS = {"uarm": syn.KIND_UARM, "pocket": syn.KIND_POCKET, "watch_only": syn.KIND_WATCH_ONLY}
KIND = syn.KIND_UARM               # the model being measured (main() sets it per --kind)
VARIANTS = {                       # name: (scaled weights, BatchedEstimator keywords, expected tc_flags)
    "split_layer_kernels": (True, dict(split_small_batch_kernel=False), 3),
    "split_small_batch_kernel": (True, dict(split_small_batch_kernel=True), 5),
    "single_pass_cluster_kernel": (False, dict(), 4),
}


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in q.split(",")]
    except Exception as e:                                       # (reported, not hidden)
        info["power_limit"] = f"unavailable: {e}"
    return info


def state_for(scaled):
    spec = syn.kind_spec(KIND)
    state = {k: v.copy() for k, v in syn.synth_state_dict(spec["I"], spec["H"], spec["L"], spec["O"], 1234 + KIND).items()}
    if scaled:
        H = spec["H"]
        for k in state:
            if k.startswith("lstm.weight_"):
                state[k] = (state[k] * np.float32(4.0)).astype(np.float32)
            if k.startswith("lstm.bias_ih_l"):
                state[k][H:2 * H] += np.float32(1.0)
    return state


def make(B, n, name):
    scaled, kw, flags = VARIANTS[name]
    spec = syn.kind_spec(KIND)
    be = BatchedEstimator(kind=KIND, layout=spec["layout"], state=state_for(scaled), seq_len=spec["T"], y_targets=spec["y_targets"],
                          stats=spec["stats"], n_streams=B, mc_samples=n, smooth=1, dropout=spec["p"], frames_per_call=1,
                          mask_mode=N.MASK_PHILOX, philox_seed=7, **kw)
    assert be.tc_flags == flags and be.tc_split == scaled, (name, be.tc_flags, be.tc_split)
    if flags == 5:
        assert be._lstm_fn() == (be.lib.ape_mc_lstm_tcxsl if be.H == 256 else be.lib.ape_mc_lstm_tc)
    return be


def pct(v):
    return {"p50_ms": float(np.percentile(v, 50)), "p99_ms": float(np.percentile(v, 99)), "n": len(v)}


def latency(rounds, calls, frames):
    out = {}
    for B in (1, 4, 16):
        rows = syn.synth_rows(KIND, B, 64, config_id=2)
        ests = {name: make(B, NS, name) for name in VARIANTS}
        eager = {name: [] for name in VARIANTS}
        graph = {name: [] for name in VARIANTS}
        lstm = {name: [] for name in VARIANTS}
        for be in ests.values():                                  # warm-up: every path at this shape, graph captured
            for f in range(10):
                be.step(rows[:, f % 64:f % 64 + 1])
                be.step_graph(rows[:, f % 64:f % 64 + 1])
        torch.cuda.synchronize()
        for _ in range(rounds):
            for name, be in ests.items():                         # alternated inside every round
                for k in range(calls):
                    r = rows[:, k % 64:k % 64 + 1]
                    t0 = time.perf_counter()
                    be.step(r)
                    eager[name].append((time.perf_counter() - t0) * 1e3)
                for k in range(frames):
                    r = rows[:, k % 64:k % 64 + 1]
                    t0 = time.perf_counter()
                    be.step_graph(r)                              # returns once the results have landed in pinned host memory
                    graph[name].append((time.perf_counter() - t0) * 1e3)
                for k in range(calls // 4):                       # the LSTM stage alone: the library's events around its one launch
                    ms = np.zeros(be.L, np.float32)
                    dev = torch.from_numpy(np.ascontiguousarray(rows[:, k % 64:k % 64 + 1])).cuda()
                    be.step_device(dev, layer_ms=ms)
                    torch.cuda.synchronize()
                    lstm[name].append(float(ms.sum()))
        out[f"{B}x{NS}"] = {name: {"eager_call": pct(eager[name]), "graph_frame": pct(graph[name]), "lstm_stage": pct(lstm[name])}
                            for name in VARIANTS}
        print(B, json.dumps(out[f"{B}x{NS}"]), flush=True)
    return out


def bitwise(calls=8):
    res = {}
    for B, n in ((1, 100), (4, 100), (16, 100), (16, 128), (64, 128)) if syn.kind_spec(KIND)["H"] == 256 else ((1, 100), (4, 100), (16, 100), (16, 128)):
        rows = syn.synth_rows(KIND, B, calls, config_id=5)
        a, b = make(B, n, "split_small_batch_kernel"), make(B, n, "split_layer_kernels")
        same = True
        for k in range(calls):
            x, y = a.step(rows[:, k:k + 1]), b.step(rows[:, k:k + 1])
            same &= bool(np.array_equal(x.msg, y.msg) and np.array_equal(x.samples, y.samples) and np.array_equal(x.std, y.std))
            x, y = a.step_graph(rows[:, k:k + 1]), b.step_graph(rows[:, k:k + 1])
            same &= bool(np.array_equal(x.msg, y.msg) and np.array_equal(x.samples, y.samples) and np.array_equal(x.std, y.std))
        res[f"{B}x{n}"] = same
    return res


def crossover():
    n, res = 128, {}
    for B in (1, 2, 4, 8, 12, 16, 24, 32, 48, 64):
        rows = syn.synth_rows(KIND, B, 64, config_id=2)
        dev = [torch.from_numpy(np.ascontiguousarray(rows[:, f:f + 1])).cuda() for f in range(64)]
        line = {}
        for name, kw in (("split_small_batch_kernel", dict(split_small_batch_kernel=True)),
                         ("split_layer_kernels", dict(split_small_batch_kernel=False, pipeline=False)),
                         ("split_layer_kernels_pipelined", dict(split_small_batch_kernel=False))):
            spec = syn.kind_spec(KIND)
            be = BatchedEstimator(kind=KIND, layout=spec["layout"], state=state_for(True), seq_len=spec["T"], y_targets=spec["y_targets"],
                                  stats=spec["stats"], n_streams=B, mc_samples=n, smooth=1, dropout=spec["p"], frames_per_call=1,
                                  mask_mode=N.MASK_PHILOX, philox_seed=7, **kw)
            assert be.tc_split and be.tc_flags == (5 if kw["split_small_batch_kernel"] else 3), (B, be.tc_flags)
            for f in range(8):
                be.step_device(dev[f], raw_ready=True)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            lat = []
            for f in range(8, 40):                                # one call at a time
                e0.record(); be.step_device(dev[f], raw_ready=True); e1.record(); e1.synchronize()
                lat.append(e0.elapsed_time(e1))
            e0.record()
            for f in range(40, 64):                               # back to back
                be.step_device(dev[f], raw_ready=True)
            e1.record(); e1.synchronize()
            line[name] = {"call_p50_ms": float(np.median(lat)), "back_to_back_ms_per_call": e0.elapsed_time(e1) / 24}
            del be
        res[B * n] = line
        print("rows", B * n, json.dumps(line), flush=True)
    return res


def measure_model(args):
    spec = syn.kind_spec(KIND)
    result = {"model": f"{syn.KIND_NAMES[KIND]} I{spec['I']} H{spec['H']} L{spec['L']} T{spec['T']} O{spec['O']}, LSTM weights x4 + "
              "forget-gate bias +1 (single-pass probe fails); floor: the same model unscaled on the single-pass cluster kernel",
              "mc_samples": NS, "masks": "Philox"}
    result["bitwise_equal_split_paths"] = bitwise()
    print("bitwise", result["bitwise_equal_split_paths"], flush=True)
    result["latency"] = latency(args.rounds, args.calls, args.frames)
    result["crossover_rows_n128"] = crossover()
    return result


def main():
    global KIND
    ap = argparse.ArgumentParser()
    ap.add_argument("--kind", nargs="+", choices=list(KINDS), default=["uarm"])
    ap.add_argument("--out", default=None, help="default: profiles/split_small_bench.json (uarm), profiles/split_small256_bench.json")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--frames", type=int, default=400)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("split_small_bench.py measures on the GPU; there is no CPU mode")
    torch.cuda.set_device(0)
    h256 = [k for k in args.kind if syn.kind_spec(KINDS[k])["H"] == 256]
    if h256 and len(h256) != len(args.kind):
        raise SystemExit("--kind: uarm (H = 128) or the H = 256 models, not both in one run")
    out = args.out or ("profiles/split_small256_bench.json" if h256 else "profiles/split_small_bench.json")
    bounds = BatchedEstimator.SMALL_BATCH_ROWS, BatchedEstimator.SPLIT256_SMALL_BATCH_ROWS
    BatchedEstimator.SMALL_BATCH_ROWS = BatchedEstimator.SPLIT256_SMALL_BATCH_ROWS = 1 << 20    # every shape on the new kernel
    if not h256:                       # (the uarm run keeps the layout of its earlier measurements)
        KIND = syn.KIND_UARM
        result = {"gpu": gpu_info(), **measure_model(args)}
        same = result["bitwise_equal_split_paths"]
    else:
        result = {"gpu": gpu_info(), "max_active_clusters": N.tcxsl_max_active_clusters(), "models": {}}
        print("max_active_clusters", result["max_active_clusters"], flush=True)
        for k in h256:
            KIND = KINDS[k]
            result["models"][k] = measure_model(args)
        same = {f"{k} {s}": v for k in h256 for s, v in result["models"][k]["bitwise_equal_split_paths"].items()}
    BatchedEstimator.SMALL_BATCH_ROWS, BatchedEstimator.SPLIT256_SMALL_BATCH_ROWS = bounds
    result["gpu_after"] = gpu_info()
    Path(out).parent.mkdir(parents=True, exist_ok=True)
    Path(out).write_text(json.dumps(result, indent=1) + "\n")
    assert all(same.values()), "the two split paths differ"
    print("wrote", out)


if __name__ == "__main__":
    main()
