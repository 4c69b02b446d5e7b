"""Throughput of the H = 256 split-precision LSTM kernel (csrc/ape_lstm_tcxs.cu) against the fp32 kernel and the single-pass tensor-core
kernel, for the watch-only and pocket models at 1024 streams x 100 MC samples, device-resident (rows already on the GPU, Philox masks).
The three variants are timed alternately in one run; per-layer launch times come from the library's layer_ms events; the layer >= 1
launch is set against a bf16 matrix-product burst measured in the same run; the GPU name and power limit are read in the same run.

    python tools/split256_bench.py [--out profiles/split256_bench.json] [--steps 20] [--rounds 3]
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

B, NS = 1024, 100
VARIANTS = ("tcx", "fp32", "tc")


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in q.split(",")]
    except Exception as e:                                       # (reported, not hidden)
        info["power_limit"] = f"unavailable: {e}"
    return info


def bf16_burst_tflops(n=8192, reps=20):
    a = torch.randn((n, n), dtype=torch.bfloat16, device="cuda")
    b = torch.randn((n, n), dtype=torch.bfloat16, device="cuda")
    for _ in range(3):
        a @ b
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        a @ b
    e1.record()
    torch.cuda.synchronize()
    return 2.0 * n ** 3 * reps / (e0.elapsed_time(e1) * 1e-3) / 1e12


def make(kind, variant):
    spec = syn.kind_spec(kind)
    state = syn.synth_state_dict(spec["I"], spec["H"], spec["L"], spec["O"], 1234 + kind)
    be = BatchedEstimator(kind=kind, layout=spec["layout"], state=state, seq_len=spec["T"], y_targets=spec["y_targets"],
                          stats=spec["stats"], n_streams=B, mc_samples=NS, smooth=1, dropout=spec["p"], frames_per_call=1,
                          mask_mode=N.MASK_PHILOX, philox_seed=11, lstm_variant=variant, pipeline=False)
    want_split = variant == "tcx"
    assert be.lstm_variant == ("fp32" if variant == "fp32" else "tc") and be.tc_split == want_split, (variant, be.lstm_variant)
    return be, spec


def layer_flops(spec, layer):
    """Algorithmic flops of one layer call (2 per multiply-add of the gate products; rows = estimates for layer 0, else x samples)."""
    H, I, T = spec["H"], spec["I"], spec["T"]
    rows = B if layer == 0 else B * NS
    kin = I if layer == 0 else H
    return 2.0 * rows * T * 4 * H * (kin + H)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/split256_bench.json")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    torch.cuda.set_device(0)
    result = {"gpu": gpu_info(), "workload": f"{B} streams x {NS} MC samples, 1 frame per call, device-resident, Philox masks",
              "steps": args.steps, "rounds": args.rounds}
    peak = bf16_burst_tflops()
    result["bf16_burst_tflops"] = peak
    for kind in (syn.KIND_WATCH_ONLY, syn.KIND_POCKET):
        name = syn.KIND_NAMES[kind]
        ests = {v: make(kind, v) for v in VARIANTS}
        spec = ests["tcx"][1]
        rows = np.tile(syn.synth_rows(kind, 8, 8, config_id=6), (B // 8, 1, 1))
        dev = [torch.from_numpy(np.ascontiguousarray(rows[:, f:f + 1])).cuda() for f in range(8)]
        times = {v: [] for v in VARIANTS}
        for v in VARIANTS:                                      # warm-up of every variant
            for f in range(3):
                ests[v][0].step_device(dev[f], raw_ready=True)
        torch.cuda.synchronize()
        for _ in range(args.rounds):                            # alternated: tcx, fp32, tc, tcx, ...
            for v in VARIANTS:
                be = ests[v][0]
                steps = args.steps if v != "fp32" else max(2, args.steps // 10)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for f in range(steps):
                    be.step_device(dev[f % 8], raw_ready=True)
                e1.record()
                torch.cuda.synchronize()
                times[v].append(e0.elapsed_time(e1) / steps)
        entry = {"model": f"I{spec['I']} H{spec['H']} L{spec['L']} T{spec['T']} O{spec['O']}"}
        for v in VARIANTS:
            be = ests[v][0]
            ms = float(np.median(times[v]))
            lm = np.zeros(spec["L"], np.float32)
            torch.cuda.synchronize()
            be.step_device(dev[0], layer_ms=lm)
            torch.cuda.synchronize()
            e = {"ms_per_call_median": ms, "ms_per_call_all": times[v], "est_per_s": B / ms * 1e3, "layer_ms": [float(x) for x in lm]}
            if v != "fp32":
                fl = layer_flops(spec, 1)
                e["layer1_algorithmic_tflops"] = fl / (float(lm[1]) * 1e-3) / 1e12
                e["layer1_fraction_of_bf16_burst"] = e["layer1_algorithmic_tflops"] / peak
                if v == "tcx":                                  # the tensor pipe runs three passes per product (+ the bias K step)
                    e["layer1_tensor_pipe_fraction_of_bf16_burst"] = 3 * e["layer1_fraction_of_bf16_burst"]
            if v == "tcx":
                e["probe_error_m"] = be.tcx_probe_error_m
            entry[v] = e
        entry["split_over_fp32"] = entry["tcx"]["est_per_s"] / entry["fp32"]["est_per_s"]
        entry["split_over_single_pass"] = entry["tcx"]["est_per_s"] / entry["tc"]["est_per_s"]
        result[name] = entry
        print(f"{name}: split {entry['tcx']['est_per_s']:.4g} est/s (layer_ms {entry['tcx']['layer_ms']}), "
              f"fp32 {entry['fp32']['est_per_s']:.4g}, single pass {entry['tc']['est_per_s']:.4g}; split / fp32 = "
              f"{entry['split_over_fp32']:.2f}x", flush=True)
        del ests
        torch.cuda.empty_cache()
        time.sleep(0.2)
    result["gpu_after"] = gpu_info()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(result, indent=1) + "\n")
    print(json.dumps({k: result[k] for k in ("gpu", "bf16_burst_tflops")}))


if __name__ == "__main__":
    main()
