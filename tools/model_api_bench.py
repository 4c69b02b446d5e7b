"""Throughput of DropoutLSTM's model API on the three deployed model shapes (dimensions read by hash, seeded weights): forward(x, hs) at 4096
rows and monte_carlo_predictions(100, x, hs) under hs_variant fp32 / tc / tcx, and forward(x) at 4096 rows under lstm_variant fp32 / tc / tcx.
Inputs and states stay on the device; each entry is CUDA events around >= 50 warmed calls, repeated --rounds times with the variants
alternated; the GPU name and power limit are read in the same run.  A variant that does not take a case (tcx with hs at H = 128) is
recorded as not supported.

    python tools/model_api_bench.py [--out profiles/model_api_split_bench.json] [--variants fp32,tc,tcx] [--calls 50] [--rounds 3]
    (profiles/model_api_bench.json: --variants fp32,tc --out profiles/model_api_bench.json)
"""
import argparse
import json
import sys
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from arm_pose_estimation_b200 import synthetic as syn  # noqa: E402
from arm_pose_estimation_b200.estimate import nn_models  # noqa: E402
from split256_bench import gpu_info  # noqa: E402

ROWS, NS = 4096, 100


def time_calls(fn, calls):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(calls):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / calls


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/model_api_split_bench.json")
    ap.add_argument("--variants", default="fp32,tc,tcx", help="comma-separated, fp32 first")
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    assert args.calls >= 50, "time at least 50 warmed calls"
    variants = tuple(args.variants.split(","))
    assert variants[0] == "fp32" and set(variants) <= {"fp32", "tc", "tcx"}, variants
    torch.cuda.set_device(0)
    result = {"gpu": gpu_info(), "calls": args.calls, "rounds": args.rounds,
              "workload": f"forward(x, hs) and forward(x) at {ROWS} rows, monte_carlo_predictions({NS}, x, hs); device-resident"}
    for kind in (syn.KIND_WATCH_ONLY, syn.KIND_POCKET, syn.KIND_UARM):
        spec = syn.kind_spec(kind)
        I, H, L, T, O = spec["I"], spec["H"], spec["L"], spec["T"], spec["O"]
        state = syn.synth_state_dict(I, H, L, O, 1234 + kind)
        models = {v: nn_models.DropoutLSTM(I, H, L, O, spec["p"], philox_seed=5, lstm_variant=v, hs_variant=v).load_state_dict(state).eval()
                  for v in variants}
        g = torch.Generator(device="cpu").manual_seed(kind)
        x = torch.randn((ROWS, T, I), generator=g).cuda()
        hs = tuple((0.5 * torch.randn((L, ROWS, H), generator=g)).cuda() for _ in range(2))
        hs_mc = tuple((0.5 * torch.randn((L, NS, H), generator=g)).cuda() for _ in range(2))
        cases = {
            "forward_hs": (ROWS, lambda m: m(x, hs)),
            "mc_hs": (NS, lambda m: m.monte_carlo_predictions(NS, x[:1], hs_mc)),
            "forward": (ROWS, lambda m: m(x)),
        }
        entry = {"model": f"seeded weights of the deployed {syn.KIND_NAMES[kind]} shape ({spec['hash'][:8]}): I{I} H{H} L{L} T{T} O{O}"}
        for case, (rows, fn) in cases.items():
            e, run = {}, []
            for v in variants:                                  # warm-up (module load, workspace, probes)
                try:
                    for _ in range(3):
                        fn(models[v])
                    run.append(v)
                except UserWarning as w:                        # e.g. tcx with hs at H = 128: no split kernel takes a state there
                    e[v] = {"not_supported": str(w)}
                models[v].eval()
            torch.cuda.synchronize()
            ms = {v: [] for v in run}
            for _ in range(args.rounds):
                for v in run:
                    ms[v].append(time_calls(lambda: fn(models[v]), args.calls))
                    models[v].eval()                            # (monte_carlo_predictions leaves the LSTM in train mode)
            for v in run:
                med = float(np.median(ms[v]))
                e[v] = {"ms_per_call_median": med, "ms_per_call_all": ms[v], "rows_per_s": rows / med * 1e3}
            line = f"{syn.KIND_NAMES[kind]} {case}: fp32 {e['fp32']['rows_per_s']:.4g} rows/s"
            for v in variants[1:]:
                if v in run:
                    e[f"{v}_over_fp32"] = e[v]["rows_per_s"] / e["fp32"]["rows_per_s"]
                    line += f", {v} {e[v]['rows_per_s']:.4g} rows/s ({e[f'{v}_over_fp32']:.2f}x)"
                else:
                    line += f", {v} not supported"
            entry[case] = e
            print(line, flush=True)
        result[syn.KIND_NAMES[kind]] = entry
        del models
        torch.cuda.empty_cache()
    result["gpu_after"] = gpu_info()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(result, indent=1) + "\n")
    print(json.dumps(result["gpu"]))


if __name__ == "__main__":
    main()
