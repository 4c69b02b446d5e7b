"""The MC-dropout feed-forward regressor (DropoutFF2D) on the batched estimation path, per estimator kind: a synthetic model of
T x I inputs, H = 256, Lh = 2 and seeded weights (uarm 6 x 38 -> 12, watch-only 8 x 20 -> 12, pocket 6 x 22 -> 14).

  * throughput: estimates per second at 1024 streams x 100 MC samples, device-resident (``step_device`` back to back, one
    synchronise at the end) and end to end with host rows (``submit`` with up to N_SLOTS - 1 calls outstanding, ``result``);
  * single-stream latency: p50 / p99 of one ``step_graph`` frame (1 stream x 100 samples, host clock around the synchronised replay);
  * stage 2: kernel time of ``ape_mc_ff_ring`` (windows read from the feature ring, predictions into the prediction ring) against
    ``ape_mc_ff`` on the same windows gathered in advance, the two alternating in the same run (CUDA events around ``reps``
    launches each), as a share of the fp32 FMA peak measured in the same run (``ape_selftest_ffma_peak``) with the algorithmic flops
    computed below from the shapes;
  * the GPU name and power limit, read in the same run.

    python tools/ff_batched_bench.py [--out profiles/ff_batched_bench.json] [--rounds 5]

The stage-2 working set (weights + 1024 windows) fits in L2, as it does in the estimator, so both kernels read it from there after
the first pass.
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
from arm_pose_estimation_b200.estimate import nn_models  # noqa: E402
from arm_pose_estimation_b200.estimate.batched import BatchedEstimator  # noqa: E402

KINDS = {"uarm": syn.KIND_UARM, "watch_only": syn.KIND_WATCH_ONLY, "pocket": syn.KIND_POCKET}
H, LH, NS, B_THROUGHPUT = 256, 2, 100, 1024


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in q.split(",")]
    except Exception as e:                                       # (reported, not hidden)
        info["power_limit"] = f"unavailable: {e}"
    return info


def ffma_peak():
    import ctypes
    scratch = torch.zeros(1024, dtype=torch.float32, device="cuda")
    tf = ctypes.c_float(0.0)
    N.check(N.load().ape_selftest_ffma_peak(N.ptr(scratch), 4096, 5, ctypes.byref(tf), N.current_stream_ptr()), "ape_selftest_ffma_peak")
    return float(tf.value)


def stage2_flops(I_in, O, E, n):
    """Multiply-adds x 2 of one stage-2 call: the hidden stack once per row, the output layer once per (row, sample)."""
    return 2.0 * E * (I_in * H + LH * H * H) + 2.0 * E * n * H * O


def model(kind):
    spec = syn.kind_spec(kind)
    state = syn.synth_ff_state_dict(spec["T"] * spec["I"], H, LH, spec["O"], seed=4242 + kind)
    return spec, state


def make(kind, B, nF=1):
    spec, state = model(kind)
    be = BatchedEstimator(kind=kind, layout=spec["layout"], state=state, seq_len=spec["T"], y_targets=spec["y_targets"],
                          stats=spec["stats"], n_streams=B, mc_samples=NS, smooth=1, dropout=spec["p"], frames_per_call=nF,
                          mask_mode=N.MASK_PHILOX, philox_seed=7)
    assert be.ff and be.T == spec["T"] and be.lstm_variant == "fp32" and be._pipe is None
    return be


def throughput(kind, rounds, steps=200, warmup=10):
    be = make(kind, B_THROUGHPUT)
    rows = syn.synth_rows(kind, B_THROUGHPUT, 8, config_id=1)
    raw = [torch.from_numpy(rows[:, f:f + 1].copy()).cuda() for f in range(8)]
    dev, e2e = [], []
    for _ in range(rounds):
        for k in range(warmup):
            be.step_device(raw[k % 8])
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for k in range(steps):
            be.step_device(raw[k % 8])
        torch.cuda.synchronize()
        dev.append(B_THROUGHPUT * steps / (time.perf_counter() - t0))
        pend = []
        for k in range(warmup):
            be.submit(rows[:, k % 8]).result()
        t0 = time.perf_counter()
        for k in range(steps):
            pend.append(be.submit(rows[:, k % 8]))
            if len(pend) >= be.N_SLOTS - 1:
                pend.pop(0).result()
        for p in pend:
            p.result()
        e2e.append(B_THROUGHPUT * steps / (time.perf_counter() - t0))
    return {"streams": B_THROUGHPUT, "mc_samples": NS, "steps_per_round": steps,
            "device_resident_est_per_s": {"median": float(np.median(dev)), "all": dev},
            "end_to_end_est_per_s": {"median": float(np.median(e2e)), "all": e2e, "outstanding_calls": be.N_SLOTS - 1},
            "launches_per_call": be.launches // max(1, be.calls)}


def latency(kind, frames=400, warmup=20):
    be = make(kind, 1)
    rows = syn.synth_rows(kind, 1, 16, config_id=2)
    for k in range(warmup):
        be.step_graph(rows[:, k % 16])
    ts = []
    for k in range(frames):
        t0 = time.perf_counter()
        be.step_graph(rows[:, k % 16])
        ts.append((time.perf_counter() - t0) * 1e3)
    return {"streams": 1, "mc_samples": NS, "frames": frames, "p50_ms": float(np.percentile(ts, 50)),
            "p99_ms": float(np.percentile(ts, 99))}


def stage2(kind, peak, rounds, reps=50):
    """ape_mc_ff_ring on the estimator's rings against ape_mc_ff on the same windows gathered in advance; bitwise check of the two."""
    spec, state = model(kind)
    I, T, O, B, E = spec["I"], spec["T"], spec["O"], B_THROUGHPUT, B_THROUGHPUT
    lib = N.load()
    blob = torch.from_numpy(nn_models.pack_ff_weights(state)).cuda()
    frame0, feat_ring = 37, T
    rng = np.random.default_rng(kind)
    feats_h = rng.normal(0, 1, (B, feat_ring, I)).astype(np.float32)
    feats = torch.from_numpy(feats_h).cuda()
    win = np.stack([np.concatenate([feats_h[b, (frame0 - T + 1 + t) % feat_ring] for t in range(T)]) for b in range(B)])
    x = torch.from_numpy(win).cuda()
    ring_preds = torch.empty((B, 1, NS, O), dtype=torch.float32, device="cuda")
    flat_preds = torch.empty((E, NS, O), dtype=torch.float32, device="cuda")
    st = N.current_stream_ptr()

    def ring():
        N.check(lib.ape_mc_ff_ring(N.ptr(blob), I, T, H, LH, O, spec["p"], N.ptr(feats), feat_ring, B, 1, frame0, None, NS,
                                   N.MASK_NONE, None, 7, 0, N.ptr(ring_preds), 1, st), "ape_mc_ff_ring")

    def flat():
        N.check(lib.ape_mc_ff(N.ptr(blob), I * T, H, LH, O, spec["p"], N.ptr(x), E, NS, N.MASK_NONE, None, 7, 0, frame0,
                              N.ptr(flat_preds), st), "ape_mc_ff")

    ring(), flat()
    torch.cuda.synchronize()
    identical = bool(torch.equal(ring_preds[:, 0].view(torch.int32), flat_preds.view(torch.int32)))

    def timed(fn):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        b.synchronize()
        return a.elapsed_time(b) / reps

    for _ in range(3):                                       # warm-up of both shapes
        timed(ring), timed(flat)
    # (the mask mode does not change the hidden stack; Philox adds the key generation per (row, sample, octet))
    res = {}
    for mode_name, mode in (("none", N.MASK_NONE), ("philox", N.MASK_PHILOX)):
        def ring_m():
            N.check(lib.ape_mc_ff_ring(N.ptr(blob), I, T, H, LH, O, spec["p"], N.ptr(feats), feat_ring, B, 1, frame0, None, NS,
                                       mode, None, 7, 0, N.ptr(ring_preds), 1, st), "ape_mc_ff_ring")

        def flat_m():
            N.check(lib.ape_mc_ff(N.ptr(blob), I * T, H, LH, O, spec["p"], N.ptr(x), E, NS, mode, None, 7, 0, frame0,
                                  N.ptr(flat_preds), st), "ape_mc_ff")
        tr, tf = [], []
        for _ in range(rounds):                              # the two kernels alternate
            tr.append(timed(ring_m))
            tf.append(timed(flat_m))
        flops = stage2_flops(I * T, O, E, NS)
        mr, mf = float(np.median(tr)), float(np.median(tf))
        res[mode_name] = {
            "ape_mc_ff_ring_ms": {"median": mr, "all": tr},
            "ape_mc_ff_gathered_ms": {"median": mf, "all": tf},
            "ring_over_gathered": mr / mf,
            "ape_mc_ff_ring_frac_of_ffma_peak": flops / (mr * 1e-3) / 1e12 / peak,
            "ape_mc_ff_gathered_frac_of_ffma_peak": flops / (mf * 1e-3) / 1e12 / peak,
        }
    return {"rows": E, "mc_samples": NS, "inputs": I * T, "H": H, "Lh": LH, "O": O, "reps_per_timing": reps,
            "flops_per_call": stage2_flops(I * T, O, E, NS), "ring_equals_gathered_bitwise_mask_none": identical, **res}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--kind", nargs="+", default=list(KINDS), choices=list(KINDS))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ff_batched_bench.py needs a CUDA device")
    torch.cuda.set_device(0)
    peak = ffma_peak()
    out = {"gpu": gpu_info(), "ffma_peak_tflops": peak,
           "ffma_peak_source": "measured in this run: ape_selftest_ffma_peak (unrolled register-only FFMA microkernel, best of 5)",
           "flops_formula": "2 E (T I H + Lh H^2) + 2 E n H O (hidden stack per row, output layer per row and sample)",
           "kinds": {}}
    for name in args.kind:
        kind = KINDS[name]
        spec = syn.kind_spec(kind)
        out["kinds"][name] = {"model": f"DropoutFF2D {spec['T']} x {spec['I']} = {spec['T'] * spec['I']} inputs, H {H}, Lh {LH}, O {spec['O']}",
                              "stage2": stage2(kind, peak, args.rounds), "throughput": throughput(kind, args.rounds),
                              "latency_step_graph": latency(kind)}
        print(name, json.dumps(out["kinds"][name]["stage2"]["philox"]["ring_over_gathered"]), flush=True)
    out["gpu_after"] = gpu_info()
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(text + "\n")


if __name__ == "__main__":
    main()
