"""What one skeleton per stream costs (ape_fk_reduce_bodies, BatchedEstimator's [B, 9] skeleton table).

  * stage 3 standalone, 32 768 estimates x 100 MC rows, O = 12 and O = 14, with the inputs of bench.fk_standalone: ``ape_fk_reduce``
    (one row), ``ape_fk_reduce_bodies`` with a table of 32 768 equal rows, and with 32 768 distinct rows of which one in eight has bone
    vectors off the x axis (the general rotation), alternating in the same run (CUDA events around ``reps`` launches each); the
    equal-row table is checked bit for bit against the one-row call;
  * ``BatchedEstimator`` uarm, 1024 streams x 100 MC samples: device-resident (``step_device`` back to back, one synchronise at the end)
    and end to end (``submit`` of host rows with up to N_SLOTS - 1 calls outstanding), the default skeleton against 1024 distinct ones,
    alternating;
  * with ``--parent-tree DIR`` (a built checkout of the previous commit): that tree's ``ape_fk_reduce`` in the stage-3 rounds above
    (and bit for bit against this one), and ``python bench.py`` from that tree and from this one, alternating, ``--ab-runs`` times each,
    with the outputs of the first run of each compared bit for bit;
  * the GPU name and power limit, read in the same run.

    python tools/stream_bodies_bench.py [--out profiles/stream_bodies_bench.json] [--rounds 5] [--parent-tree DIR]

The stage-3 inputs (157 MB of predictions) exceed the 126 MB L2, as in bench.fk_standalone; the 1.2 MB table does not.
"""
import argparse
import json
import os
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from arm_pose_estimation_b200 import _native as N, synthetic as syn  # noqa: E402
from arm_pose_estimation_b200.data_types.bone_map import body_measurements_row  # noqa: E402
from arm_pose_estimation_b200.estimate.batched import BatchedEstimator  # noqa: E402

E_FK, NS, B_EST = 32768, 100, 1024
BENCH_ARGS = ["--gpus", "1", "--steps", "100", "--warmup", "5", "--no-cpu-baseline", "--no-other-models", "--no-sustained",
              "--no-relabel", "--no-realtime"]


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in q.split(",")]
    except Exception as e:                                       # (reported, not hidden)
        info["power_limit"] = f"unavailable: {e}"
    return info


def distinct_rows(n, seed=5):
    """``n`` skeletons: arm lengths and shoulder origins spread around the defaults; every eighth row has bone vectors off the x axis."""
    rng = np.random.default_rng(seed)
    rows = np.repeat(body_measurements_row(), n, axis=0)
    rows[:, 0] *= rng.uniform(0.8, 1.2, n)
    rows[:, 3] *= rng.uniform(0.8, 1.2, n)
    rows[:, 6:9] += rng.uniform(-0.03, 0.03, (n, 3))
    off = np.arange(n) % 8 == 7
    rows[off, 1:3] = rng.uniform(-0.05, 0.05, (off.sum(), 2))
    rows[off, 4:6] = rng.uniform(-0.05, 0.05, (off.sum(), 2))
    return rows


def stage3(kind, rounds, reps=20, parent_lib=None):
    spec = syn.kind_spec(kind)
    O, tgt = spec["O"], {12: N.TARGET_ORI_CAL_LARM_UARM, 14: N.TARGET_ORI_CAL_LARM_UARM_HIPS}[spec["O"]]
    g = torch.Generator(device="cuda").manual_seed(3)
    preds = torch.randn((E_FK, 1, NS, O), generator=g, device="cuda", dtype=torch.float32)
    yy_m = torch.as_tensor(np.asarray(spec["stats"]["yy_m"], np.float32)).cuda()
    yy_s = torch.as_tensor(np.asarray(spec["stats"]["yy_s"], np.float32)).cuda()
    one = torch.as_tensor(body_measurements_row().astype(np.float32).ravel()).cuda()
    equal = one.repeat(E_FK, 1).contiguous()
    distinct = torch.as_tensor(distinct_rows(E_FK).astype(np.float32)).cuda()
    lib, st = N.load(), N.current_stream_ptr()
    outs = {}

    def run(which):
        o = outs.setdefault(which, dict(msg=torch.empty((E_FK, 25), device="cuda"), std=torch.empty((E_FK, 6), device="cuda"),
                                        samples=torch.empty((E_FK, NS, 6), device="cuda"),
                                        status=torch.zeros(E_FK, dtype=torch.int32, device="cuda")))
        tail = (tgt, O, E_FK, 1, 0, None, NS, 1, N.ptr(o["msg"]), N.ptr(o["samples"]), N.ptr(o["std"]), None, N.ptr(o["status"]), st)
        if which in ("fk_reduce", "parent_fk_reduce"):
            fk = lib.ape_fk_reduce if which == "fk_reduce" else parent_lib.ape_fk_reduce
            N.check(fk(N.ptr(preds), 1, N.ptr(yy_m), N.ptr(yy_s), N.ptr(one), *tail), which)
        else:
            table = equal if which == "bodies_equal" else distinct
            N.check(lib.ape_fk_reduce_bodies(N.ptr(preds), 1, N.ptr(yy_m), N.ptr(yy_s), N.ptr(table), 9, *tail), "ape_fk_reduce_bodies")

    names = ("fk_reduce", "bodies_equal", "bodies_distinct") + (("parent_fk_reduce",) if parent_lib else ())
    for name in names:
        for _ in range(3):
            run(name)
    times = {name: [] for name in names}
    for _ in range(rounds):
        for name in names:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                run(name)
            e1.record()
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1) / reps)
    same = lambda a, b: all(torch.equal(outs[a][k].view(torch.int32), outs[b][k].view(torch.int32)) for k in outs[a])
    res = {"O": O, "estimates": E_FK, "mc_rows": NS, "reps_per_round": reps,
           "equal_table_bit_identical_to_fk_reduce": same("fk_reduce", "bodies_equal")}
    if parent_lib:
        res["fk_reduce_bit_identical_to_parent"] = same("fk_reduce", "parent_fk_reduce")
    for name in names:
        res[name] = {"ms_per_launch_median": float(np.median(times[name])), "ms_per_launch_min": float(np.min(times[name])),
                     "ms_per_launch_rounds": times[name]}
    base = res["fk_reduce"]["ms_per_launch_median"]
    for name in names[1:]:
        res[name]["vs_fk_reduce"] = res[name]["ms_per_launch_median"] / base
    return res


def estimator(rounds, steps=100, warmup=10):
    kind = syn.KIND_UARM
    spec = syn.kind_spec(kind)
    state = syn.synth_state_dict(spec["I"], spec["H"], spec["L"], spec["O"], 1234 + kind)
    rows = syn.synth_rows(kind, B_EST, 8, config_id=1)
    raw = [torch.from_numpy(rows[:, f:f + 1].copy()).cuda() for f in range(8)]
    ests = {}
    for name, bms in (("default", None), ("distinct", distinct_rows(B_EST, seed=9))):
        ests[name] = BatchedEstimator(kind=kind, layout=spec["layout"], state=state, seq_len=spec["T"], y_targets=spec["y_targets"],
                                      stats=spec["stats"], n_streams=B_EST, mc_samples=NS, smooth=1, dropout=spec["p"],
                                      mask_mode=N.MASK_PHILOX, philox_seed=7, bonemaps=bms)
    res = {name: {"device_resident": [], "end_to_end": []} for name in ests}
    for name, be in ests.items():
        for f in range(warmup):
            be.step_device(raw[f % 8], raw_ready=True)
            be.step(rows[:, f % 8])
        torch.cuda.synchronize()
    for _ in range(rounds):
        for name, be in ests.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for f in range(steps):
                be.step_device(raw[f % 8], raw_ready=True)
            torch.cuda.synchronize()
            res[name]["device_resident"].append(B_EST * steps / (time.perf_counter() - t0))
            t0 = time.perf_counter()
            pend = []
            for f in range(steps):
                pend.append(be.submit(rows[:, f % 8]))
                if len(pend) >= be.N_SLOTS - 1:
                    pend.pop(0).result()
            for p in pend:
                p.result()
            res[name]["end_to_end"].append(B_EST * steps / (time.perf_counter() - t0))
    out = {"workload": f"uarm {B_EST} streams x {NS} MC samples, one frame per call", "steps_per_round": steps,
           "lstm_variant": ests["default"].lstm_variant, "native_pipeline": ests["default"]._pipe is not None, "unit": "estimates/s"}
    for name in ests:
        out[name] = {k: {"median": float(np.median(v)), "rounds": v} for k, v in res[name].items()}
    for k in ("device_resident", "end_to_end"):
        out[f"{k}_distinct_vs_default"] = out["distinct"][k]["median"] / out["default"][k]["median"]
    return out


def bench_ab(parent, runs):
    """``python bench.py`` from the parent tree and from this one, alternating; the headline and end-to-end values of each run."""
    import tempfile
    env = {k: v for k, v in os.environ.items() if k != "APE_B200_LIB"}
    res = {"args": BENCH_ARGS, "parent": [], "this": []}
    dumps = {name: tempfile.mkdtemp(prefix=f"bench_{name}_") for name in ("parent", "this")}
    for i in range(runs):
        for name, tree in (("parent", Path(parent).resolve()), ("this", ROOT)):
            extra = ["--dump-outputs", dumps[name]] if i == 0 else []       # (the first run of each: its results, compared below)
            p = subprocess.run([sys.executable, "bench.py", *BENCH_ARGS, *extra], cwd=tree, env=env, capture_output=True, text=True,
                               timeout=1800)
            if p.returncode != 0:
                raise SystemExit(f"bench.py in {name} failed:\n{p.stderr[-3000:]}")
            line = json.loads(p.stdout.strip().splitlines()[-1])
            res[name].append({"value": line["value"], "e2e": line["e2e"]["value"]})
    files = sorted(f.name for f in Path(dumps["parent"]).glob("*.npy"))
    res["outputs_bit_identical_to_parent"] = {f: bool(np.array_equal(np.load(Path(dumps["parent"]) / f).view(np.int32),
                                                                      np.load(Path(dumps["this"]) / f).view(np.int32))) for f in files}
    for name in ("parent", "this"):
        v = [r["value"] for r in res[name]]
        e = [r["e2e"] for r in res[name]]
        res[f"{name}_summary"] = {"value_median": float(np.median(v)), "value_min": float(min(v)), "value_max": float(max(v)),
                                  "e2e_median": float(np.median(e)), "e2e_min": float(min(e)), "e2e_max": float(max(e))}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "stream_bodies_bench.json"))
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--parent-tree", default=None)
    ap.add_argument("--ab-runs", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("stream_bodies_bench.py needs a CUDA device")
    out = {"gpu": gpu_info()}
    parent_lib = None
    if args.parent_tree:                     # the previous commit's stage 3 (ape_fk_reduce), timed in the same rounds
        import ctypes
        parent_lib = ctypes.CDLL(str(Path(args.parent_tree).resolve() / "arm_pose_estimation_b200" / "lib" / "libape_b200.so"))
        parent_lib.ape_fk_reduce.restype = ctypes.c_int
        parent_lib.ape_fk_reduce.argtypes = N.load().ape_fk_reduce.argtypes
    out["stage3"] = {name: stage3(kind, args.rounds, parent_lib=parent_lib)
                     for name, kind in (("O12_uarm", syn.KIND_UARM), ("O14_pocket", syn.KIND_POCKET))}
    print(json.dumps(out["stage3"], indent=1), flush=True)
    out["estimator"] = estimator(args.rounds)
    print(json.dumps(out["estimator"], indent=1), flush=True)
    if args.parent_tree:
        out["bench_ab"] = bench_ab(args.parent_tree, args.ab_runs)
        print(json.dumps(out["bench_ab"], indent=1), flush=True)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
