"""Seeded synthetic weights and IMU streams of the deployed shapes (SURVEY.md §8d).

The reference ships no ``checkpoint.pt`` (``.MISSING_LARGE_BLOBS``) and no recorded data, so benchmarks and
parity tests use weights drawn like PyTorch's default init, ``U(-1/sqrt(H), 1/sqrt(H))``, from a numpy PCG64
stream (stable across library versions, unlike ``torch.manual_seed``), and raw rows in the wire layouts of
``data_types/messaging.py`` whose feature columns follow the shipped normalisation statistics.
"""
import json
from pathlib import Path

import numpy as np

from arm_pose_estimation_b200 import config
from arm_pose_estimation_b200.data_types import messaging
from arm_pose_estimation_b200.utility import data_stats
from arm_pose_estimation_b200.utility.names import NNS_INPUTS, NNS_TARGETS

# estimator kind -> (deployed hash, wire layout id); kinds are the ids of include/ape_b200.h (APE_KIND_*)
KIND_WATCH_ONLY, KIND_POCKET, KIND_UARM = 0, 1, 2
KIND_NAMES = {KIND_WATCH_ONLY: "watch_only", KIND_POCKET: "pocket", KIND_UARM: "uarm"}
KIND_HASH = {
    KIND_WATCH_ONLY: "04f4ad63bfccb3668f7598c9375403e10b1fae2a",
    KIND_POCKET: "670b66fa7664252d1cfb3b5a8a362002ffeeba5c",
    KIND_UARM: "7cb5cdf94ef4c66388c7f15f642005d5e008146a",
}
KIND_LAYOUT = {
    KIND_WATCH_ONLY: messaging.LAYOUT_WATCH_ONLY,
    KIND_POCKET: messaging.LAYOUT_WATCH_PHONE,
    KIND_UARM: messaging.LAYOUT_WATCH_PHONE,
}


def load_params(hash_str):
    path = Path(config.PATHS["deploy"]) / "nn" / hash_str / "results.json"
    if not path.exists():
        raise UserWarning(f"no json found {path}")
    return json.loads(path.read_text())


def kind_spec(kind):
    """dict(I, H, L, T, O, p, x_inputs, y_targets, stats, lookup, ncols) of a deployed estimator kind."""
    params = load_params(KIND_HASH[kind])
    x_in, y_tg = NNS_INPUTS[params["x_inputs_n"]], NNS_TARGETS[params["y_targets_n"]]
    layout = KIND_LAYOUT[kind]
    return dict(
        kind=kind, hash=KIND_HASH[kind], params=params,
        I=len(params["x_inputs_v"]), H=params["hidden_layer_size"], L=params["hidden_layer_count"],
        T=params["sequence_len"], O=len(params["y_targets_v"]), p=params["dropout"],
        x_inputs=x_in, y_targets=y_tg, stats=data_stats.get_norm_stats(x_in, y_tg),
        layout=layout, ncols=messaging.LAYOUT_NCOLS[layout],
        lookup=messaging.WATCH_ONLY_IMU_LOOKUP if layout == messaging.LAYOUT_WATCH_ONLY else messaging.WATCH_PHONE_IMU_LOOKUP,
    )


def synth_state_dict(I, H, L, O, seed=1234):
    """Reference state-dict keys (``lstm.weight_ih_l{k}`` ..., ``output_layer.*``) with U(-1/sqrt(H), 1/sqrt(H))
    float32 numpy values, drawn in a fixed key order from ``default_rng(seed)``."""
    rng = np.random.default_rng(seed)
    k = 1.0 / np.sqrt(H)
    u = lambda *shape: rng.uniform(-k, k, size=shape).astype(np.float32)
    sd = {}
    for l in range(L):
        sd[f"lstm.weight_ih_l{l}"] = u(4 * H, I if l == 0 else H)
        sd[f"lstm.weight_hh_l{l}"] = u(4 * H, H)
        sd[f"lstm.bias_ih_l{l}"] = u(4 * H)
        sd[f"lstm.bias_hh_l{l}"] = u(4 * H)
    sd["output_layer.weight"] = u(O, H)
    sd["output_layer.bias"] = u(O)
    return sd


def synth_imu_pose_state_dict(I, O, seed=1234):
    """State dict of the reference's ``ImuPoseLSTM`` (``input_layer.*`` + a 2-layer LSTM(256, 256) + ``output_layer.*``,
    nn_models.py:223-234) with seeded numpy values like ``synth_state_dict``."""
    rng = np.random.default_rng(seed)
    k = 1.0 / np.sqrt(I)
    sd = {"input_layer.weight": rng.uniform(-k, k, size=(256, I)).astype(np.float32),
          "input_layer.bias": rng.uniform(-k, k, size=(256,)).astype(np.float32)}
    sd.update(synth_state_dict(256, 256, 2, O, seed + 1))
    return sd


def synth_ff_state_dict(I, H, Lh, O, seed=1234):
    """State dict of the reference's ``DropoutFF`` / ``DropoutFF2D`` (``_input_layer.*``, ``_hidden_layers.{k}.*``,
    ``_output_layer.*``; a ``DropoutFF2D`` of ``seq_len`` frames of ``input_size`` features has I = seq_len * input_size) with
    U(-1/sqrt(K), 1/sqrt(K)) float32 numpy values (torch's Linear init, K = the layer's inputs) drawn from ``default_rng(seed)``."""
    rng = np.random.default_rng(seed)
    u = lambda k, *shape: rng.uniform(-1 / np.sqrt(k), 1 / np.sqrt(k), size=shape).astype(np.float32)
    sd = {"_input_layer.weight": u(I, H, I), "_input_layer.bias": u(I, H)}
    for l in range(Lh):
        sd[f"_hidden_layers.{l}.weight"] = u(H, H, H)
        sd[f"_hidden_layers.{l}.bias"] = u(H, H)
    sd["_output_layer.weight"] = u(H, O, H)
    sd["_output_layer.bias"] = u(H, O)
    return sd


def write_synthetic_deploy(dst, seed=1234):
    """Create a deploy directory ``dst`` (results.json + stats of this package, plus a seeded synthetic
    ``checkpoint.pt`` per deployed hash, saved as the ``(model_state, optimizer_state)`` tuple the reference's
    loader expects, nn_models.py:410).  Returns ``dst``."""
    import shutil
    import torch
    dst = Path(dst)
    src = Path(__file__).parent / "data_deploy"
    shutil.copytree(src, dst, dirs_exist_ok=True)
    for kind, h in KIND_HASH.items():
        params = json.loads((dst / "nn" / h / "results.json").read_text())
        sd = synth_state_dict(len(params["x_inputs_v"]), params["hidden_layer_size"], params["hidden_layer_count"],
                              len(params["y_targets_v"]), seed + kind)
        torch.save(({k: torch.from_numpy(v) for k, v in sd.items()}, None), dst / "nn" / h / "checkpoint.pt")
    return dst


def _unit(q):
    return q / np.linalg.norm(q, axis=-1, keepdims=True)


def _qmul(a, b):
    aw, ax, ay, az = a[..., 0], a[..., 1], a[..., 2], a[..., 3]
    bw, bx, by, bz = b[..., 0], b[..., 1], b[..., 2], b[..., 3]
    return np.stack([aw * bw - ax * bx - ay * by - az * bz, aw * bx + ax * bw + ay * bz - az * by,
                     aw * by - ax * bz + ay * bw + az * bx, aw * bz + ax * by - ay * bx + az * bw], axis=-1)


def _quat_walk(rng, n_frames, sigma=0.05):
    """Unit-quaternion random walk: per frame multiply by a small random rotation (sigma rad)."""
    q = np.empty((n_frames, 4))
    q[0] = _unit(rng.normal(size=4))
    rv = rng.normal(scale=sigma, size=(n_frames, 3))
    ang = np.linalg.norm(rv, axis=-1, keepdims=True)
    dq = np.concatenate([np.cos(ang / 2), np.sin(ang / 2) * rv / np.maximum(ang, 1e-12)], axis=-1)
    for f in range(1, n_frames):
        q[f] = _qmul(q[f - 1], dq[f])
    return _unit(q)


def synth_rows(kind, n_streams, n_frames, config_id=0, first_stream=0):
    """Raw rows ``(n_streams, n_frames, ncols)`` float32.  Stream ``s`` uses seed ``1000*config_id + first_stream + s``
    so any shard of a job regenerates exactly its own streams."""
    spec = kind_spec(kind)
    lk, xm, xs = spec["lookup"], spec["stats"]["xx_m"], spec["stats"]["xx_s"]
    names = list(spec["x_inputs"].value)
    out = np.zeros((n_streams, n_frames, spec["ncols"]), np.float32)
    for s in range(n_streams):
        rng = np.random.default_rng(1000 * config_id + first_stream + s)
        for j, col in enumerate(names):
            if col in lk:                                     # plain sensor columns: N(mean, std) of the stats
                out[s, :, lk[col]] = rng.normal(xm[j], xs[j], size=n_frames)
        out[s, :, lk["sw_dt"]] = np.maximum(out[s, :, lk["sw_dt"]], 1e-3)
        jp = names.index("sw_pres_cal")
        out[s, :, lk["sw_init_pres"]] = 1000.0
        out[s, :, lk["sw_pres"]] = 1000.0 + rng.normal(xm[jp], xs[jp], size=n_frames)
        devs = ("sw",) if spec["layout"] == messaging.LAYOUT_WATCH_ONLY else ("sw", "ph")
        for dev in devs:
            walk, fwd = _quat_walk(rng, n_frames), _unit(rng.normal(size=4))
            for i, c in enumerate("wxyz"):
                out[s, :, lk[f"{dev}_rotvec_{c}"]] = walk[:, i]
                out[s, :, lk[f"{dev}_forward_{c}"]] = fwd[i]
    return out
