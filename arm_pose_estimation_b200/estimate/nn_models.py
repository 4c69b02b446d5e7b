"""The MC-dropout LSTM regressor behind the reference's model API (``estimate/nn_models.py:160-207``, ``:373-424``).

``DropoutLSTM`` keeps the constructor, attributes, ``forward(x, hs=None)``, ``monte_carlo_predictions(n_samples, x,
hs=None)``, ``load_state_dict`` / ``state_dict`` / ``eval`` surface of the reference module, but the arithmetic is
the CUDA path of ``csrc/`` reached through the C ABI (``include/ape_b200.h``): there is no torch.nn module
underneath and no CPU fallback.  Differences a caller can see:

* dropout masks come from counter-based Philox keyed by ``(seed; stream, call index, sample, gap, t, unit)``
  instead of torch's CPU generator; ``monte_carlo_predictions(..., masks=...)`` injects explicit masks
  (time-major ``(L-1, T, n, H)``, the order torch draws them - SURVEY.md §3.2) for bit-comparable runs;
* layer 0 is evaluated once per input row, layers >= 1 once per MC sample (same results, fewer flops).
"""
import hashlib
import json
import logging
from pathlib import Path

import numpy as np
import torch

from arm_pose_estimation_b200 import _native as N
from arm_pose_estimation_b200 import config


def lstm_dims(state):
    """(I, H, L, O) from the reference's state-dict key shapes."""
    H4, I = state["lstm.weight_ih_l0"].shape
    L = sum(1 for k in state if k.startswith("lstm.weight_ih_l"))
    return int(I), int(H4) // 4, int(L), int(state["output_layer.weight"].shape[0])


def pack_lstm_weights(state):
    """Reference state dict -> the flat float32 blob of ``csrc/ape_lstm_pack.h``.

    Per layer a K-major matrix ``Wp[k][4*u + g]`` (input rows zero-padded to a multiple of 16, then the
    recurrent rows) followed by the summed bias; then ``output_layer.weight`` (O, H) and ``.bias`` (O)."""
    st = {k: np.asarray(v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else v, dtype=np.float32)
          for k, v in state.items()}
    I, H, L, O = lstm_dims(st)
    parts = []
    for l in range(L):
        w_ih, w_hh = st[f"lstm.weight_ih_l{l}"], st[f"lstm.weight_hh_l{l}"]
        kin = w_ih.shape[1]
        kin_pad = -(-kin // N.KSLICE) * N.KSLICE if l == 0 else H
        wp = np.zeros((kin_pad + H, 4 * H), np.float32)
        wp[:kin] = w_ih.reshape(4, H, kin).transpose(2, 1, 0).reshape(kin, 4 * H)
        wp[kin_pad:] = w_hh.reshape(4, H, H).transpose(2, 1, 0).reshape(H, 4 * H)
        bias = (st[f"lstm.bias_ih_l{l}"] + st[f"lstm.bias_hh_l{l}"]).reshape(4, H).T.reshape(4 * H)
        parts += [wp.ravel(), bias]
    parts += [st["output_layer.weight"].ravel(), st["output_layer.bias"].ravel()]
    return np.ascontiguousarray(np.concatenate(parts), dtype=np.float32)


def pack_lstm_weights_tc(state):
    """Reference state dict -> the fp16 blob of the tensor-core path (``csrc/ape_lstm_tc.cu``), as uint8 bytes.

    Per layer: for each CTA r of the pair, for each chunk c of 32 hidden units, the 64 gate columns  n = 64 r + nl
    of the chunk's 128 (n = 4 * u_local + g, i.e. units 16 r .. 16 r + 15 with gates i, f, g, o interleaved) as
    K-major no-swizzle tiles ``[k-group][64][8]`` halfs - first the input weights (layer 0: K zero-padded to a
    multiple of 16), then the recurrent weights; after both CTAs the bias ``b_ih + b_hh`` in column order 4u + g,
    scaled for the epilogue's ``sigmoid(x) = 0.5 + 0.5 tanh(x / 2)`` form: 0.5 b for i, f, o and b for g, so every
    tanh argument comes out of one FMA.  After all layers: ``output_layer.weight`` (first 16 rows; 32 for H = 256) as two fp16 operand tiles, rounding and remainder."""
    st = {k: np.asarray(v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else v, dtype=np.float32)
          for k, v in state.items()}
    I, H, L, O = lstm_dims(st)
    parts = []
    nl = np.arange(64)

    def tile(w, rows, kpad):
        t = np.zeros((64, kpad), np.float16)
        t[:, : w.shape[1]] = w[rows].astype(np.float16)
        return np.ascontiguousarray(t.reshape(64, kpad // 8, 8).transpose(1, 0, 2)).view(np.uint8).ravel()

    for l in range(L):
        w_ih, w_hh = st[f"lstm.weight_ih_l{l}"], st[f"lstm.weight_hh_l{l}"]
        kin_pad = -(-w_ih.shape[1] // N.KSLICE) * N.KSLICE if l == 0 else H
        for r in range(2):
            n = 64 * r + nl
            for c in range(H // 32):
                rows = (n % 4) * H + 32 * c + n // 4
                parts += [tile(w_ih, rows, kin_pad), tile(w_hh, rows, H)]
        bias = (st[f"lstm.bias_ih_l{l}"] + st[f"lstm.bias_hh_l{l}"]).reshape(4, H).T.copy()       # [u][g]
        bias[:, [0, 1, 3]] *= np.float32(0.5)
        parts.append(np.ascontiguousarray(bias.reshape(-1), dtype=np.float32).view(np.uint8))
    # output layer as a tensor-core operand (the H <= 128 kernel multiplies h_T by it, N = 32): CTA 0 holds the fp16 rounding of
    # W_o for the 16 outputs (zero rows beyond O), CTA 1 the fp16 remainder W_o - fp16(W_o) - the kernel sums the two products, so
    # W_o enters with ~22 bits; each as a K-major tile [H/8][16][8] halfs
    # (the H = 256 kernel does the same with 32 output columns per CTA)
    n_cols = 32 if H > 128 else 16
    w_full = np.zeros((n_cols, H), np.float32)
    w_full[: min(O, n_cols)] = st["output_layer.weight"][:n_cols]
    w_hi = w_full.astype(np.float16)
    w_lo = (w_full - w_hi.astype(np.float32)).astype(np.float16)
    for w in (w_hi, w_lo):
        parts.append(np.ascontiguousarray(w.reshape(n_cols, H // 8, 8).transpose(1, 0, 2)).view(np.uint8).ravel())
    # The two-layer wavefront kernel (csrc/ape_lstm_tcw.cu; H = 128, L >= 3) streams the layers >= 1 as ring pieces: per CTA and
    # chunk an x-piece [16 + 2 k-groups][64][8] and an h-piece [16][64][8].  The i, f, o columns are halved (exact in fp16 but for
    # subnormals) so the accumulator is the tanh argument of sigmoid(x) = 0.5 + 0.5 tanh(x / 2); the x-piece's extra K = 16 step
    # holds the scaled bias as an fp16 pair (rounding, remainder) in its rows 0 and 1 - the kernel multiplies it by a tile of ones.
    if H == 128 and L >= 3:
        half = np.float16(0.5)
        for l in range(1, L):
            w_ih, w_hh = st[f"lstm.weight_ih_l{l}"], st[f"lstm.weight_hh_l{l}"]
            bias = st[f"lstm.bias_ih_l{l}"] + st[f"lstm.bias_hh_l{l}"]
            for r in range(2):
                n = 64 * r + nl
                halved = (n % 4) != 2                                       # gate order i, f, g, o: all but g
                for c in range(H // 32):
                    rows = (n % 4) * H + 32 * c + n // 4
                    b_s = np.where(halved, np.float32(0.5), np.float32(1.0)) * bias[rows]
                    b_hi = b_s.astype(np.float16)
                    b_lo = (b_s - b_hi.astype(np.float32)).astype(np.float16)
                    for w, with_bias in ((w_ih, True), (w_hh, False)):
                        t = w[rows].astype(np.float16)
                        t[halved] = t[halved] * half
                        if with_bias:
                            ext = np.zeros((64, 16), np.float16)
                            ext[:, 0], ext[:, 1] = b_hi, b_lo
                            t = np.concatenate([t, ext], axis=1)
                        kp = t.shape[1]
                        parts.append(np.ascontiguousarray(t.reshape(64, kp // 8, 8).transpose(1, 0, 2)).view(np.uint8).ravel())
    return np.ascontiguousarray(np.concatenate(parts))


def pack_lstm_weights_tcx(state):
    """Reference state dict -> the blob of the SPLIT-PRECISION tensor-core kernels (``csrc/ape_lstm_tcx.cu``, H = 128, and
    ``csrc/ape_lstm_tcxs.cu``, H = 256: the same layout at either width), as uint8 bytes.

    Every weight enters as an fp16 pair ``hi = fp16(w)``, ``lo = fp16(w - hi)``; the i, f, o columns are halved first (exact), so the
    accumulator is the ex2 argument of the cell update up to one constant.  Per layer, CTA ``r`` of the pair and 32-unit chunk ``c``
    (gate columns as in ``pack_lstm_weights_tc``) four K-major tiles ``[k-group][64][8]``: ``Wx_hi`` with one extra K = 16 step whose
    rows 0 and 1 hold the scaled bias as an fp16 pair (the kernel multiplies it by a tile of ones), ``Wx_lo``, ``Wh_hi``, ``Wh_lo``.
    After all layers the output layer as in ``pack_lstm_weights_tc`` (fp16 rounding and remainder, 16 columns; 32 for H = 256)."""
    st = {k: np.asarray(v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else v, dtype=np.float32)
          for k, v in state.items()}
    I, H, L, O = lstm_dims(st)
    if H not in (128, 256):
        raise UserWarning("the split-precision tensor-core kernels take H = 128 or 256")
    parts, nl = [], np.arange(64)

    def tiles(w):                                                  # [cols, K] fp32 -> (hi, lo) K-major uint8 tiles
        hi = w.astype(np.float16)
        lo = (w - hi.astype(np.float32)).astype(np.float16)
        cols, k = w.shape
        return [np.ascontiguousarray(t.reshape(cols, k // 8, 8).transpose(1, 0, 2)).view(np.uint8).ravel() for t in (hi, lo)]

    for l in range(L):
        w_ih, w_hh = st[f"lstm.weight_ih_l{l}"], st[f"lstm.weight_hh_l{l}"]
        bias = st[f"lstm.bias_ih_l{l}"] + st[f"lstm.bias_hh_l{l}"]
        kin_pad = -(-w_ih.shape[1] // N.KSLICE) * N.KSLICE if l == 0 else H
        for r in range(2):
            n = 64 * r + nl
            scale = np.where((n % 4) != 2, np.float32(0.5), np.float32(1.0))[:, None]     # gate order i, f, g, o: all but g halved
            for c in range(H // 32):
                rows = (n % 4) * H + 32 * c + n // 4
                wx = np.zeros((64, kin_pad + 16), np.float32)
                wx[:, : w_ih.shape[1]] = w_ih[rows] * scale
                b_s = bias[rows] * scale[:, 0]
                b_hi = b_s.astype(np.float16)
                # the bias K step lives in the hi tile only: rows kin_pad (fp16(b)) and kin_pad + 1 (b - fp16(b))
                ext = np.zeros((64, kin_pad + 16), np.float16)
                ext[:, : kin_pad] = wx[:, : kin_pad].astype(np.float16)
                ext[:, kin_pad] = b_hi
                ext[:, kin_pad + 1] = (b_s - b_hi.astype(np.float32)).astype(np.float16)
                p0 = np.ascontiguousarray(ext.reshape(64, (kin_pad + 16) // 8, 8).transpose(1, 0, 2)).view(np.uint8).ravel()
                p1 = tiles(wx[:, : kin_pad])[1]
                wh_hi, wh_lo = tiles(w_hh[rows] * scale)
                parts += [p0, p1, wh_hi, wh_lo]
    n_cols = 32 if H > 128 else 16
    w_full = np.zeros((n_cols, H), np.float32)
    w_full[: min(O, n_cols)] = st["output_layer.weight"][:n_cols]
    for t in tiles(w_full):
        parts.append(t)
    return np.ascontiguousarray(np.concatenate(parts))


def packed_floats(I, H, L, O):
    """Python mirror of ``ape_pack_total_floats`` (checked against the library in tests/test_cabi.py)."""
    kin0 = -(-I // N.KSLICE) * N.KSLICE
    return (kin0 + H) * 4 * H + 4 * H + (L - 1) * (2 * H * 4 * H + 4 * H) + O * H + O


class _LstmMode:
    """Stand-in for the ``model.lstm`` sub-module: only its train / eval switch matters (nn_models.py:204)."""

    def __init__(self):
        self.training = False

    def train(self, mode=True):
        self.training = bool(mode)
        return self

    def eval(self):
        return self.train(False)


def _require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError("arm_pose_estimation_b200 needs a CUDA device (sm_100a); there is no CPU fallback")


class DropoutLSTM:
    """The reference's ``DropoutLSTM`` module surface (nn_models.py:160-207) over the CUDA path.

    ``lstm_variant``: ``"fp32"`` = the exact FFMA kernel, ``"tc"`` = the tcgen05 tensor-core kernels (fp16 operands, fp32
    accumulation and state), ``"auto"`` (default) = tensor cores when this model's shape is supported AND a probe on its own
    weights keeps the tensor-core outputs within ``tc_tolerance`` (normalised output units; 2e-4 is ~3e-5 m of hand position)
    of the fp32 kernel's.  ``"tcx"`` = the split-precision tensor-core kernels (every operand an fp16 pair, fp32-grade results at
    ~0.4 of the single-pass throughput; ``csrc/ape_lstm_tcx.cu`` for H = 128, ``csrc/ape_lstm_tcxs.cu`` for H = 256), for a model
    whose weights make the single-pass probe fail; ``"auto"`` never picks it.

    ``hs_variant`` picks the kernel of calls with a caller-supplied ``hs``: ``"fp32"`` (default), ``"tc"`` (the one-layer
    tensor-core kernels, which start every row from its (h_0, c_0)), ``"tcx"`` (the split-precision kernel, H = 256 only), or
    ``"auto"`` = ``"tc"`` when a probe with a random initial state keeps the outputs within ``tc_tolerance`` of the fp32 kernel's
    (``hs_probe_error``, ``hs_choice``), else ``"fp32"``."""

    def __init__(self, input_size, hidden_layer_size, hidden_layer_count, output_size, dropout=0.2,
                 philox_seed=None, precision="fp32", lstm_variant="auto", tc_tolerance=2e-4, hs_variant="fp32"):
        self.output_size = int(output_size)
        self.input_size = int(input_size)
        self.hidden_layer_size = int(hidden_layer_size)
        self.hidden_layer_count = int(hidden_layer_count)
        self.dropout = float(dropout)
        self.precision = precision
        if lstm_variant not in ("auto", "fp32", "tc", "tcx"):
            raise UserWarning(f"lstm_variant must be 'auto', 'fp32', 'tc' or 'tcx', got {lstm_variant!r}")
        self.lstm_variant = lstm_variant
        if hs_variant not in ("auto", "fp32", "tc", "tcx"):
            raise UserWarning(f"hs_variant must be 'auto', 'fp32', 'tc' or 'tcx', got {hs_variant!r}")
        self.hs_variant = hs_variant
        self.tc_tolerance = float(tc_tolerance)
        self.tc_probe_error = None           # max |tc - fp32| over the probe batch, once measured
        self.hs_probe_error = None           # the same for calls with hs (hs_variant="auto")
        self.hs_choice = None                # the kernel hs_variant="auto" picked: "tc" or "fp32"
        self.lstm = _LstmMode()
        self.philox_seed = int(torch.initial_seed() if philox_seed is None else philox_seed) & (2 ** 64 - 1)
        self._calls = 0                      # Philox "frame" counter: fresh masks on every call
        self._state = None
        self._blob = None                    # device copy of the packed weights (built lazily)
        self._blob_tc = None
        self._blob_tcx = None
        self._ws = None
        self._tc_ok = None                   # outcome of the probe (None: not run yet)

    # ---- torch.nn.Module-like surface ---------------------------------------------------------------
    def load_state_dict(self, state):
        I, H, L, O = lstm_dims(state)
        if (I, H, L, O) != (self.input_size, self.hidden_layer_size, self.hidden_layer_count, self.output_size):
            raise RuntimeError(f"state dict is for (I,H,L,O)={(I, H, L, O)}, model is "
                               f"{(self.input_size, self.hidden_layer_size, self.hidden_layer_count, self.output_size)}")
        self._state = {k: torch.as_tensor(np.asarray(v.detach().cpu() if isinstance(v, torch.Tensor) else v,
                                                     dtype=np.float32)) for k, v in state.items()}
        self._blob = self._blob_tc = self._blob_tcx = self._tc_ok = None
        self.hs_choice = self.hs_probe_error = None
        return self

    def state_dict(self):
        return dict(self._state)

    def eval(self):
        self.lstm.eval()
        return self

    def train(self, mode=True):
        self.lstm.train(mode)
        return self

    def packed_weights(self):
        """Device tensor holding the packed weight blob."""
        _require_cuda()
        if self._state is None:
            raise UserWarning("model has no weights: call load_state_dict first")
        if self._blob is None:
            self._blob = torch.from_numpy(pack_lstm_weights(self._state)).cuda()
        return self._blob

    def packed_weights_tc(self):
        """Device tensor holding the fp16 blob of the tensor-core kernels."""
        self.packed_weights()
        if self._blob_tc is None:
            self._blob_tc = torch.from_numpy(pack_lstm_weights_tc(self._state)).cuda()
        return self._blob_tc

    def packed_weights_tcx(self):
        """Device tensor holding the blob of the split-precision tensor-core kernels."""
        self.packed_weights()
        if self._blob_tcx is None:
            self._blob_tcx = torch.from_numpy(pack_lstm_weights_tcx(self._state)).cuda()
        return self._blob_tcx

    def _dims(self):
        return self.input_size, self.hidden_layer_size, self.hidden_layer_count, self.output_size

    def _workspace(self, T, E, n, kernel):
        I, H, L, O = self._dims()
        if kernel == "tcx":
            need = N.split_workspace_bytes(I, H, L, T, O, E, n, all_steps=True)
        else:
            need = N.workspace_bytes(I, H, L, T, O, E, n, tensor_core=kernel == "tc", all_steps=kernel == "tc")
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device="cuda")
        return self._ws

    def _tc_supported(self, T):
        I, H, L, O = self._dims()
        return N.tc_supported(I, H, L, O) and T <= 40

    def _split_kernel(self, T, hs):
        """``"tcx"`` when the split-precision kernels take this call, else ``UserWarning``."""
        I, H, L, O = self._dims()
        if not (N.split_supported(I, H, L, O) and T <= 40):
            raise UserWarning(f"the split-precision tensor-core LSTM kernels do not take (I,H,L,O)={self._dims()} with T={T}")
        if hs and H != 256:
            raise UserWarning(f"the split-precision tensor-core LSTM kernels take an initial state at H = 256 only, not H = {H}")
        return "tcx"

    def _kernel(self, T):
        """Which kernel a call without ``hs`` takes (see the class docstring): ``"fp32"``, ``"tc"`` or ``"tcx"``."""
        if self.lstm_variant == "fp32":
            return "fp32"
        if self.lstm_variant == "tcx":
            return self._split_kernel(T, False)
        if not self._tc_supported(T):
            if self.lstm_variant == "tc":
                raise UserWarning(f"the tensor-core LSTM kernels do not take (I,H,L,O)={self._dims()} with T={T}")
            return "fp32"
        if self.lstm_variant == "tc":
            return "tc"
        if self._tc_ok is None:                  # probe: N(0,1) windows, dropout active, the same Philox masks through both kernels
            g = torch.Generator(device="cpu").manual_seed(1234)
            x = torch.randn((8, T, self.input_size), generator=g, dtype=torch.float32).cuda()
            calls = self._calls
            outs = []
            for kernel in ("fp32", "tc"):
                self._calls = 0x5EED
                outs.append(self._launch(x, 16, N.MASK_PHILOX, None, None, kernel))
            self._calls = calls
            self.tc_probe_error = float((outs[0] - outs[1]).abs().max().item())
            self._tc_ok = self.tc_probe_error <= self.tc_tolerance
        return "tc" if self._tc_ok else "fp32"

    def _kernel_hs(self, T):
        """Which kernel a call with ``hs`` takes (see the class docstring): ``"fp32"``, ``"tc"`` or ``"tcx"``."""
        if self.hs_variant == "fp32":
            return "fp32"
        if self.hs_variant == "tcx":
            return self._split_kernel(T, True)
        if not self._tc_supported(T):
            if self.hs_variant == "tc":
                raise UserWarning(f"the tensor-core LSTM kernels do not take (I,H,L,O)={self._dims()} with T={T}")
            return "fp32"
        if self.hs_variant == "tc":
            return "tc"
        if self.hs_choice is None:               # probe: N(0,1) windows, N(0, 0.5^2) states, the same Philox masks through both kernels
            I, H, L, _ = self._dims()
            g = torch.Generator(device="cpu").manual_seed(1234)
            x = torch.randn((128, T, I), generator=g, dtype=torch.float32).cuda()
            hs = [(0.5 * torch.randn((L, 128, H), generator=g, dtype=torch.float32)).cuda() for _ in range(2)]
            calls = self._calls
            outs = []
            for kernel in ("fp32", "tc"):
                self._calls = 0x5EED
                outs.append(self._launch(x, 1, N.MASK_PHILOX, None, hs, kernel))
            self._calls = calls
            self.hs_probe_error = float((outs[0] - outs[1]).abs().max().item())
            self.hs_choice = "tc" if self.hs_probe_error <= self.tc_tolerance else "fp32"
        return self.hs_choice

    def _launch(self, xd, n_kernel, mask_mode, md, hs, kernel):
        """One call of the C ABI on ``kernel`` ("fp32", "tc" or "tcx"): ``xd [E, T, I]`` on the device -> ``[E, n_kernel, T, O]``."""
        I, H, L, O = self._dims()
        E, T, _ = xd.shape
        preds = torch.empty((E, n_kernel, T, O), dtype=torch.float32, device="cuda")
        a = N.LstmArgs()
        a.weights = self.packed_weights().data_ptr()
        a.weights_tc = self.packed_weights_tc().data_ptr() if kernel == "tc" else None
        if kernel == "tcx":                                  # split precision: its own blob, tc_flags = 3
            a.weights_tcx, a.tc_flags = self.packed_weights_tcx().data_ptr(), 3
        a.I, a.H, a.L, a.T, a.O = I, H, L, T, O
        a.dropout_p = self.dropout
        a.x_dense, a.feat_ring_buf, a.feat_ring = xd.data_ptr(), None, 0
        a.B, a.nF, a.frame0 = E, 1, self._calls & 0x7FFFFFFF
        a.n_samples = n_kernel
        a.mask_mode = mask_mode
        if md is not None:
            a.masks = md.data_ptr()
        if hs is not None:
            a.h0, a.c0 = hs[0].data_ptr(), hs[1].data_ptr()
        a.philox_seed, a.stream_id0 = self.philox_seed, 0
        a.workspace = self._workspace(T, E, n_kernel, kernel).data_ptr()
        a.preds, a.pred_ring, a.all_steps = preds.data_ptr(), 1, 1
        fn, what = (N.load().ape_mc_lstm_fma, "ape_mc_lstm_fma") if kernel == "fp32" else (N.load().ape_mc_lstm_tc, "ape_mc_lstm_tc")
        N.check(fn(a, N.current_stream_ptr()), what)
        return preds

    def _initial_state(self, hs, rows):
        """``hs = (h_0, c_0)``, each ``[L, rows, H]`` like torch.nn.LSTM takes them -> contiguous float32 device tensors."""
        L, H = self.hidden_layer_count, self.hidden_layer_size
        if not isinstance(hs, (tuple, list)) or len(hs) != 2:
            raise UserWarning("hs must be the pair (h_0, c_0)")
        out = []
        for name, v in zip(("h_0", "c_0"), hs):
            v = torch.as_tensor(v).detach().to(device="cuda", dtype=torch.float32).contiguous()
            if tuple(v.shape) != (L, rows, H):
                raise UserWarning(f"{name} must be [{L}, {rows}, {H}] (layers, batch, hidden), got {tuple(v.shape)}")
            out.append(v)
        return out

    def _run(self, x, n_samples, mask_mode, masks=None, hs=None):
        _require_cuda()
        if x.dim() != 3 or x.shape[2] != self.input_size:
            raise UserWarning(f"expected x of shape [batch, sequence, {self.input_size}], got {tuple(x.shape)}")
        host_in = not x.is_cuda
        xd = x.detach().to(device="cuda", dtype=torch.float32).contiguous()
        E, T, _ = xd.shape
        L, H, O = self.hidden_layer_count, self.hidden_layer_size, self.output_size
        n_kernel = 1 if L == 1 else n_samples            # no dropout in a single-layer model: samples are identical
        md = None
        if mask_mode == N.MASK_INJECTED and L > 1:
            md = torch.as_tensor(np.asarray(masks) if not isinstance(masks, torch.Tensor) else masks)
            md = md.to(device="cuda", dtype=torch.uint8).contiguous()
            if md.numel() != E * (L - 1) * T * n_kernel * H:
                raise UserWarning(f"masks must hold E*(L-1)*T*n*H = {E * (L - 1) * T * n_kernel * H} entries, got {md.numel()}")
        if hs is not None:
            # torch.nn.LSTM(x, hs) with a per-row state (nn_models.py:180-207; batch = n_samples in the MC call): every MC sample
            # becomes an estimate of its own, so layer 0 runs per row too - it no longer sees the same state for all samples
            rows = E * n_samples
            state = self._initial_state(hs, rows)
            if n_samples > 1:
                xd = xd.repeat_interleave(n_samples, dim=0)
                if md is not None:                       # [E][L-1][T][n][H] -> [E * n][L-1][T][1][H]
                    md = md.view(E, L - 1, T, n_samples, H).permute(0, 3, 1, 2, 4).contiguous()
            out = self._launch(xd, 1, mask_mode, md, state, self._kernel_hs(T)).reshape(rows, T, O)
            self._calls += 1
            return out.cpu() if host_in else out
        preds = self._launch(xd, n_kernel, mask_mode, md, None, self._kernel(T))
        self._calls += 1
        out = preds.reshape(E * n_kernel, T, O)
        if n_kernel != n_samples:
            out = out.repeat_interleave(n_samples, dim=0)
        return out.cpu() if host_in else out

    def forward(self, x, hs=None):
        """``x [batch, sequence, input] -> [batch, sequence, output]`` (nn_models.py:180-189); ``hs``: optional ``(h_0, c_0)``,
        each ``[layers, batch, hidden]``."""
        return self._run(x, 1, N.MASK_PHILOX if self.lstm.training else N.MASK_NONE, hs=hs)

    __call__ = forward

    def monte_carlo_predictions(self, n_samples, x, hs=None, masks=None):
        """``x [1, sequence, input] -> [n_samples, sequence, output]`` with dropout active (nn_models.py:191-207); ``hs``:
        optional ``(h_0, c_0)``, each ``[layers, n_samples, hidden]`` (the batch the reference's LSTM sees is the repeated input)."""
        if x.shape[0] > 1:
            raise UserWarning("MC predictions only for batch size 1")
        self.lstm.train()
        return self._run(x, n_samples, N.MASK_INJECTED if masks is not None else N.MASK_PHILOX, masks, hs)


def ff_dims(state):
    """(I, H, Lh, O) from the reference's feed-forward state-dict keys."""
    H, I = state["_input_layer.weight"].shape
    Lh = sum(1 for k in state if k.startswith("_hidden_layers.") and k.endswith(".weight"))
    return int(I), int(H), int(Lh), int(state["_output_layer.weight"].shape[0])


def pack_ff_weights(state):
    """Reference ``DropoutFF`` / ``DropoutFF2D`` state dict -> flat float32 blob of ``csrc/ape_ff.cu``: dense layers transposed
    (``W^T [K][H]`` then bias) so threads over output units read them coalesced, the output layer as is."""
    st = {k: np.asarray(v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else v, dtype=np.float32)
          for k, v in state.items()}
    I, H, Lh, O = ff_dims(st)
    parts = [st["_input_layer.weight"].T.ravel(), st["_input_layer.bias"]]
    for l in range(Lh):
        parts += [st[f"_hidden_layers.{l}.weight"].T.ravel(), st[f"_hidden_layers.{l}.bias"]]
    parts += [st["_output_layer.weight"].ravel(), st["_output_layer.bias"]]
    return np.ascontiguousarray(np.concatenate([np.ascontiguousarray(p).ravel() for p in parts]), dtype=np.float32)


class _DropoutSwitch:
    """Stand-in for the ``model._do`` dropout sub-module: only its train / eval switch matters (nn_models.py:364)."""

    def __init__(self):
        self.training = False

    def train(self, mode=True):
        self.training = bool(mode)
        return self

    def eval(self):
        return self.train(False)


class DropoutFF:
    """MC-dropout feed-forward regressor behind the reference API (``nn_models.py:313-370``): ``forward(x)``,
    ``monte_carlo_predictions(n_samples, x)``; the hidden stack runs once per input row, the output layer per sample."""

    def __init__(self, output_size, hidden_layer_size, hidden_layer_count, input_size, dropout=0.2, philox_seed=None):
        self.output_size = int(output_size)
        self.input_size = int(input_size)
        self.hidden_layer_size = int(hidden_layer_size)
        self.hidden_layer_count = int(hidden_layer_count)
        self.dropout = float(dropout)
        self._do = _DropoutSwitch()
        self.philox_seed = int(torch.initial_seed() if philox_seed is None else philox_seed) & (2 ** 64 - 1)
        self._calls = 0
        self._state = None
        self._blob = None

    def _flat_inputs(self):
        return self.input_size

    def load_state_dict(self, state):
        I, H, Lh, O = ff_dims(state)
        if (I, H, Lh, O) != (self._flat_inputs(), self.hidden_layer_size, self.hidden_layer_count, self.output_size):
            raise RuntimeError(f"state dict is for (I,H,Lh,O)={(I, H, Lh, O)}, model is "
                               f"{(self._flat_inputs(), self.hidden_layer_size, self.hidden_layer_count, self.output_size)}")
        self._state = {k: torch.as_tensor(np.asarray(v.detach().cpu() if isinstance(v, torch.Tensor) else v, dtype=np.float32))
                       for k, v in state.items()}
        self._blob = None
        return self

    def state_dict(self):
        return dict(self._state)

    def eval(self):
        self._do.eval()
        return self

    def train(self, mode=True):
        self._do.train(mode)
        return self

    def _run(self, x2d, n_samples, mask_mode, masks=None):
        _require_cuda()
        if self._state is None:
            raise UserWarning("model has no weights: call load_state_dict first")
        if self._blob is None:
            self._blob = torch.from_numpy(pack_ff_weights(self._state)).cuda()
        host_in = not x2d.is_cuda
        xd = x2d.detach().to(device="cuda", dtype=torch.float32).contiguous()
        rows = int(xd.shape[0])
        H, O = self.hidden_layer_size, self.output_size
        preds = torch.empty((rows, n_samples, O), dtype=torch.float32, device="cuda")
        md = None
        if mask_mode == N.MASK_INJECTED:
            md = torch.as_tensor(np.asarray(masks) if not isinstance(masks, torch.Tensor) else masks)
            md = md.to(device="cuda", dtype=torch.uint8).contiguous()
            if md.numel() != rows * n_samples * H:
                raise UserWarning(f"masks must hold rows*n*H = {rows * n_samples * H} entries, got {md.numel()}")
        N.check(N.load().ape_mc_ff(N.ptr(self._blob), self._flat_inputs(), H, self.hidden_layer_count, O, self.dropout,
                                   N.ptr(xd), rows, n_samples, mask_mode, N.ptr(md), self.philox_seed, 0,
                                   self._calls & 0x7FFFFFFF, N.ptr(preds), N.current_stream_ptr()), "ape_mc_ff")
        self._calls += 1
        return preds.cpu() if host_in else preds

    def _flatten(self, x):
        return x.reshape(-1, self.input_size)

    def forward(self, x):
        """``x [..., input] -> [..., output]`` (nn_models.py:338-353); dropout is active only after ``train()`` / an MC call."""
        lead = tuple(x.shape[:-1])
        out = self._run(self._flatten(x), 1, N.MASK_PHILOX if self._do.training else N.MASK_NONE)
        return out.reshape(*lead, self.output_size)

    __call__ = forward

    def monte_carlo_predictions(self, n_samples, x, masks=None):
        """``x [1, input] -> [n_samples, 1, output]`` with the output dropout active (nn_models.py:355-370)."""
        if x.shape[0] > 1:
            raise UserWarning("MC predictions only for batch size 1")
        self._do.train()
        out = self._run(self._flatten(x), n_samples, N.MASK_INJECTED if masks is not None else N.MASK_PHILOX, masks)
        return out.reshape(n_samples, 1, self.output_size)


class DropoutFF2D(DropoutFF):
    """``DropoutFF`` on the flattened ``[seq_len, input]`` window (``nn_models.py:252-310``)."""

    def __init__(self, output_size, hidden_layer_size, hidden_layer_count, input_size, seq_len, dropout=0.2, philox_seed=None):
        super().__init__(output_size, hidden_layer_size, hidden_layer_count, input_size, dropout, philox_seed)
        self.seq_len = int(seq_len)

    def _flat_inputs(self):
        return self.input_size * self.seq_len

    def _flatten(self, x):
        return x.reshape(x.shape[0], -1)

    def forward(self, x):
        out = self._run(self._flatten(x), 1, N.MASK_PHILOX if self._do.training else N.MASK_NONE)
        return out.reshape(x.shape[0], self.output_size)

    __call__ = forward

    def monte_carlo_predictions(self, n_samples, x, masks=None):
        """``x [1, seq_len, input] -> [n_samples, output]`` (nn_models.py:294-310: the repeated rows are flattened again by
        ``forward``, so the sample axis is the only leading axis)."""
        if x.shape[0] > 1:
            raise UserWarning("MC predictions only for batch size 1")
        self._do.train()
        out = self._run(self._flatten(x), n_samples, N.MASK_INJECTED if masks is not None else N.MASK_PHILOX, masks)
        return out.reshape(n_samples, self.output_size)


class ImuPoseLSTM:
    """``Linear(input, 256) + relu -> LSTM(256, 256, 2 layers) -> Linear(256, output)`` behind the reference API
    (``nn_models.py:210-249``; hidden size and depth are fixed there, the constructor keeps the unused arguments).  The input
    layer is one dense kernel (``ape_dense_act``), the rest the fp32 MC-LSTM kernel on the 256 activations.  Inter-layer
    dropout is only active in train mode; ``monte_carlo_predictions`` is a plain forward pass, like the reference's."""

    WIDTH, DEPTH = 256, 2

    def __init__(self, input_size, hidden_layer_size=None, hidden_layer_count=None, output_size=None, dropout=0.2, philox_seed=None):
        self.input_size, self.output_size = int(input_size), int(output_size)
        self._core = DropoutLSTM(self.WIDTH, self.WIDTH, self.DEPTH, self.output_size, dropout, philox_seed, lstm_variant="fp32")
        self.lstm = self._core.lstm
        self._state = None
        self._w_in = None                    # (W^T [I][256], b [256]) on the device, built lazily

    def load_state_dict(self, state):
        w = state["input_layer.weight"]
        if tuple(w.shape) != (self.WIDTH, self.input_size):
            raise RuntimeError(f"input_layer.weight is {tuple(w.shape)}, model expects {(self.WIDTH, self.input_size)}")
        self._state = {k: torch.as_tensor(np.asarray(v.detach().cpu() if isinstance(v, torch.Tensor) else v, dtype=np.float32))
                       for k, v in state.items()}
        self._core.load_state_dict({k: v for k, v in self._state.items() if not k.startswith("input_layer.")})
        self._w_in = None
        return self

    def state_dict(self):
        return dict(self._state)

    def eval(self):
        self.lstm.eval()
        return self

    def train(self, mode=True):
        self.lstm.train(mode)
        return self

    def forward(self, x, hs=None):
        """``x [batch, sequence, input] -> [batch, sequence, output]`` (nn_models.py:237-245)."""
        _require_cuda()
        if self._state is None:
            raise UserWarning("model has no weights: call load_state_dict first")
        if x.dim() != 3 or x.shape[2] != self.input_size:
            raise UserWarning(f"expected x of shape [batch, sequence, {self.input_size}], got {tuple(x.shape)}")
        if self._w_in is None:
            self._w_in = (self._state["input_layer.weight"].t().contiguous().cuda(), self._state["input_layer.bias"].contiguous().cuda())
        host_in = not x.is_cuda
        xd = x.detach().to(device="cuda", dtype=torch.float32).contiguous()
        E, T, _ = xd.shape
        act = torch.empty((E, T, self.WIDTH), dtype=torch.float32, device="cuda")
        N.check(N.load().ape_dense_act(N.ptr(self._w_in[0]), N.ptr(self._w_in[1]), N.ptr(xd), N.ptr(act), E * T, self.input_size,
                                       self.WIDTH, 1, N.current_stream_ptr()), "ape_dense_act")
        out = self._core.forward(act, hs)
        return out.cpu() if host_in else out

    __call__ = forward

    def monte_carlo_predictions(self, n_samples, x, masks=None):
        """The reference's model has no MC dropout path: a regular forward pass (nn_models.py:247-252)."""
        return self(x, None)

    # what the estimators read from any model they load (estimate/estimator.py)
    @property
    def dropout(self):
        return self._core.dropout

    @property
    def philox_seed(self):
        return self._core.philox_seed

    @philox_seed.setter
    def philox_seed(self, seed):
        self._core.philox_seed = int(seed) & (2 ** 64 - 1)


# results.json "model" names -> classes behind the same constructor keywords (nn_models.py:392-399)
_MODEL_CLASSES = {"DropoutLSTM": DropoutLSTM, "DropoutFF": DropoutFF, "ImuPoseLSTM": ImuPoseLSTM}


def _deploy_files(hash_str):
    """``(results.json, checkpoint.pt)`` of a deployed model directory; a missing file is a ``UserWarning`` like the reference's."""
    folder = Path(config.PATHS["deploy"]) / "nn" / hash_str
    files = {"json": folder / "results.json", "checkpoint": folder / "checkpoint.pt"}
    for kind, path in files.items():
        if not path.exists():
            raise UserWarning(f"no {kind} found {path}")
    return files["json"], files["checkpoint"]


def load_deployed_model_from_hash(hash_str: str):
    """``(model, params)`` of the deployed model ``<deploy>/nn/<hash_str>`` - what nn_models.py:373-415 returns: the parameter
    dictionary of ``results.json`` with ``params["model"]`` replaced by the class, and an instance of that class in eval mode
    holding the weights of ``checkpoint.pt`` (the ``(model_state, optimizer_state)`` pair the training code saved)."""
    json_path, checkpoint_path = _deploy_files(hash_str)
    params = json.loads(json_path.read_text())
    try:
        cls = _MODEL_CLASSES[params["model"]]
    except KeyError:
        raise UserWarning(f"{params['model']} not handled") from None
    params["model"] = cls
    model = cls(input_size=len(params["x_inputs_v"]), output_size=len(params["y_targets_v"]),
                **{k: params[k] for k in ("hidden_layer_size", "hidden_layer_count", "dropout")})
    weights = torch.load(checkpoint_path, map_location="cpu")[0]
    model.load_state_dict(weights).eval()
    logging.info("loaded model in eval mode from %s", json_path.parent)
    return model, params


def get_nn_name(params):
    """Directory name of a model: SHA-1 hex digest of ``str(params)`` (nn_models.py:418-424)."""
    return hashlib.sha1(str(params).encode("utf-8")).hexdigest()
