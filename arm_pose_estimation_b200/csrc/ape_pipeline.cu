// The cross-call pipeline of the batched estimation path as ONE host call per batch (ape_pipeline_*).
//
// What the reference does per frame in Python (estimator.py:174-176: parse_row_to_xx -> add_xx_to_row_hist_and_make_prediction ->
// msg_from_pred) is here a fixed sequence of enqueues per call of B streams x nF frames:
//
//     side stream (high priority):  H2D of the staged raw rows -> ape_features -> MC-LSTM layer 0       (up to three calls ahead)
//     lane stream (call & 1):       MC-LSTM layers >= 1 -> ape_fk_reduce                                  (two calls in flight)
//     copy stream:                  D2H of [messages | std | status | sample positions] into pinned memory
//
// estimate/batched.py drives the same sequence call by call through torch streams and events (it still does, for profiling legs,
// injected masks and the CUDA-graph path); at 0.3 ms of device time per call the ~40 Python-level stream / event operations of one
// submit() had become what the GPU waited for.  This object owns nothing but CUDA streams and events: every buffer is the caller's.
//
// Nothing orders the last LSTM layer of call k behind stage 3 of call k-1 (the other lane) as long as every stream's frames move
// forward: the prediction ring holds two calls' frames plus the smoothing window, so call k writes no slot call k-1 still reads.
// A stream's counter may go back (a restarted stream, a shared counter reset with calls in flight), or jump; when call k then
// writes a slot of call k-1's smoothing window (pred_window_alias), its layers >= 1 wait for call k-1's stage 3.
#include <cstring>
#include <new>

#include "ape_common.cuh"
#include "ape_b200.h"

namespace {
constexpr int MAX_SLOTS = APE_PIPELINE_MAX_SLOTS;

// Do frames f .. f + nF - 1 of a stream share a slot of a ring of `ring` frames with the smoothing windows of a call of nF1 frames
// from frame f1 (frames f1 - smooth + 1 .. f1 + nF1 - 1, those before 0 read as frame 0)?  (estimate/batched.py: the same rule)
bool pred_window_alias(long long f, int nF, long long f1, int nF1, int smooth, int ring) {
    const long long lo = f1 - smooth + 1 > 0 ? f1 - smooth + 1 : 0;           // oldest frame read
    long long o = (f - lo) % ring;                             // where the written frames start, counted from its slot
    if (o < 0) o += ring;
    return o < f1 + nF1 - lo || o + nF > ring;
}
}

struct ape_pipeline {
    ape_pipeline_desc d;
    int device;
    cudaStream_t side, lane[2], copy;
    cudaEvent_t ev_in, ev0[4], done[4], lstm_done[2], slot_ev[MAX_SLOTS];
    bool done_valid[4], lstm_done_valid, slot_busy[MAX_SLOTS];
    int last_lane;
    long long calls, submits;
    // the previous call, while its stage 3 may still be running: its frames (shared frame0, or per-stream counters in
    // frames_host[prev_slot], which the next n_slots - 1 calls leave alone)
    bool prev_valid, prev_sf;
    int prev_nF, prev_frame0, prev_slot;
};

#define PIPE_TRY(expr) do { int _rc = (expr); if (_rc != APE_OK) return _rc; } while (0)

extern "C" int ape_pipeline_create(const ape_pipeline_desc* d, ape_pipeline** out) {
    if (!d || !out) return APE_ERR_BAD_ARG;
    if (d->n_slots < 2 || d->n_slots > MAX_SLOTS || d->B < 1 || d->nF_max < 1 || d->ncols < 1 || d->smooth < 1) return APE_ERR_BAD_ARG;
    const bool split = d->lstm.tc_flags == 3;                  // the split-precision variant brings its own blob
    if (!d->raw || !d->feats || !(split ? d->lstm.weights_tcx : d->lstm.weights_tc) || !d->lstm.preds || !d->lane_workspace[0] ||
        !d->lane_workspace[1] || !d->body9)
        return APE_ERR_BAD_ARG;
    for (int s = 0; s < d->n_slots; ++s)
        if (!d->out_dev[s] || !d->raw_host[s] || !d->out_host[s]) return APE_ERR_BAD_ARG;
    if (d->lstm.mask_mode == APE_MASK_INJECTED) return APE_ERR_UNSUPPORTED;      // injected masks change per call: the caller's path
    if (!(split ? (ape_mc_lstm_tcx_supported(d->lstm.I, d->lstm.H, d->lstm.L, d->lstm.O) ||
                   ape_mc_lstm_tcxs_supported(d->lstm.I, d->lstm.H, d->lstm.L, d->lstm.O))
                : ape_mc_lstm_tc_supported(d->lstm.I, d->lstm.H, d->lstm.L, d->lstm.O))) return APE_ERR_UNSUPPORTED;
    ape_pipeline* p = new (std::nothrow) ape_pipeline();
    if (!p) return APE_ERR_BAD_ARG;
    p->d = *d;
    APE_CUDA_TRY(cudaGetDevice(&p->device));
    int lo = 0, hi = 0;
    APE_CUDA_TRY(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    // (high priority: the few dozen CTAs of stage 1 + layer 0 take the first SMs any big launch frees)
    APE_CUDA_TRY(cudaStreamCreateWithPriority(&p->side, cudaStreamNonBlocking, hi));
    for (int i = 0; i < 2; ++i) APE_CUDA_TRY(cudaStreamCreateWithFlags(&p->lane[i], cudaStreamNonBlocking));
    APE_CUDA_TRY(cudaStreamCreateWithFlags(&p->copy, cudaStreamNonBlocking));
    auto mk = [](cudaEvent_t* e) { return cudaEventCreateWithFlags(e, cudaEventDisableTiming); };
    APE_CUDA_TRY(mk(&p->ev_in));
    for (int i = 0; i < 4; ++i) { APE_CUDA_TRY(mk(&p->ev0[i])); APE_CUDA_TRY(mk(&p->done[i])); p->done_valid[i] = false; }
    for (int i = 0; i < 2; ++i) APE_CUDA_TRY(mk(&p->lstm_done[i]));
    for (int i = 0; i < MAX_SLOTS; ++i) { APE_CUDA_TRY(mk(&p->slot_ev[i])); p->slot_busy[i] = false; }
    p->lstm_done_valid = false;
    p->last_lane = 0;
    p->calls = p->submits = 0;
    p->prev_valid = false;
    *out = p;
    return APE_OK;
}

extern "C" int ape_pipeline_destroy(ape_pipeline* p) {
    if (!p) return APE_OK;
    cudaStreamSynchronize(p->side); cudaStreamSynchronize(p->lane[0]); cudaStreamSynchronize(p->lane[1]); cudaStreamSynchronize(p->copy);
    cudaEventDestroy(p->ev_in);
    for (int i = 0; i < 4; ++i) { cudaEventDestroy(p->ev0[i]); cudaEventDestroy(p->done[i]); }
    for (int i = 0; i < 2; ++i) cudaEventDestroy(p->lstm_done[i]);
    for (int i = 0; i < MAX_SLOTS; ++i) cudaEventDestroy(p->slot_ev[i]);
    cudaStreamDestroy(p->side); cudaStreamDestroy(p->lane[0]); cudaStreamDestroy(p->lane[1]); cudaStreamDestroy(p->copy);
    delete p;
    return APE_OK;
}

// host-blocking drain of everything this pipeline has enqueued (before the caller touches its buffers from another path)
extern "C" int ape_pipeline_sync(ape_pipeline* p) {
    if (!p) return APE_ERR_BAD_ARG;
    APE_CUDA_TRY(cudaStreamSynchronize(p->side));
    APE_CUDA_TRY(cudaStreamSynchronize(p->lane[0]));
    APE_CUDA_TRY(cudaStreamSynchronize(p->lane[1]));
    APE_CUDA_TRY(cudaStreamSynchronize(p->copy));
    for (int i = 0; i < MAX_SLOTS; ++i) p->slot_busy[i] = false;
    p->prev_valid = false;                                     // (everything has drained: the next call follows nothing)
    return APE_OK;
}

// the pipeline's streams, for a caller that orders its own work against one of them: 0 side, 1 lane 0, 2 lane 1, 3 copy
extern "C" int ape_pipeline_stream(ape_pipeline* p, int which, void** stream) {
    if (!p || !stream || which < 0 || which > 3) return APE_ERR_BAD_ARG;
    const cudaStream_t s[4] = {p->side, p->lane[0], p->lane[1], p->copy};
    *stream = (void*)s[which];
    return APE_OK;
}

// everything enqueued AFTER this call waits for what `stream` holds now (work the caller did on the shared buffers elsewhere)
extern "C" int ape_pipeline_fence(ape_pipeline* p, void* stream) {
    if (!p) return APE_ERR_BAD_ARG;
    APE_CUDA_TRY(cudaEventRecord(p->ev_in, (cudaStream_t)stream));
    APE_CUDA_TRY(cudaStreamWaitEvent(p->side, p->ev_in, 0));
    APE_CUDA_TRY(cudaStreamWaitEvent(p->lane[0], p->ev_in, 0));
    APE_CUDA_TRY(cudaStreamWaitEvent(p->lane[1], p->ev_in, 0));
    return APE_OK;
}

extern "C" int ape_pipeline_wait(ape_pipeline* p, int slot) {
    if (!p || slot < 0 || slot >= p->d.n_slots) return APE_ERR_BAD_ARG;
    if (p->slot_busy[slot]) { APE_CUDA_TRY(cudaEventSynchronize(p->slot_ev[slot])); p->slot_busy[slot] = false; }
    return APE_OK;
}

extern "C" int ape_pipeline_query(ape_pipeline* p, int slot, int* landed) {
    if (!p || !landed || slot < 0 || slot >= p->d.n_slots) return APE_ERR_BAD_ARG;
    *landed = 1;
    if (p->slot_busy[slot]) {
        const cudaError_t e = cudaEventQuery(p->slot_ev[slot]);
        if (e == cudaErrorNotReady) *landed = 0;
        else if (e != cudaSuccess) return ape::cuda_fail(e);
    }
    return APE_OK;
}

extern "C" int ape_pipeline_submit(ape_pipeline* p, const float* rows_host, const float* rows_dev, int nF, int frame0,
                                   const int32_t* stream_frames_host, int flags, void* caller_stream, int* slot_out) {
    if (!p || !slot_out || nF < 1 || nF > p->d.nF_max || (!rows_host == !rows_dev)) return APE_ERR_BAD_ARG;
    const ape_pipeline_desc& d = p->d;
    if (stream_frames_host && (!d.frames_dev[0] || !d.frames_host[0])) return APE_ERR_BAD_ARG;
    int dev = -1;
    APE_CUDA_TRY(cudaGetDevice(&dev));
    if (dev != p->device) return APE_ERR_BAD_ARG;
    cudaStream_t caller = (cudaStream_t)caller_stream;
    const int slot = (int)(p->submits % d.n_slots);
    const long long k = p->calls;
    const int parity = (int)(k & 1), bufset = (int)(k & 3);
    cudaStream_t side = p->side, lane = p->lane[parity];
    const size_t E = (size_t)d.B * nF, Em = (size_t)d.B * d.nF_max;

    // the slot's previous results have landed on the host: its pinned staging and its device result buffer are free
    PIPE_TRY(ape_pipeline_wait(p, slot));
    if (rows_host) std::memcpy(d.raw_host[slot], rows_host, E * d.ncols * sizeof(float));
    const int32_t* sf_dev = nullptr;
    if (stream_frames_host) {
        std::memcpy(d.frames_host[slot], stream_frames_host, (size_t)d.B * sizeof(int32_t));
        sf_dev = d.frames_dev[bufset];
    }
    if (flags & APE_PIPE_INPUT_PENDING) {                      // rows_dev is still being produced on the caller's stream
        APE_CUDA_TRY(cudaEventRecord(p->ev_in, caller));
        APE_CUDA_TRY(cudaStreamWaitEvent(side, p->ev_in, 0));
    }
    // Stage 1 only touches buffers whose other users are on this stream too (the raw rows, the feature ring), so a call without
    // per-stream frame counters copies its rows and runs stage 1 as soon as it is submitted; what has to wait for the last call
    // on this buffer set (call k-4: its copy of layer 0's output, its frame counters) is layer 0 - and the counters' copy.
    if (sf_dev && p->done_valid[bufset]) APE_CUDA_TRY(cudaStreamWaitEvent(side, p->done[bufset], 0));
    const float* raw = rows_dev;
    if (rows_host) {
        APE_CUDA_TRY(cudaMemcpyAsync(d.raw, d.raw_host[slot], E * d.ncols * sizeof(float), cudaMemcpyHostToDevice, side));
        raw = d.raw;
    }
    if (sf_dev)
        APE_CUDA_TRY(cudaMemcpyAsync((void*)sf_dev, d.frames_host[slot], (size_t)d.B * sizeof(int32_t), cudaMemcpyHostToDevice, side));
    const int f0 = sf_dev ? 0 : frame0;
    PIPE_TRY(ape_features(raw, d.layout, d.kind, d.xx_m, d.xx_s, d.normalize, d.feats, d.B, nF, f0, sf_dev, d.feat_ring, side));
    if (!sf_dev && p->done_valid[bufset]) APE_CUDA_TRY(cudaStreamWaitEvent(side, p->done[bufset], 0));
    ape_lstm_args a = d.lstm;
    a.nF = nF; a.frame0 = f0; a.stream_frames = sf_dev;
    a.workspace = d.lane_workspace[parity];
    a.layer_ms = nullptr; a.trace = nullptr;
    a.layer_begin = 0; a.layer_end = 1; a.ws_parity = bufset >> 1;
    PIPE_TRY(ape_mc_lstm_tc(&a, side));
    APE_CUDA_TRY(cudaEventRecord(p->ev0[bufset], side));

    APE_CUDA_TRY(cudaStreamWaitEvent(lane, p->ev0[bufset], 0));
    // a stream whose counter went back (or jumped) may write a prediction slot that stage 3 of call k-1 (the other lane) still reads;
    // call k-2 ran on this lane, so only call k-1 needs the check.  A change between the shared and the per-stream counters fences too.
    if (p->prev_valid) {
        const int ring = d.lstm.pred_ring;
        bool alias = p->prev_sf != (sf_dev != nullptr);
        if (!alias && !sf_dev) {
            alias = pred_window_alias(frame0, nF, p->prev_frame0, p->prev_nF, d.smooth, ring);
        } else if (!alias) {
            const int32_t* prev = d.frames_host[p->prev_slot];
            for (int b = 0; b < d.B && !alias; ++b)
                alias = prev[b] >= 0 && stream_frames_host[b] >= 0 &&
                        pred_window_alias(stream_frames_host[b], nF, prev[b], p->prev_nF, d.smooth, ring);
        }
        if (alias) APE_CUDA_TRY(cudaStreamWaitEvent(lane, p->done[(k - 1) & 3], 0));
    }
    a.layer_begin = 1; a.layer_end = a.L;
    PIPE_TRY(ape_mc_lstm_tc(&a, lane));
    // the smoothing window of stage 3 reaches into the previous call's predictions (written on the other lane)
    if (p->lstm_done_valid) APE_CUDA_TRY(cudaStreamWaitEvent(lane, p->lstm_done[p->last_lane], 0));
    APE_CUDA_TRY(cudaEventRecord(p->lstm_done[parity], lane));
    p->lstm_done_valid = true;
    p->last_lane = parity;
    float* out = d.out_dev[slot];
    float* samples = d.emit_samples ? out + Em * 32 : nullptr;
    PIPE_TRY(ape_fk_reduce(d.lstm.preds, d.lstm.pred_ring, d.yy_m, d.yy_s, d.body9, d.target, d.lstm.O, d.B, nF, f0, sf_dev,
                           d.lstm.n_samples, d.smooth, out, samples, out + Em * 25, nullptr, (int32_t*)(out + Em * 31), lane));
    APE_CUDA_TRY(cudaEventRecord(p->done[bufset], lane));
    p->done_valid[bufset] = true;
    if (flags & APE_PIPE_CALLER_WAITS) APE_CUDA_TRY(cudaStreamWaitEvent(caller, p->done[bufset], 0));
    if (flags & APE_PIPE_D2H) {
        APE_CUDA_TRY(cudaStreamWaitEvent(p->copy, p->done[bufset], 0));
        float* host = d.out_host[slot];
        const size_t S6 = (size_t)d.smooth * d.lstm.n_samples * 6;
        if (nF == d.nF_max) {
            const size_t words = Em * 32 + (d.emit_samples ? Em * S6 : 0);
            APE_CUDA_TRY(cudaMemcpyAsync(host, out, words * sizeof(float), cudaMemcpyDeviceToHost, p->copy));
        } else {                                               // short call: E estimates packed at the front of each part
            const size_t off[4] = {0, Em * 25, Em * 31, Em * 32}, width[4] = {25, 6, 1, S6};
            for (int i = 0; i < (d.emit_samples ? 4 : 3); ++i)
                APE_CUDA_TRY(cudaMemcpyAsync(host + off[i], out + off[i], E * width[i] * sizeof(float), cudaMemcpyDeviceToHost, p->copy));
        }
        APE_CUDA_TRY(cudaEventRecord(p->slot_ev[slot], p->copy));
        p->slot_busy[slot] = true;
    }
    p->prev_valid = true;
    p->prev_sf = sf_dev != nullptr;
    p->prev_nF = nF; p->prev_frame0 = frame0; p->prev_slot = slot;
    p->calls += 1;
    p->submits += 1;
    *slot_out = slot;
    return APE_OK;
}
