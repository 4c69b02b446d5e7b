// Shared between the fp32 (ape_lstm_fma.cu) and tensor-core (ape_lstm_tc.cu) MC-LSTM paths: the argument check, the tiling
// plan of the fp32 layer kernels, the launcher of one fp32 layer, and the per-layer timer of ape_lstm_args::layer_ms.
#pragma once
#include "ape_common.cuh"

namespace ape {

struct FmaPlan {
    int rt0, rt1;                     // rows per tile / 16 of layer 0 and of layers >= 1
    long long tiles0, tiles1;
    size_t seq0_bytes, seq1_bytes, total;
};

int check_lstm_args(const ape_lstm_args* g);
int make_plan(int I, int H, int L, int T, long long E, int n, FmaPlan* p);
int fma_launch_layer(const ape_lstm_args* g, int l, const FmaPlan& p, const float* seq_in, float* seq_out, cudaStream_t st);

// ape_lstm_args::layer_ms: CUDA events at the layer boundaries of a call (none when layer_ms is null or L > 16).  start() creates
// them and marks the start of layer 0, mark(b) the end of a launch whose last layer is b - 1, finish() synchronises the stream and
// writes each launch's device time to the entry of its first layer (0 to the other layers of a launch that runs several).  The
// destructor destroys the events, so they do not leak when a launch fails.
class LayerTimer {
    float* ms_;
    int L_;
    cudaStream_t st_;
    cudaEvent_t ev_[17] = {};
    uint32_t marked_ = 0;

  public:
    LayerTimer(float* layer_ms, int L, cudaStream_t st) : ms_(L <= 16 ? layer_ms : nullptr), L_(L), st_(st) {}
    ~LayerTimer() { for (cudaEvent_t e : ev_) if (e) cudaEventDestroy(e); }
    int start() {
        if (!ms_) return APE_OK;
        for (int b = 0; b <= L_; ++b) APE_CUDA_TRY(cudaEventCreate(&ev_[b]));
        return mark(0);
    }
    int mark(int b) {
        if (!ms_) return APE_OK;
        APE_CUDA_TRY(cudaEventRecord(ev_[b], st_));
        marked_ |= 1u << b;
        return APE_OK;
    }
    int finish() {
        if (!ms_) return APE_OK;
        APE_CUDA_TRY(cudaStreamSynchronize(st_));
        for (int l = 0, next; l < L_; l = next) {
            for (next = l + 1; next < L_ && !(marked_ >> next & 1); ++next) ms_[next] = 0.0f;
            APE_CUDA_TRY(cudaEventElapsedTime(&ms_[l], ev_[l], ev_[next]));
        }
        return APE_OK;
    }
};

}  // namespace ape
