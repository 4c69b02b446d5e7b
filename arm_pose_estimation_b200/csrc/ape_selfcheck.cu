// Host twins of the __host__ __device__ math in ape_common.cuh / ape_features.cuh / ape_fk.cuh, exported so the
// CPU test suite (no GPU in the build container) can pin the exact source the kernels compile - Philox against
// the Random123 known-answer vectors, stage-1 / stage-3 row math against the golden fixtures.  TEST HOOKS ONLY:
// nothing in the product package calls them (tests/test_cabi.py greps for that); they process one row per call.
#include "ape_features.cuh"
#include "ape_fk.cuh"

extern "C" int ape_selfcheck_philox(const uint32_t* ctr4, const uint32_t* key2, uint32_t* out4) {
    if (!ctr4 || !key2 || !out4) return APE_ERR_BAD_ARG;
    const ape::Philox4 r = ape::philox4x32_10(ctr4[0], ctr4[1], ctr4[2], ctr4[3], key2[0], key2[1]);
    for (int i = 0; i < 4; ++i) out4[i] = r.v[i];
    return APE_OK;
}

extern "C" int ape_selfcheck_keep8(uint64_t seed, uint32_t stream, uint32_t frame, uint32_t sample, uint32_t gap,
                                   uint32_t t, uint32_t group, float dropout_p, uint32_t* keep_bits) {
    if (!keep_bits) return APE_ERR_BAD_ARG;
    *keep_bits = ape::philox_keep8(seed, stream, frame, sample, gap, t, group, ape::keep_threshold16(dropout_p));
    return APE_OK;
}

// the branch-free two-lane compare of the tensor-core and batched feed-forward kernels (keep_compare / keep_flags_word) on n
// Philox output words; keep_thr16 == 65536 gives the all-kept flags philox_keep_flags_rk returns for p = 0
extern "C" int ape_selfcheck_keep_flags(const uint32_t* words, int n, uint32_t keep_thr16, uint32_t* flags) {
    if (!words || !flags || n < 0 || keep_thr16 > 65536u) return APE_ERR_BAD_ARG;
    const ape::KeepCompare kc = ape::keep_compare(keep_thr16);
    for (int i = 0; i < n; ++i) flags[i] = keep_thr16 == 65536u ? ape::KEEP_ALL_FLAGS : ape::keep_flags_word(words[i], kc);
    return APE_OK;
}

namespace {
struct HostRow {
    const float* p;
    __host__ __device__ float operator[](int i) const { return p[i]; }
};
}  // namespace

extern "C" int ape_selfcheck_features(int kind, int layout, const float* row, double* xx, int* n_features) {
    if (!row || !xx || !n_features) return APE_ERR_BAD_ARG;
    if (kind < APE_KIND_WATCH_ONLY || kind > APE_KIND_UARM) return APE_ERR_BAD_ARG;
    if (layout != APE_LAYOUT_WATCH_ONLY && layout != APE_LAYOUT_WATCH_PHONE) return APE_ERR_BAD_ARG;
    if (kind != APE_KIND_WATCH_ONLY && layout != APE_LAYOUT_WATCH_PHONE) return APE_ERR_BAD_ARG;
    *n_features = ape::compute_features(kind, layout, HostRow{row}, xx);
    return APE_OK;
}

template <typename F> static int row_pose_host(int target, const double* preds, const double* body9, double* est, int* bad) {
    using namespace ape;
    const int O = target_num_outputs(target);
    F p[20];
    for (int i = 0; i < O; ++i) p[i] = (F)preds[i];
    Body<F> body{{(F)body9[0], (F)body9[1], (F)body9[2]}, {(F)body9[3], (F)body9[4], (F)body9[5]}, {(F)body9[6], (F)body9[7], (F)body9[8]}};
    body.bones_along_x = bones_are_along_x(body);       // the same path the kernel takes for this skeleton
    bool b = false;
    const RowPose<F> r = row_pose<F>(target, p, body, b);
    int k = 0;
    est[k++] = r.hand.x; est[k++] = r.hand.y; est[k++] = r.hand.z;
    est[k++] = r.elbow.x; est[k++] = r.elbow.y; est[k++] = r.elbow.z;
    if (target != APE_TARGET_ORI_CAL_LARM_UARM) { est[k++] = r.shoulder.x; est[k++] = r.shoulder.y; est[k++] = r.shoulder.z; }
    est[k++] = r.larm.w; est[k++] = r.larm.x; est[k++] = r.larm.y; est[k++] = r.larm.z;
    est[k++] = r.uarm.w; est[k++] = r.uarm.x; est[k++] = r.uarm.y; est[k++] = r.uarm.z;
    if (target != APE_TARGET_ORI_CAL_LARM_UARM) { est[k++] = r.hips.w; est[k++] = r.hips.x; est[k++] = r.hips.y; est[k++] = r.hips.z; }
    if (bad) *bad = b ? 1 : 0;
    return APE_OK;
}

// one de-normalised target row -> est row (14 | 21 doubles); use_float != 0 evaluates in float like the kernel
extern "C" int ape_selfcheck_row_pose(int target, const double* preds, const double* body9, int use_float, double* est, int* bad) {
    if (!preds || !body9 || !est) return APE_ERR_BAD_ARG;
    if (target < APE_TARGET_ORI_CAL_LARM_UARM || target > APE_TARGET_ORI_POS_CAL_LARM_UARM_HIPS) return APE_ERR_BAD_ARG;
    return use_float ? row_pose_host<float>(target, preds, body9, est, bad) : row_pose_host<double>(target, preds, body9, est, bad);
}
