// Stage 3 kernel: de-normalise the network targets, 6D rotation -> quaternion, forward kinematics through
// shoulder -> elbow -> hand for every MC / smoothing row, then the per-estimate reduction: sign-aligned
// quaternion average (transformations.py:32-51), FK again from the averaged quaternions (compose_msg.py:59-61,
// :92-93), population std of the per-row hand / elbow positions.  One HALF-WARP per estimate (two estimates per warp: 100 rows are
// 6.25 passes of 16 lanes instead of 3.1 passes of 32, and every reduction instruction serves two estimates), lanes stride over the
// S = smooth * n_samples rows (consecutive lanes read consecutive rows), reductions by shuffles inside the half-warp, results staged
// through shared memory so the 25-float message leaves coalesced.
#include "ape_fk_x2.cuh"

namespace ape {

// Warps per CTA and resident CTAs per SM -> registers per thread.  The row math wants 96 registers (O = 12) / 128 (O = 14, 20) to run without
// spills (measured, 32 768 estimates x 100 rows, four-warp CTAs: O = 12 at 80 / 96 / 128 registers 0.066 / 0.053 / 0.058 ms; O = 14 at
// 96 / 128: 0.067 / 0.0666 ms, at 160: 0.071).  ONE warp per CTA (two estimates): 0.0524 ms against 0.0532 with four warps and 0.0576 with
// eight (O = 14: 0.0651 / 0.0666 / 0.0699) - the finer the CTAs, the shorter the ragged end of the last wave, and a small launch (1024
// estimates inside the pipeline) spreads over 512 CTAs instead of 128.
#ifndef APE_FK_WARPS
#define APE_FK_WARPS 1
#endif
#ifndef APE_FK_MIN_BLOCKS
#define APE_FK_MIN_BLOCKS(TARGET) (((TARGET) == APE_TARGET_ORI_CAL_LARM_UARM ? 20 : 16) / APE_FK_WARPS)
#endif
constexpr int FK_WARPS_PER_CTA = APE_FK_WARPS;

struct FkArgs {
    const float* preds;
    int pred_ring;
    const float* yy_m;
    const float* yy_s;
    const float* body9;
    int body_stride;                // floats between the skeleton rows of consecutive streams (0: one row for the whole launch)
    int O, B, nF, frame0, n, smooth;
    const int32_t* stream_frames;   // per-stream frame counters (null: frame0 for all); < 0: skip the stream
    float* msg;
    float* samples;
    float* stdev;
    float* est_rows;
    int32_t* status;
    const float* est_in;      // FROM_EST: [E][S][W] rows of arm_pose_from_nn_targets instead of network targets
};

#ifndef APE_FK_L2_PREFETCH
#define APE_FK_L2_PREFETCH 1
#endif
#ifndef APE_FK_LANES
#define APE_FK_LANES 16
#endif
constexpr int FK_LANES = APE_FK_LANES;             // lanes per estimate (fixes the summation order: never chosen by batch size)
constexpr int FK_SUB = 32 / FK_LANES;              // estimates per warp
static_assert(FK_LANES == 8 || FK_LANES == 16, "lanes per estimate");

constexpr unsigned FK_FULL = 0xffffffffu;
// Sums over the FK_LANES lanes of a sub-warp.  Every lane of the warp takes part (full mask: a plain SHFL.BFLY - with a sub-warp mask
// the compiler wraps each shuffle in a MATCH / REDUX / VOTE convergence check, a fifth of the kernel's instructions); the xor
// distances stay below FK_LANES, so the two estimates of a warp never mix.
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = FK_LANES / 2; o > 0; o >>= 1) v += __shfl_xor_sync(FK_FULL, v, o);
    return v;
}
__device__ __forceinline__ F2 warp_sum(F2 v) {
#pragma unroll
    for (int o = FK_LANES / 2; o > 0; o >>= 1) v = v + shfl_xor2(v, o);
    return v;
}

template <typename T> __device__ __forceinline__ Quat<T> bcast0(const Quat<T>& q, int l0) {   // from the sub-warp's lane 0
    return {__shfl_sync(FK_FULL, q.w, l0), __shfl_sync(FK_FULL, q.x, l0), __shfl_sync(FK_FULL, q.y, l0), __shfl_sync(FK_FULL, q.z, l0)};
}

// accumulate q flipped onto the hemisphere of q0 (transformations.py:44-49)
__device__ __forceinline__ void acc_aligned(Quat<float>& s, const Quat<float>& q, const Quat<float>& q0) {
    const float d = q.w * q0.w + q.x * q0.x + q.y * q0.y + q.z * q0.z;
    const float sg = d < 0.0f ? -1.0f : 1.0f;
    s.w += sg * q.w; s.x += sg * q.x; s.y += sg * q.y; s.z += sg * q.z;
}
__device__ __forceinline__ void acc_aligned(Quat2& s, const Quat2& q, const Quat2& q0) {          // lower and upper arm at once
    const F2 d = fma2(q.w, q0.w, fma2(q.x, q0.x, fma2(q.y, q0.y, q.z * q0.z)));
    const F2 sg = pk(lo(d) < 0.0f ? -1.0f : 1.0f, hi(d) < 0.0f ? -1.0f : 1.0f);
    s.w = fma2(sg, q.w, s.w); s.x = fma2(sg, q.x, s.x); s.y = fma2(sg, q.y, s.y); s.z = fma2(sg, q.z, s.z);
}

__device__ __forceinline__ Quat<float> warp_sum_normalised(Quat<float> s) {
    s.w = warp_sum(s.w); s.x = warp_sum(s.x); s.y = warp_sum(s.y); s.z = warp_sum(s.z);
    const float inv = inv_sqrt(s.w * s.w + s.x * s.x + s.y * s.y + s.z * s.z);
    return {s.w * inv, s.x * inv, s.y * inv, s.z * inv};
}
__device__ __forceinline__ Quat2 warp_sum_normalised(Quat2 s) {
    s.w = warp_sum(s.w); s.x = warp_sum(s.x); s.y = warp_sum(s.y); s.z = warp_sum(s.z);
    const F2 inv = rsq2(fma2(s.w, s.w, fma2(s.x, s.x, fma2(s.y, s.y, s.z * s.z))));
    return {s.w * inv, s.x * inv, s.y * inv, s.z * inv};
}

template <int TARGET, bool FROM_EST>
__global__ void __launch_bounds__(FK_WARPS_PER_CTA * 32, APE_FK_MIN_BLOCKS(TARGET)) fk_reduce_kernel(FkArgs a) {
    constexpr int O = TARGET == APE_TARGET_ORI_CAL_LARM_UARM ? 12 : (TARGET == APE_TARGET_ORI_CAL_LARM_UARM_HIPS ? 14 : 20);
    constexpr int W = TARGET == APE_TARGET_ORI_CAL_LARM_UARM ? 14 : 21;
    constexpr bool HIPS = TARGET != APE_TARGET_ORI_CAL_LARM_UARM;
    constexpr bool POS = TARGET == APE_TARGET_ORI_POS_CAL_LARM_UARM_HIPS;
    constexpr int OL = POS ? 3 : 0, OU = POS ? 12 : 6, OH = POS ? 18 : 12;      // first column of the lower-arm / upper-arm 6D, of the hips (sin, cos)
    __shared__ float s_msg[FK_WARPS_PER_CTA * FK_SUB][32];
    __shared__ __align__(16) float s_m[O], s_s[O];

    if (threadIdx.x < O) {
        s_m[threadIdx.x] = a.yy_m ? a.yy_m[threadIdx.x] : 0.0f;
        s_s[threadIdx.x] = a.yy_s ? a.yy_s[threadIdx.x] : 1.0f;
    }
    __syncthreads();

    const int warp = threadIdx.x >> 5, half = (threadIdx.x & 31) / FK_LANES, lane = threadIdx.x & (FK_LANES - 1);   // lane within the sub-warp
    const unsigned hm = ((1u << FK_LANES) - 1u) << (FK_LANES * half);   // this sub-warp's lanes
    const int l0 = FK_LANES * half;                    // its first lane
    const int e = (blockIdx.x * FK_WARPS_PER_CTA + warp) * FK_SUB + half;
    const int E = a.B * a.nF;
    // A sub-warp without an estimate (past the end, or a stream with no new frame in this call: its outputs stay untouched) stays in
    // the warp as a passive participant of the full-mask shuffles; a warp without any estimate leaves.
    bool dead = e >= E;
    int b = 0, f = 0;
    if (!dead) {
        b = a.nF == 1 ? e : e / a.nF;                  // (an integer division is ~20 instructions: the usual shapes go around them)
        const int fb = a.stream_frames ? a.stream_frames[b] : a.frame0;
        dead = fb < 0;
        f = fb + (e - b * a.nF);
    }
    if (__all_sync(FK_FULL, dead)) return;
    const int S = a.smooth * a.n;

    // This estimate's skeleton: row b of the table (stride 0: the one shared row), staged in shared memory by the sub-warp's first nine
    // lanes.  A sub-warp past the end keeps b = 0 and an idle stream's b is in range, so no lane reads outside the table.  Only the two
    // bone lengths of the x-axis rotation stay in registers; the rest of the row is read back (volatile: not hoisted into registers)
    // where it is used - a per-lane row held in registers costs ~10 registers more than the one row the whole launch shared, which the
    // compiler kept in uniform registers, and spills at the launch bounds above.
    // The two estimates of a warp may have different skeletons, one on the short x-axis rotation and one on the general qrot: those
    // branches hold no shuffle, every full-mask shuffle comes before or after them.
    __shared__ float s_body[FK_WARPS_PER_CTA * FK_SUB][9];
    volatile float* sb = s_body[warp * FK_SUB + half];
    if (lane < 9) sb[lane] = __ldg(a.body9 + (size_t)b * a.body_stride + lane);
    __syncwarp();
    auto body_vec = [&](int k) { return Vec3<float>{sb[k], sb[k + 1], sb[k + 2]}; };     // 0: larm_vec, 3: uarm_vec, 6: uarm_orig
    auto body_row = [&]() {
        Body<float> r;
        r.larm_vec = body_vec(0);
        r.uarm_vec = body_vec(3);
        r.uarm_orig = body_vec(6);
        r.bones_along_x = bones_are_along_x(r);
        return r;
    };
    const bool along_x = body_row().bones_along_x;
    const F2 len = pk(sb[0], sb[3]), len2 = len + len;

    const F2 zero2 = splat(0.0f);
    Quat2 q0{zero2, zero2, zero2, zero2}, sq{zero2, zero2, zero2, zero2};          // lo: lower arm, hi: upper arm
    Quat<float> q0h{}, sh{0, 0, 0, 0};
    // hand / elbow positions as the three pairs the samples row stores: (hand.x, hand.y), (hand.z, elbow.x), (elbow.y, elbow.z)
    F2 piv[3] = {zero2, zero2, zero2}, d1[3] = {zero2, zero2, zero2}, d2[3] = {zero2, zero2, zero2};
    F2 psum[3] = {zero2, zero2, zero2};            // ORI_POS target: plain means of hand / elbow / shoulder
    float pshl[3] = {0, 0, 0};
    float sh0[3] = {0, 0, 0};                      // shoulder of row 0 (S == 1: the message copies row 0)
    bool bad = false;

    int rw = lane < a.n ? 0 : lane / a.n, rs = lane - rw * a.n;        // the row this lane requests next: i = rw * n + rs (window frame, MC sample), advanced by FK_LANES per pass
    int ireq = lane;                                  // its index
    // first prediction row of window frame rw (frames clamp to frame 0, estimator.py:114-115; the ring slot costs an integer
    // division, so it is re-derived only when the lane moves on to the next window frame - not per row)
    auto frame_rows = [&](int w) {
        int fw = f - a.smooth + 1 + w;
        fw = fw < 0 ? 0 : fw;
        return a.preds + ((size_t)b * a.pred_ring + (size_t)(fw < a.pred_ring ? fw : fw % a.pred_ring)) * a.n * O;
    };
    if (dead || lane >= S) { rw = 0; rs = 0; ireq = S; }          // no row of its own: reads row 0 (of the buffer, when there is no estimate)
    const float* wrows = FROM_EST ? nullptr : (dead ? a.preds : frame_rows(rw));
    // The prediction row of the NEXT pass is requested before this pass's arithmetic (a lane reads 48 - 80 bytes per pass: with the
    // load issued where it is consumed, a third of the kernel's warp-cycles were spent waiting for it).  Loads and arithmetic are
    // unconditional (no divergent region around them, no predicated register updates): a lane that has run out of rows reads its last
    // row again, and only the sums and the stores ask whether the lane has a row in this pass.
    float pre[O];
    auto request = [&]() {
        const float* row = wrows + rs * O;
        if (O % 4 == 0) {                                        // 48 / 80-byte rows: 16-byte loads
#pragma unroll
            for (int j = 0; j < O / 4; ++j) {
                const float4 v = __ldg(reinterpret_cast<const float4*>(row) + j);
                pre[4 * j] = v.x; pre[4 * j + 1] = v.y; pre[4 * j + 2] = v.z; pre[4 * j + 3] = v.w;
            }
        } else {                                                 // 56-byte rows: 8-byte loads
#pragma unroll
            for (int j = 0; j < O / 2; ++j) {
                const float2 v = __ldg(reinterpret_cast<const float2*>(row) + j);
                pre[2 * j] = v.x; pre[2 * j + 1] = v.y;
            }
        }
        if (ireq + FK_LANES < S) {                               // (the last row is simply read again by the passes that have none)
            ireq += FK_LANES;
            rs += FK_LANES;
            if (rs >= a.n) {
                do { rs -= a.n; ++rw; } while (rs >= a.n);
                wrows = frame_rows(rw);
            }
        }
    };
    if (!FROM_EST) {
        request();
#if APE_FK_L2_PREFETCH
        // ... and ALL rows of the estimate are asked into the L2 right away: one bulk prefetch per window frame (its n rows are
        // contiguous), issued by lane w for frame w.  The register prefetch above then sees the L2's latency instead of the DRAM's from
        // the second pass on (one pass of look-ahead is about 0.7 us of work per SM quarter - less than a loaded DRAM round trip).
        const unsigned fbytes = (unsigned)a.n * O * 4u;
        if (!dead && fbytes % 16u == 0) {
            for (int w = lane; w < a.smooth; w += FK_LANES) {
                const float* fr = frame_rows(w);
                if ((reinterpret_cast<uintptr_t>(fr) & 15) == 0)
                    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(fr), "r"(fbytes) : "memory");
            }
        }
#endif
    }
    unsigned long long* smp = a.samples ? reinterpret_cast<unsigned long long*>(a.samples + ((size_t)e * S + lane) * 6) : nullptr;   // this lane's row of the pass
    Quat2 q{splat(1.0f), zero2, zero2, zero2};
    Quat<float> hips{1.0f, 0.0f, 0.0f, 0.0f};
    Vec3<float> shoulder = body_vec(6);
    F2 P[3] = {zero2, zero2, zero2};
    for (int i0 = 0; i0 < S; i0 += FK_LANES) {
        const int i = i0 + lane;
        const bool live = !dead && i < S;
        if (FROM_EST) {                                              // compose_msg.py entry: rows already hold quats + origins
            if (live) {
                const float* src = a.est_in + ((size_t)e * S + i) * W;
                P[0] = pk(src[0], src[1]); P[1] = pk(src[2], src[3]); P[2] = pk(src[4], src[5]);
                int k = 6;
                if (W == 21) { shoulder = {src[6], src[7], src[8]}; k = 9; }
                q = {pk(src[k], src[k + 4]), pk(src[k + 1], src[k + 5]), pk(src[k + 2], src[k + 6]), pk(src[k + 3], src[k + 7])};
                if (W == 21) hips = {src[k + 8], src[k + 9], src[k + 10], src[k + 11]};
            }
        } else {
            float p[O];
#pragma unroll
            for (int j = 0; j < O; ++j) p[j] = fmaf(pre[j], s_s[j], s_m[j]);   // estimator.py:108-109
            request();
            bool rb = false;
            q = six_to_quat_x2(p + OL, p + OU, rb);                  // estimate_joints.py:20-92
            bad |= rb && live;
            if (HIPS) {
                hips = hips_quat(p[OH], p[OH + 1]);
                shoulder = qrot(hips, body_vec(6));
            }
            if (POS) {                                               // positions are network outputs
                P[0] = pk(p[0], p[1]); P[1] = pk(p[2], p[9]); P[2] = pk(p[10], p[11]);
            } else if (along_x) {                                    // shoulder -> elbow -> hand (estimate_joints.py:61-63 / :84-85)
                if (!HIPS) shoulder = body_vec(6);
                F2 vx, vy, vz;
                qrot_x2(q, len, len2, vx, vy, vz);
                const float ex = hi(vx) + shoulder.x, ey = hi(vy) + shoulder.y, ez = hi(vz) + shoulder.z;
                P[0] = pk(lo(vx) + ex, lo(vy) + ey); P[1] = pk(lo(vz) + ez, ex); P[2] = pk(ey, ez);
            } else {
                if (!HIPS) shoulder = body_vec(6);
                const Vec3<float> el = vadd(qrot(q_hi(q), body_vec(3)), shoulder), ha = vadd(qrot(q_lo(q), body_vec(0)), el);
                P[0] = pk(ha.x, ha.y); P[1] = pk(ha.z, el.x); P[2] = pk(el.y, el.z);
            }
        }
        if (i0 == 0) {                                               // row 0 anchors the sign alignment and the std pivot
            q0 = {shfl_idx2(q.w, l0), shfl_idx2(q.x, l0), shfl_idx2(q.y, l0), shfl_idx2(q.z, l0)};
            if (HIPS) q0h = bcast0(hips, l0);
#pragma unroll
            for (int j = 0; j < 3; ++j) piv[j] = shfl_idx2(P[j], l0);
            sh0[0] = __shfl_sync(FK_FULL, shoulder.x, l0);
            sh0[1] = __shfl_sync(FK_FULL, shoulder.y, l0);
            sh0[2] = __shfl_sync(FK_FULL, shoulder.z, l0);
        }
        if (live) {
            acc_aligned(sq, q, q0);
            if (HIPS) acc_aligned(sh, hips, q0h);
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                const F2 d = P[j] - piv[j];
                d1[j] = d1[j] + d;
                d2[j] = fma2(d, d, d2[j]);
            }
            if (POS) {
#pragma unroll
                for (int j = 0; j < 3; ++j) psum[j] = psum[j] + P[j];
                pshl[0] += shoulder.x; pshl[1] += shoulder.y; pshl[2] += shoulder.z;
            }
            if (smp) {
                smp[0] = P[0].v; smp[1] = P[1].v; smp[2] = P[2].v;
                smp += FK_LANES * 3;
            }
            if (a.est_rows) {
                float* dst = a.est_rows + ((size_t)e * S + i) * W;
                int k = 0;
#pragma unroll
                for (int j = 0; j < 3; ++j) { dst[k++] = lo(P[j]); dst[k++] = hi(P[j]); }
                if (W == 21) { dst[k++] = shoulder.x; dst[k++] = shoulder.y; dst[k++] = shoulder.z; }
                dst[k++] = lo(q.w); dst[k++] = lo(q.x); dst[k++] = lo(q.y); dst[k++] = lo(q.z);
                dst[k++] = hi(q.w); dst[k++] = hi(q.x); dst[k++] = hi(q.y); dst[k++] = hi(q.z);
                if (W == 21) { dst[k++] = hips.w; dst[k++] = hips.x; dst[k++] = hips.y; dst[k++] = hips.z; }
            }
        }
    }

    // ---- reduction over the S rows --------------------------------------------------------------------
    RowPose<float> m;
    const Quat2 mq = S == 1 ? q0 : warp_sum_normalised(sq);                   // one row: copied, not re-normalised
    m.larm = q_lo(mq);
    m.uarm = q_hi(mq);
    m.hips = !HIPS ? Quat<float>{1.0f, 0.0f, 0.0f, 0.0f} : (S == 1 ? q0h : warp_sum_normalised(sh));
    const float invS = 1.0f / (float)S;
    if (POS) {
#pragma unroll
        for (int j = 0; j < 3; ++j) psum[j] = warp_sum(psum[j]) * splat(invS);    // compose_msg.py:27-29
#pragma unroll
        for (int j = 0; j < 3; ++j) pshl[j] = warp_sum(pshl[j]) * invS;
        m.hand = {lo(psum[0]), hi(psum[0]), lo(psum[1])};
        m.elbow = {hi(psum[1]), lo(psum[2]), hi(psum[2])};
        m.shoulder = {pshl[0], pshl[1], pshl[2]};
    } else if (S > 1) {
        chain(TARGET, body_row(), m);                                               // FK again from the means
    } else {                                                                  // one row: copied as is (compose_msg.py:62-66)
        m.hand = {lo(piv[0]), hi(piv[0]), lo(piv[1])};
        m.elbow = {hi(piv[1]), lo(piv[2]), hi(piv[2])};
        m.shoulder = {sh0[0], sh0[1], sh0[2]};
    }
    float sd[6];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        const F2 m1 = warp_sum(d1[j]) * splat(invS), m2 = warp_sum(d2[j]) * splat(invS), var = fma2(-m1, m1, m2);
        asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(sd[2 * j]) : "f"(fmaxf(lo(var), 0.0f)));
        asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(sd[2 * j + 1]) : "f"(fmaxf(hi(var), 0.0f)));
    }
    const unsigned any_bad = __ballot_sync(FK_FULL, bad) & hm;

    if (lane == 0 && !dead) {
        float* o = s_msg[warp * FK_SUB + half];                                             // compose_msg.py:67-79 / :100-108
        o[0] = m.larm.w; o[1] = m.larm.x; o[2] = m.larm.y; o[3] = m.larm.z;
        o[4] = m.hand.x; o[5] = m.hand.y; o[6] = m.hand.z;
        o[7] = m.larm.w; o[8] = m.larm.x; o[9] = m.larm.y; o[10] = m.larm.z;
        o[11] = m.elbow.x; o[12] = m.elbow.y; o[13] = m.elbow.z;
        o[14] = m.uarm.w; o[15] = m.uarm.x; o[16] = m.uarm.y; o[17] = m.uarm.z;
        o[18] = m.shoulder.x; o[19] = m.shoulder.y; o[20] = m.shoulder.z;
        o[21] = m.hips.w; o[22] = m.hips.x; o[23] = m.hips.y; o[24] = m.hips.z;
        if (a.status) a.status[e] = any_bad ? 1 : 0;
    }
    __syncwarp();
    if (dead) return;
    for (int k = lane; k < 25; k += FK_LANES) a.msg[(size_t)e * 25 + k] = s_msg[warp * FK_SUB + half][k];
    if (a.stdev && lane < 6) {
        float v = sd[0];
#pragma unroll
        for (int j = 1; j < 6; ++j) v = lane == j ? sd[j] : v;
        a.stdev[(size_t)e * 6 + lane] = v;
    }
}

}  // namespace ape

extern "C" int ape_fk_reduce_bodies(const float* preds, int pred_ring, const float* yy_m, const float* yy_s,
                                    const float* bodies, int body_stride, int target, int O, int B, int nF, int frame0,
                                    const int32_t* stream_frames, int n_samples, int smooth, float* msg, float* samples, float* stdev,
                                    float* est_rows, int32_t* status, void* stream) {
    using namespace ape;
    if (!preds || !bodies || !msg || B < 0 || nF < 0 || frame0 < 0 || n_samples < 1 || smooth < 1 || pred_ring < 1)
        return APE_ERR_BAD_ARG;
    if (body_stride < 0 || (body_stride > 0 && body_stride < 9)) return APE_ERR_BAD_ARG;   // rows of 9 floats must not overlap
    if (target < APE_TARGET_ORI_CAL_LARM_UARM || target > APE_TARGET_ORI_POS_CAL_LARM_UARM_HIPS) return APE_ERR_BAD_ARG;
    if (O != target_num_outputs(target)) return APE_ERR_BAD_ARG;
    if ((yy_m == nullptr) != (yy_s == nullptr)) return APE_ERR_BAD_ARG;
    if (nF + smooth - 1 > pred_ring) return APE_ERR_BAD_ARG;          // the smoothing window must still be in the ring
    const long long E = (long long)B * nF;
    if (E == 0) return APE_OK;
    if (E > 0x7fffffffLL || (long long)smooth * n_samples > 0x7fffffffLL) return APE_ERR_BAD_ARG;
    FkArgs a{preds, pred_ring, yy_m, yy_s, bodies, body_stride, O, B, nF, frame0, n_samples, smooth, stream_frames, msg, samples, stdev,
             est_rows, status, nullptr};
    const int grid = (int)((E + FK_SUB * FK_WARPS_PER_CTA - 1) / (FK_SUB * FK_WARPS_PER_CTA));
    cudaStream_t st = (cudaStream_t)stream;
    if (target == APE_TARGET_ORI_CAL_LARM_UARM)
        fk_reduce_kernel<APE_TARGET_ORI_CAL_LARM_UARM, false><<<grid, FK_WARPS_PER_CTA * 32, 0, st>>>(a);
    else if (target == APE_TARGET_ORI_CAL_LARM_UARM_HIPS)
        fk_reduce_kernel<APE_TARGET_ORI_CAL_LARM_UARM_HIPS, false><<<grid, FK_WARPS_PER_CTA * 32, 0, st>>>(a);
    else
        fk_reduce_kernel<APE_TARGET_ORI_POS_CAL_LARM_UARM_HIPS, false><<<grid, FK_WARPS_PER_CTA * 32, 0, st>>>(a);
    return check_launch();
}

// one skeleton for every stream: the table form with stride 0 (the same kernel, the same arithmetic)
extern "C" int ape_fk_reduce(const float* preds, int pred_ring, const float* yy_m, const float* yy_s,
                             const float* body9, int target, int O, int B, int nF, int frame0, const int32_t* stream_frames, int n_samples,
                             int smooth, float* msg, float* samples, float* stdev, float* est_rows,
                             int32_t* status, void* stream) {
    return ape_fk_reduce_bodies(preds, pred_ring, yy_m, yy_s, body9, 0, target, O, B, nF, frame0, stream_frames, n_samples, smooth,
                                msg, samples, stdev, est_rows, status, stream);
}

extern "C" int ape_msg_from_est(const float* est, int W, const float* body9, int target, int E, int S, float* msg,
                                float* stdev, void* stream) {
    using namespace ape;
    if (!est || !body9 || !msg || E < 0 || S < 1) return APE_ERR_BAD_ARG;
    if (target < APE_TARGET_ORI_CAL_LARM_UARM || target > APE_TARGET_ORI_POS_CAL_LARM_UARM_HIPS) return APE_ERR_BAD_ARG;
    if (W != (target == APE_TARGET_ORI_CAL_LARM_UARM ? 14 : 21)) return APE_ERR_BAD_ARG;
    if (E == 0) return APE_OK;
    FkArgs a{nullptr, 1, nullptr, nullptr, body9, 0, target_num_outputs(target), E, 1, 0, S, 1, nullptr, msg, nullptr, stdev, nullptr, nullptr, est};
    const int grid = (E + FK_SUB * FK_WARPS_PER_CTA - 1) / (FK_SUB * FK_WARPS_PER_CTA);
    cudaStream_t st = (cudaStream_t)stream;
    if (target == APE_TARGET_ORI_CAL_LARM_UARM)
        fk_reduce_kernel<APE_TARGET_ORI_CAL_LARM_UARM, true><<<grid, FK_WARPS_PER_CTA * 32, 0, st>>>(a);
    else if (target == APE_TARGET_ORI_CAL_LARM_UARM_HIPS)
        fk_reduce_kernel<APE_TARGET_ORI_CAL_LARM_UARM_HIPS, true><<<grid, FK_WARPS_PER_CTA * 32, 0, st>>>(a);
    else
        fk_reduce_kernel<APE_TARGET_ORI_POS_CAL_LARM_UARM_HIPS, true><<<grid, FK_WARPS_PER_CTA * 32, 0, st>>>(a);
    return check_launch();
}
