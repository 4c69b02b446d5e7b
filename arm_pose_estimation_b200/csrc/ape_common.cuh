// Shared host/device helpers of the B200 arm-pose kernels: error plumbing, quaternion algebra,
// Philox4x32-10.  Everything marked APE_HD also compiles for the host so tests/test_host_math.py can
// exercise the exact same source on the CPU box (see csrc/host_check.cu).
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/ape_b200.h"

#define APE_HD __host__ __device__ __forceinline__

namespace ape {

// ---- error plumbing -------------------------------------------------------------------------------
extern thread_local cudaError_t g_last_err;
inline int cuda_fail(cudaError_t e) { g_last_err = e; return APE_ERR_CUDA; }
#define APE_CUDA_TRY(expr) do { cudaError_t _e = (expr); if (_e != cudaSuccess) return ape::cuda_fail(_e); } while (0)

inline int check_launch() {
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? APE_OK : cuda_fail(e);
}

// ---- per-stream frame counters ----------------------------------------------------------------------
// A launch either advances all streams in lock-step (frame0) or takes one absolute frame number per stream
// (stream_frames[b]; a NEGATIVE entry means "this stream has no new frame in this call": its rows are still part of
// the tiles, but nothing of it is written anywhere).
APE_HD int stream_frame0(const int32_t* stream_frames, int frame0, int b) { return stream_frames ? stream_frames[b] : frame0; }

// ---- quaternion algebra, [w,x,y,z], templated on the float type -----------------------------------
template <typename F> struct Quat { F w, x, y, z; };
template <typename F> struct Vec3 { F x, y, z; };

// Hamilton product; component formulas of transformations.py:141-144
template <typename F> APE_HD Quat<F> qmul(const Quat<F>& a, const Quat<F>& b) {
    return {a.w * b.w - a.x * b.x - a.y * b.y - a.z * b.z,
            a.w * b.x + a.x * b.w + a.y * b.z - a.z * b.y,
            a.w * b.y - a.x * b.z + a.y * b.w + a.z * b.x,
            a.w * b.z + a.x * b.y - a.y * b.x + a.z * b.w};
}
template <typename F> APE_HD Quat<F> qconj(const Quat<F>& q) { return {q.w, -q.x, -q.y, -q.z}; }

// q (x) [0,v] (x) conj(q) without normalising q (transformations.py:105-121)
template <typename F> APE_HD Vec3<F> qrot(const Quat<F>& q, const Vec3<F>& v) {
    // the two Hamilton products written out without the terms that multiply the zero scalar part of [0, v] and without the
    // scalar part of the result (which is not used): the same sums in the same order
    const Quat<F> a = {-q.x * v.x - q.y * v.y - q.z * v.z,
                       q.w * v.x + q.y * v.z - q.z * v.y,
                       q.w * v.y - q.x * v.z + q.z * v.x,
                       q.w * v.z + q.x * v.y - q.y * v.x};
    return {-a.w * q.x + a.x * q.w - a.y * q.z + a.z * q.y,
            -a.w * q.y + a.x * q.z + a.y * q.w - a.z * q.x,
            -a.w * q.z - a.x * q.y + a.y * q.x + a.z * q.w};
}
// qrot for a vector along the x axis, v = (vx, 0, 0) - the default bone vectors (bone_map.py:42-45) - written out: vx times the
// first column of the (unnormalised) rotation matrix of q.  10 operations instead of 42.
// The first two squares are ONE fused multiply-add, x^2 fused onto w^2, written out: left to the compiler, which of the two products
// it fuses depended on the code around the call (the last bit of the stage-3 message moved with an unrelated change of the kernel).
APE_HD float fmadd(float a, float b, float c) { return fmaf(a, b, c); }
APE_HD double fmadd(double a, double b, double c) { return fma(a, b, c); }
template <typename F> APE_HD Vec3<F> qrot_x(const Quat<F>& q, F vx) {
    return {vx * (fmadd(q.x, q.x, q.w * q.w) - q.y * q.y - q.z * q.z), vx * F(2) * (q.x * q.y + q.w * q.z), vx * F(2) * (q.x * q.z - q.w * q.y)};
}
// conjugate / squared norm (transformations.py:244-254)
template <typename F> APE_HD Quat<F> qinv(const Quat<F>& q) {
    F n = q.w * q.w + q.x * q.x + q.y * q.y + q.z * q.z;
    return {q.w / n, -q.x / n, -q.y / n, -q.z / n};
}
// android [w,x,y,z] -> global axis swap [-w,x,z,y] (transformations.py:225-229)
template <typename F> APE_HD Quat<F> android_swap(const Quat<F>& q) { return {-q.w, q.x, q.z, q.y}; }

// ---- Philox4x32-10 (Salmon et al. 2011), the counter-based generator of APE_MASK_PHILOX ------------
struct Philox4 { uint32_t v[4]; };

APE_HD void mulhilo32(uint32_t a, uint32_t b, uint32_t& hi, uint32_t& lo) {
    const uint64_t p = (uint64_t)a * (uint64_t)b;          // one IMAD.WIDE.U32 on the device
    lo = (uint32_t)p;
    hi = (uint32_t)(p >> 32);
}

APE_HD Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0, lo0, hi1, lo1;
        mulhilo32(M0, c0, hi0, lo0);
        mulhilo32(M1, c2, hi1, lo1);
        uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += W0; k1 += W1;
    }
    return {{c0, c1, c2, c3}};
}

// Dropout keep-bits of 8 consecutive hidden units [8*group, 8*group+8) of one (stream, frame, sample, gap, t).
// Counter = (stream id, absolute frame, sample | gap<<20 | t<<24, unit group); key = 64-bit seed.
// Each 32-bit output word yields two 16-bit lanes (low half first); unit j is kept iff lane_j < keep_thr16,
// keep_thr16 = round((1-p) * 65536).  Independent of tiling, launch shape and GPU count by construction.
APE_HD uint32_t philox_keep8(uint64_t seed, uint32_t stream, uint32_t frame, uint32_t sample, uint32_t gap,
                             uint32_t t, uint32_t group, uint32_t keep_thr16) {
    Philox4 r = philox4x32_10(stream, frame, (sample & 0xFFFFFu) | ((gap & 0xFu) << 20) | ((t & 0xFFu) << 24), group,
                              (uint32_t)seed, (uint32_t)(seed >> 32));
    uint32_t bits = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        bits |= ((r.v[i] & 0xFFFFu) < keep_thr16 ? 1u : 0u) << (2 * i);
        bits |= ((r.v[i] >> 16) < keep_thr16 ? 1u : 0u) << (2 * i + 1);
    }
    return bits;
}

#ifdef __CUDACC__
// The same draw as philox_keep8, returned as four half2 AND-masks (0xFFFF per kept 16-bit lane: unit 2i in the low
// half of word i, unit 2i+1 in the high half) so fp16 operand units can be masked without unpacking.
__device__ __forceinline__ uint4 philox_keep_halfmask(uint64_t seed, uint32_t stream, uint32_t frame, uint32_t sample,
                                                      uint32_t gap, uint32_t t, uint32_t group, uint32_t keep_thr16) {
    if (keep_thr16 >= 65536u) return make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu);
    const Philox4 r = philox4x32_10(stream, frame, (sample & 0xFFFFFu) | ((gap & 0xFu) << 20) | ((t & 0xFFu) << 24), group,
                                    (uint32_t)seed, (uint32_t)(seed >> 32));
    const uint32_t thr2 = keep_thr16 | (keep_thr16 << 16);
    return make_uint4(__vcmpltu2(r.v[0], thr2), __vcmpltu2(r.v[1], thr2), __vcmpltu2(r.v[2], thr2), __vcmpltu2(r.v[3], thr2));
}
#endif

// Philox4x32-10's key schedule depends on the seed alone: the host evaluates the 10 round keys once and passes them as kernel
// parameters, so on the device they are constant-bank / uniform-register operands of the round's XORs - a round is then
// 2 IMAD.WIDE + 2 LOP3 instead of 8 issue slots (the tensor-core kernels' loader warps are issue-bound).
struct PhiloxRoundKeys { uint32_t k[20]; };
APE_HD PhiloxRoundKeys philox_round_keys(uint64_t seed) {
    PhiloxRoundKeys rk;
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    for (int r = 0; r < 10; ++r) { rk.k[2 * r] = k0; rk.k[2 * r + 1] = k1; k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
    return rk;
}
// Keep FLAGS of the 8 lanes of a draw: bit 15 (low lane) and bit 31 (high lane) of word i are set iff that 16-bit lane is
// < keep_thr16 - the same decision as `lane < keep_thr16` above, evaluated for both lanes of a word with three integer
// operations instead of an emulated SIMD compare (the loader warps of the tensor-core kernels are issue-bound):
//   lane < thr  <=>  thr.bit15 ? (lane.bit15 == 0 || lane.low15 < thr.low15) : (lane.bit15 == 0 && lane.low15 < thr.low15)
//   lane.low15 < thr.low15  <=>  bit 15 of (0x7FFF + thr.low15 - lane.low15)   (no borrow between the lanes: 0 <= . <= 0xFFFE)
// Valid for keep_thr16 <= 0xFFFF; 65536 (p = 0) is the caller's shortcut.  Host and device, so ape_selfcheck_keep_flags can
// check every lane value on the CPU.
struct KeepCompare { uint32_t k2, top; };      // k2: (0x7FFF + thr.low15) in both lanes; top: all ones iff thr.bit15
APE_HD KeepCompare keep_compare(uint32_t keep_thr16) {
    const uint32_t k = 0x7FFFu + (keep_thr16 & 0x7FFFu);
    return {k | (k << 16), (keep_thr16 & 0x8000u) ? 0xFFFFFFFFu : 0u};
}
APE_HD uint32_t keep_flags_word(uint32_t c, const KeepCompare kc) {
    const uint32_t d = kc.k2 - (c & 0x7FFF7FFFu);
    return (~c & d) | (kc.top & (~c | d));     // one LOP3: top ? (~c | d) : (~c & d)
}
// the flag words of p = 0 (keep_thr16 == 65536): every lane kept
constexpr uint32_t KEEP_ALL_FLAGS = 0x80008000u;
#ifdef __CUDACC__
// flags (bits 15 / 31) -> half2 AND-mask (0xFFFF per kept lane): one byte permute with sign replication
__device__ __forceinline__ uint32_t keep_flags_to_halfmask(uint32_t flags) {
    uint32_t m;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(m) : "r"(flags), "r"(0u), "r"(0xBB99u));
    return m;
}
// the four flag words of one draw (Philox4x32-10 with precomputed round keys; counter layout of philox_keep8)
__device__ __forceinline__ uint4 philox_keep_flags_rk(const PhiloxRoundKeys& rk, uint32_t stream, uint32_t frame, uint32_t sample,
                                                      uint32_t gap, uint32_t t, uint32_t group, uint32_t keep_thr16) {
    if (keep_thr16 >= 65536u) return make_uint4(KEEP_ALL_FLAGS, KEEP_ALL_FLAGS, KEEP_ALL_FLAGS, KEEP_ALL_FLAGS);
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
    uint32_t c0 = stream, c1 = frame, c2 = (sample & 0xFFFFFu) | ((gap & 0xFu) << 20) | ((t & 0xFFu) << 24), c3 = group;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0, lo0, hi1, lo1;
        mulhilo32(M0, c0, hi0, lo0);
        mulhilo32(M1, c2, hi1, lo1);
        const uint32_t n0 = hi1 ^ c1 ^ rk.k[2 * r], n2 = hi0 ^ c3 ^ rk.k[2 * r + 1];
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    }
    const KeepCompare kc = keep_compare(keep_thr16);
    return make_uint4(keep_flags_word(c0, kc), keep_flags_word(c1, kc), keep_flags_word(c2, kc), keep_flags_word(c3, kc));
}
// philox_keep_halfmask with precomputed round keys: bit-identical draws
__device__ __forceinline__ uint4 philox_keep_halfmask_rk(const PhiloxRoundKeys& rk, uint32_t stream, uint32_t frame, uint32_t sample,
                                                         uint32_t gap, uint32_t t, uint32_t group, uint32_t keep_thr16) {
    const uint4 f = philox_keep_flags_rk(rk, stream, frame, sample, gap, t, group, keep_thr16);
    return make_uint4(keep_flags_to_halfmask(f.x), keep_flags_to_halfmask(f.y), keep_flags_to_halfmask(f.z), keep_flags_to_halfmask(f.w));
}
#endif

APE_HD uint32_t keep_threshold16(float p) {
    float k = (1.0f - p) * 65536.0f + 0.5f;
    return k >= 65536.0f ? 65536u : (k <= 0.0f ? 0u : (uint32_t)k);
}

}  // namespace ape
