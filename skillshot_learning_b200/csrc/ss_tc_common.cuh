// ss_tc_common.cuh -- shared pieces of the tcgen05 (5th-generation tensor core) kernels:
// PTX wrappers, the shared-memory operand layout, descriptors, weight staging.
//
// Operand layout.  Every bf16 matrix that the tensor core reads lives in shared memory as
// "chunked" tiles  [cols / 8][rows][8]:  element (row r, col c) at
//     (c / 8) * rows * 16  +  r * 16  +  (c % 8) * 2      bytes.
// That one image is a valid UMMA canonical no-swizzle operand in BOTH orientations:
//   * K-major  with K = c  (8 rows x 16 B core matrices, SBO = 128 B between 8-row groups,
//     LBO = rows * 16 B between K chunks)           -- forward:  out[r][n] += tile[r][c] * W[n][c]
//   * MN-major with MN = c, K = r  (SBO = rows * 16 B between 8-column groups, LBO = 128 B
//     between 8-row K groups)                        -- weight gradients:  dW[c][n] += tile[r][c] * d[r][n]
// so activations written once by an epilogue serve the next layer's GEMM and, in the backward
// pass, the weight-gradient GEMMs whose reduction runs over the 128 rows of the tile; the
// weight image of layer 2 serves the forward GEMM (K-major) and the input-gradient GEMM
// (MN-major) alike.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/skillshot_b200.h"
#include "ss_launch.cuh"
#include "ss_rng.cuh"

namespace sstc {

using namespace ss;

constexpr int NET_ACTOR = 0, NET_CRITIC = 1;

constexpr int TM = 128;                  // rows per tile = UMMA M = tensor-memory lanes
constexpr int DS = SS_DIM_STATE, DA = SS_DIM_ACTION, H1 = SS_HIDDEN1, H2 = SS_HIDDEN2;
// layer-1 K: [s hi 12 | 1 1 0 0 | s lo 12 | 0 x4]; rows 12, 13 of B1 = b1 hi, lo
constexpr int K1 = 32;
// the forward kernels run layer 1 in fp16 instead (11-bit significands on both operands: finer than a pixel on
// the positions and finer than bf16 on the weights), K = 16: [s 12 | 1 1 0 0]; rows 12, 13 of B1 = b1 hi, lo (fp16)
constexpr int K1F = 16;
// layer-2 K: [h1 256 | tail 8 | 0 x8]; tail = actor {1 1 0..}            B2 rows 256.. = {b2 hi, b2 lo}
//                                      critic {a0h a1h a0l a1l 1 1 0 0}  B2 rows 256.. = {W2[256] W2[257] W2[256] W2[257] b2 hi, b2 lo}
constexpr int K2 = H1 + 16;

// flat parameter vectors (Keras get_weights() order); W1, b1, W2 start at the same offsets in both nets
constexpr int P_W1 = 0, P_B1 = P_W1 + DS * H1, P_W2 = P_B1 + H1;
constexpr int A_B2 = P_W2 + H1 * H2, A_W3 = A_B2 + H2, A_B3 = A_W3 + H2 * DA, A_N = A_B3 + DA;
constexpr int C_B2 = P_W2 + (H1 + DA) * H2, C_W3 = C_B2 + H2, C_B3 = C_W3 + H2, C_N = C_B3 + 1;
static_assert(A_N == SS_ACTOR_PARAMS && C_N == SS_CRITIC_PARAMS, "parameter counts");

constexpr uint32_t CHUNK_A = TM * 16;    // 2048: chunk stride of a 128-row activation tile
constexpr uint32_t CHUNK_B1 = H1 * 16;   // 4096: chunk stride of the layer-1 weight image (256 rows)
constexpr uint32_t CHUNK_B2 = H2 * 16;   // 2048: chunk stride of the layer-2 weight image (128 rows)
constexpr uint32_t CORE = 128;           // 8 rows x 16 B
constexpr uint32_t B1_BYTES = (K1 / 8) * CHUNK_B1;          // 16,384
constexpr uint32_t B2_BYTES = (K2 / 8) * CHUNK_B2;          // 69,632
constexpr uint32_t X2_BYTES = (K2 / 8) * CHUNK_A;           // 69,632
constexpr uint32_t ONES = 0x3F803F80u;                      // bf16 {1, 1}

// ---- PTX wrappers -----------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_test(uint32_t bar, uint32_t parity) {      // may park the thread for a while
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
// Waits for the phase with the given parity.  try_wait parks the thread in hardware for a bounded
// time per call; a barrier that never completes is a protocol bug, so give up after ~10^6 attempts
// and trap instead of hanging the device.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t spins = 0;
    while (!mbar_test(bar, parity)) {
        if (++spins > (1u << 22)) __trap();
    }
}
// For a barrier that has usually completed by the time it is looked at (the MMA-issuing thread's waits): one
// non-suspending test first -- try_wait costs ~170 cycles even on a completed phase, test_wait a fraction of that --
// and the parking wait only if the phase is still open.
__device__ __forceinline__ bool mbar_poll(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait_likely_done(uint32_t bar, uint32_t parity) {
    if (!mbar_poll(bar, parity)) mbar_wait(bar, parity);
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t cols) {   // one full warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}

// shared-memory matrix descriptor: start address, leading / stride byte offsets (all >> 4),
// descriptor version 1 (sm_100), layout type 0 = no swizzle
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(sbo >> 4) << 32) |
           (1ull << 46);
}
// chunked tile [cols/8][rows][8] read K-major (K = cols): consecutive MMA K-steps (16 cols) are 2 chunks apart
__device__ __forceinline__ uint64_t desc_kmajor(uint32_t saddr, uint32_t chunk_bytes) {
    return umma_desc(saddr, chunk_bytes, CORE);
}
// the same tile read MN-major (MN = cols, K = rows): consecutive K-steps (16 rows) are 256 B apart
__device__ __forceinline__ uint64_t desc_mnmajor(uint32_t saddr, uint32_t chunk_bytes) {
    return umma_desc(saddr, CORE, chunk_bytes);
}
__device__ __forceinline__ uint64_t desc_advance(uint64_t d, uint32_t bytes) { return d + (uint64_t)(bytes >> 4); }

// instruction descriptor, kind::f16: D = f32, A = B = bf16, shape M x N (x 16); *_mn = operand is MN-major
__host__ __device__ constexpr uint32_t umma_idesc(int M, int N, int a_mn = 0, int b_mn = 0) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) |
           ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// the same with A = B = fp16 (format code 0), both K-major
__host__ __device__ constexpr uint32_t umma_idesc_f16(int M, int N) {
    return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        :
        : "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrives on the mbarrier once every tcgen05 operation this thread issued so far has retired
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// 32 consecutive fp32 columns of this thread's tensor-memory lane
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- bf16 packing -------------------------------------------------------------
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
    uint32_t d;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));        // first source -> upper half
    return d;
}
// ReLU fused into the conversion: max(x, 0) rounded to bf16, two at a time
__device__ __forceinline__ uint32_t pack_relu_bf16(float lo, float hi) {
    uint32_t d;
    asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    return d;
}
__device__ __forceinline__ uint32_t pack_f16(float lo, float hi) {
    uint32_t d;
    asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));         // first source -> upper half
    return d;
}
__device__ __forceinline__ uint32_t hi_lo_f16(float w) {                       // fp16 {hi, lo} with hi + lo = w to 2^-22
    const float hi = __half2float(__float2half_rn(w));
    return pack_f16(hi, w - hi);
}
__device__ __forceinline__ float bf16_round(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }
__device__ __forceinline__ uint32_t hi_lo_bf16(float w) {                     // {hi, lo} with hi + lo = w to 2^-17
    const float hi = bf16_round(w);
    return pack_bf16(hi, w - hi);
}
__device__ __forceinline__ float bf16_lo(uint32_t p) { return __uint_as_float(p << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t p) { return __uint_as_float(p & 0xFFFF0000u); }

// 32 accumulator columns -> ReLU -> bf16 -> four 16-byte chunks of this thread's row of a 128-row tile
__device__ __forceinline__ void relu_pack_store(const uint32_t (&v)[32], uint8_t *dst) {
#pragma unroll
    for (int c = 0; c < 4; ++c)
        *reinterpret_cast<uint4 *>(dst + c * CHUNK_A) = make_uint4(
            pack_relu_bf16(__uint_as_float(v[c * 8 + 0]), __uint_as_float(v[c * 8 + 1])),
            pack_relu_bf16(__uint_as_float(v[c * 8 + 2]), __uint_as_float(v[c * 8 + 3])),
            pack_relu_bf16(__uint_as_float(v[c * 8 + 4]), __uint_as_float(v[c * 8 + 5])),
            pack_relu_bf16(__uint_as_float(v[c * 8 + 6]), __uint_as_float(v[c * 8 + 7])));
}

// observation row -> the two fp16 layer-1 chunks [x 0..7][x 8..11, 1, 1, 0, 0] of the forward kernels (K = 16)
__device__ __forceinline__ void store_obs_row_f16(const float4 (&x)[3], uint8_t *row) {
    *reinterpret_cast<uint4 *>(row) =
        make_uint4(pack_f16(x[0].x, x[0].y), pack_f16(x[0].z, x[0].w), pack_f16(x[1].x, x[1].y), pack_f16(x[1].z, x[1].w));
    *reinterpret_cast<uint4 *>(row + CHUNK_A) = make_uint4(pack_f16(x[2].x, x[2].y), pack_f16(x[2].z, x[2].w), 0x3C003C00u, 0u);
}
// observation row -> the bf16 layer-1 chunks [hi 0..7][hi 8..11, 1, 1, 0, 0][lo 0..7][lo 8..11, 0 x4] of its tile row
// (K = 32, gradient kernel): slice 0 writes the two high chunks, slice 1 the two low ones (two warps share a row)
__device__ __forceinline__ void store_obs_half(const float4 (&xin)[3], uint8_t *row, int slice) {
    const float x[12] = {xin[0].x, xin[0].y, xin[0].z, xin[0].w, xin[1].x, xin[1].y,
                         xin[1].z, xin[1].w, xin[2].x, xin[2].y, xin[2].z, xin[2].w};
    float v[12];
#pragma unroll
    for (int e = 0; e < 12; ++e) {
        const float hi = bf16_round(x[e]);
        v[e] = slice == 0 ? hi : x[e] - hi;
    }
    *reinterpret_cast<uint4 *>(row + (2 * slice) * CHUNK_A) =
        make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
    *reinterpret_cast<uint4 *>(row + (2 * slice + 1) * CHUNK_A) =
        make_uint4(pack_bf16(v[8], v[9]), pack_bf16(v[10], v[11]), slice == 0 ? ONES : 0u, 0u);
}
// the constant / action chunk of the layer-2 tile (chunk 32): actor {1 1 0..}, critic {a0h a1h a0l a1l 1 1 0 0}
__device__ __forceinline__ uint4 tail_chunk_actor() { return make_uint4(ONES, 0u, 0u, 0u); }
__device__ __forceinline__ uint4 tail_chunk_critic(float a0, float a1) {
    const float h0 = bf16_round(a0), h1 = bf16_round(a1);
    return make_uint4(pack_bf16(h0, h1), pack_bf16(a0 - h0, a1 - h1), ONES, 0u);
}
__device__ __forceinline__ void load_obs(const float *obs, int64_t row, int64_t end, float4 (&x)[3]) {
    if (row < end) {
        const float4 *src = reinterpret_cast<const float4 *>(obs + row * DS);
        x[0] = __ldg(src); x[1] = __ldg(src + 1); x[2] = __ldg(src + 2);
    } else {
        x[0] = x[1] = x[2] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
}

// ---- weight staging ------------------------------------------------------------
struct Stager {
    const float *theta;      // flat parameter vector of the network
    uint8_t *b1, *b2;        // weight images in shared memory (zero-filled beforehand)
    float4 *w3x;             // layer 3.  actor: [64] float4 = W3[128][2] as stored; critic: [128] {W3[k], W3[k] W2[256][k], W3[k] W2[257][k], 0}
    float *b3;               // [2]
    bool noisy;
    float sd;
    uint64_t seed, counter;
    uint32_t group;
    // four consecutive parameters starting at p (p % 4 == 0), perturbed if asked (SkillshotLearner.py:260-265)
    __device__ __forceinline__ void perturb(int p, float4 &v) const {
        if (!noisy) return;
        float z[4];
        normal4_fast(seed, kTagParamNoise, (uint32_t)(p >> 2), group, counter, z);   // ~3e-6 off the float32 path's draw
        v.x += v.x * (sd * z[0]); v.y += v.y * (sd * z[1]); v.z += v.z * (sd * z[2]); v.w += v.w * (sd * z[3]);
    }
    __device__ __forceinline__ float4 load(int p) const { return __ldg(reinterpret_cast<const float4 *>(theta + p)); }
};

// Weights are [k][n] with n contiguous in HBM and [k/8][n][k%8] bf16 in shared memory.  A task takes
// one K chunk (8 rows) of four consecutive columns: 8 independent 16-byte loads (coalesced over the
// lanes), 8 Philox quads if the weights are perturbed, then one 16-byte store per column.
// WITH_L1 = false skips the layer-1 image (the frame-stacked actor builds its own wider one).
template <int NET, int NTHREADS, bool L1F16 = false, bool WITH_L1 = true>
__device__ __forceinline__ void stage_weights(const Stager &S) {
    constexpr int T_W2 = (H1 / 8) * (H2 / 4), T_W1 = WITH_L1 ? 2 * (H1 / 4) : 0, T_TAIL = H2 / 4;
    for (int t = threadIdx.x; t < T_W2 + T_W1 + T_TAIL + 1; t += NTHREADS) {
        if (t < T_W2) {
            const int kc = t / (H2 / 4), n = (t % (H2 / 4)) * 4;
            float4 v[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = S.load(P_W2 + (kc * 8 + i) * H2 + n);
#pragma unroll
            for (int i = 0; i < 8; ++i) S.perturb(P_W2 + (kc * 8 + i) * H2 + n, v[i]);
            uint8_t *dst = S.b2 + (uint32_t)(kc * H2 + n) * 16;
            *reinterpret_cast<uint4 *>(dst + 0) = make_uint4(pack_bf16(v[0].x, v[1].x), pack_bf16(v[2].x, v[3].x), pack_bf16(v[4].x, v[5].x), pack_bf16(v[6].x, v[7].x));
            *reinterpret_cast<uint4 *>(dst + 16) = make_uint4(pack_bf16(v[0].y, v[1].y), pack_bf16(v[2].y, v[3].y), pack_bf16(v[4].y, v[5].y), pack_bf16(v[6].y, v[7].y));
            *reinterpret_cast<uint4 *>(dst + 32) = make_uint4(pack_bf16(v[0].z, v[1].z), pack_bf16(v[2].z, v[3].z), pack_bf16(v[4].z, v[5].z), pack_bf16(v[6].z, v[7].z));
            *reinterpret_cast<uint4 *>(dst + 48) = make_uint4(pack_bf16(v[0].w, v[1].w), pack_bf16(v[2].w, v[3].w), pack_bf16(v[4].w, v[5].w), pack_bf16(v[6].w, v[7].w));
        } else if (t < T_W2 + T_W1) {
            // W1 rows 0..7 (chunk 0) or rows 8..11 + the bias pair b1 hi, lo at K = 12, 13 (chunk 1);
            // the same rows serve the low half of the observation two chunks further on
            const int tt = t - T_W2, kc = tt / (H1 / 4), n = (tt % (H1 / 4)) * 4;
            float4 v[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int k = kc * 8 + i;
                v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (k < DS) { v[i] = S.load(P_W1 + k * H1 + n); S.perturb(P_W1 + k * H1 + n, v[i]); }
            }
            uint32_t e45[4] = {0u, 0u, 0u, 0u};
            if (kc == 1) {
                float4 b = S.load(P_B1 + n);
                S.perturb(P_B1 + n, b);
                if (L1F16) { e45[0] = hi_lo_f16(b.x); e45[1] = hi_lo_f16(b.y); e45[2] = hi_lo_f16(b.z); e45[3] = hi_lo_f16(b.w); }
                else { e45[0] = hi_lo_bf16(b.x); e45[1] = hi_lo_bf16(b.y); e45[2] = hi_lo_bf16(b.z); e45[3] = hi_lo_bf16(b.w); }
            }
            uint8_t *dst = S.b1 + (uint32_t)(kc * H1 + n) * 16;
            const float c[4][8] = {{v[0].x, v[1].x, v[2].x, v[3].x, v[4].x, v[5].x, v[6].x, v[7].x},
                                   {v[0].y, v[1].y, v[2].y, v[3].y, v[4].y, v[5].y, v[6].y, v[7].y},
                                   {v[0].z, v[1].z, v[2].z, v[3].z, v[4].z, v[5].z, v[6].z, v[7].z},
                                   {v[0].w, v[1].w, v[2].w, v[3].w, v[4].w, v[5].w, v[6].w, v[7].w}};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (L1F16) {      // one fp16 image, K = 16
                    const uint32_t w01 = pack_f16(c[j][0], c[j][1]), w23 = pack_f16(c[j][2], c[j][3]);
                    const uint32_t w45 = pack_f16(c[j][4], c[j][5]), w67 = pack_f16(c[j][6], c[j][7]);
                    *reinterpret_cast<uint4 *>(dst + j * 16) = make_uint4(w01, w23, kc == 1 ? e45[j] : w45, w67);
                } else {          // bf16 image against the high and the low half of the observation, K = 32
                    const uint32_t w01 = pack_bf16(c[j][0], c[j][1]), w23 = pack_bf16(c[j][2], c[j][3]);
                    const uint32_t w45 = pack_bf16(c[j][4], c[j][5]), w67 = pack_bf16(c[j][6], c[j][7]);
                    *reinterpret_cast<uint4 *>(dst + j * 16) = make_uint4(w01, w23, kc == 1 ? e45[j] : w45, w67);
                    *reinterpret_cast<uint4 *>(dst + j * 16 + 2 * CHUNK_B1) = make_uint4(w01, w23, kc == 1 ? 0u : w45, w67);
                }
            }
        } else if (t < T_W2 + T_W1 + T_TAIL) {
            // four hidden-2 units n..n+3: b2 (and the critic's two action rows of W2) -> chunk 32 of B2; layer 3
            const int n = (t - T_W2 - T_W1) * 4;
            uint8_t *dst = S.b2 + (uint32_t)((H1 / 8) * H2 + n) * 16;
            if (NET == NET_ACTOR) {
                float4 b = S.load(A_B2 + n);
                S.perturb(A_B2 + n, b);
                const float bb[4] = {b.x, b.y, b.z, b.w};
                float4 wa = S.load(A_W3 + 2 * n), wb = S.load(A_W3 + 2 * n + 4);        // W3[n..n+3][0..1]
                S.perturb(A_W3 + 2 * n, wa);
                S.perturb(A_W3 + 2 * n + 4, wb);
#pragma unroll
                for (int j = 0; j < 4; ++j) *reinterpret_cast<uint4 *>(dst + j * 16) = make_uint4(hi_lo_bf16(bb[j]), 0u, 0u, 0u);
                S.w3x[n / 2] = wa;
                S.w3x[n / 2 + 1] = wb;
            } else {
                const float4 b = S.load(C_B2 + n), r0 = S.load(P_W2 + H1 * H2 + n), r1 = S.load(P_W2 + (H1 + 1) * H2 + n);
                const float4 w3 = S.load(C_W3 + n);
                const float bb[4] = {b.x, b.y, b.z, b.w}, a0[4] = {r0.x, r0.y, r0.z, r0.w}, a1[4] = {r1.x, r1.y, r1.z, r1.w};
                const float ww[4] = {w3.x, w3.y, w3.z, w3.w};
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const uint32_t a01 = pack_bf16(a0[j], a1[j]);
                    *reinterpret_cast<uint4 *>(dst + j * 16) = make_uint4(a01, a01, hi_lo_bf16(bb[j]), 0u);
                    S.w3x[n + j] = make_float4(ww[j], ww[j] * a0[j], ww[j] * a1[j], 0.f);
                }
            }
        } else {                                     // b3
            if (NET == NET_ACTOR) {
                float4 w = make_float4(S.theta[A_B3], S.theta[A_B3 + 1], 0.f, 0.f);
                S.perturb(A_B3, w);
                S.b3[0] = w.x; S.b3[1] = w.y;
            } else {
                S.b3[0] = S.theta[C_B3]; S.b3[1] = 0.f;
            }
        }
    }
}

// ---- launchers shared between translation units (host side) ------------------------------------
// frames_l1_kernel (ss_frames_tc.cu) alone: H1 tiles of `params`' first layer from fp16 operand tiles whose columns are in
// frame order (the layout ss_obs_stack_push_tc writes with ring head = frames - 1)
int frames_layer1_tc(const float *params, const void *xt, int frames, int64_t n, void *h1, cudaStream_t st);
// reduce_parts_kernel (ss_mlp_grad_tc.cu): grad[p] = fixed-order sum of `parts` slices of n_params + 1 floats, aux = extra slot
int reduce_slices(const float *work, int parts, int n_params, float *grad, float *aux, cudaStream_t st);
// the TD3 target's two CUDA-core steps around the tensor-core forwards (ss_mlp_grad_tc.cu): td3_smooth (ss_rng.cuh) on the
// target actions act[n][2] of global rows row_offset.., in place; y = reward + gamma (1 - done) min(q1, q2)
int td3_smooth_actions(float *act, int64_t n, float sigma, float clip, uint64_t seed, uint64_t counter, int64_t row_offset,
                       cudaStream_t st);
int td3_min_target(const float *q1, const float *q2, const float *reward, const uint8_t *done, float gamma, float *y, int64_t n,
                   cudaStream_t st);

}  // namespace sstc
