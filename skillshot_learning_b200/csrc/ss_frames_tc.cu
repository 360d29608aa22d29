// ss_frames_tc.cu -- the frame-stacked planning actor on the tensor cores (tcgen05.mma, sm_100a).
//
// BASELINE.json configs[4] / readme.md:18-20 of the reference (no reference code): the actor of
// model_define_actor (SkillshotLearner.py:70-96) fed the last `frames` observations of a player,
// oldest first: 12 * frames -> 256 relu -> 128 relu -> 2 tanh.  With 20 frames layer 1 is a real
// GEMM (K = 240, 76 % of the MACs) and its weight image alone takes 128 KB of shared memory, so the
// three layers cannot share one resident CTA the way ss_mlp_tc.cu's do.  Two kernels:
//
//   frames_l1_kernel    H1[tile] = relu(X[128 x K1] . W1'[K1 x 256])      fp16 operands, fp32 accumulate
//       W1' stays resident (K1 = 12 * frames + bias rows, padded to 16: 256 for 20 frames).  The history
//       ring of this path is kept in HBM as fp16 tiles already in the tensor core's operand layout
//       (ss_obs_stack_push_tc), columns in ring-slot order; the rotation that makes the network see the
//       oldest frame first is applied to W1's rows while staging instead.  One thread streams each tile
//       in with four 16 KB bulk copies (a ring of 64-column K stages), the MMA warp consumes a stage
//       while the next ones land, accumulating into one of two 256-column tensor-memory buffers; four
//       epilogue warps drain the other buffer -> ReLU -> bf16 -> the tile's layer-2 operand image in global
//       memory (64 KB per tile, the exact shared-memory layout of ss_tc_common.cuh).
//       (A first version gathered fp32 rows with eight loader warps and converted in registers: 55 us per
//       131,072 rows, bound by the 64 KB of loads a CTA's registers can keep in flight.)
//   frames_l23_kernel   act = tanh(relu(H1 . W2') . W3 + b3)
//       W2' resident; one thread streams the 64 KB operand images back with cp.async.bulk into a
//       two-slot ring (they were written moments earlier and mostly still sit in the 126 MB L2), the MMA
//       warp runs the 17-step layer-2 chain into one of two accumulators, four warps do the 128 -> 2
//       layer and tanh in fp32 from the other.
//
// Parameter noise (SkillshotLearner.py:260-265): the caller passes one perturbed parameter vector per
// noise group (ss_param_noise_groups); a CTA restages its weights when its tiles cross into the next
// group, and the launch gives every CTA exactly one group when the groups fit the SMs.
//
// Precision as in ss_mlp_tc.cu: observations and W1 in fp16 (11-bit significands), hidden layer 1
// and W2 in bf16, biases as high + low pairs against constant-one K columns, fp32 accumulation;
// results agree with ss_actor_forward_frames (the exact float32 path) to about 1e-2 on the action.
#include "ss_tc_common.cuh"

namespace {

using namespace sstc;

constexpr int MAXF = SS_MAX_FRAMES;
constexpr int K1MAX = (DS * MAXF + 2 + 15) / 16 * 16;       // 256
constexpr int KSTAGE = 64, NSTAGE = K1MAX / KSTAGE;         // the X ring: four K stages of 64 columns
constexpr uint32_t W1IMG_BYTES = (K1MAX / 8) * CHUNK_B1;    // 131,072
constexpr uint32_t XSTAGE_BYTES = (KSTAGE / 8) * CHUNK_A;   // 16,384
constexpr uint32_t H1TILE_BYTES = (H1 / 8) * CHUNK_A;       // 65,536: hidden layer 1 of one tile as a layer-2 operand

struct FramesArgs {
    const float *theta;          // [groups][stride] parameter vectors (stride 0: one vector)
    const uint8_t *xt;           // history tiles [tile][k1 / 8][128][8] fp16, columns in ring (slot-major) order
    float *act;                  // [n][2]
    uint8_t *h1;                 // [units][H1TILE_BYTES] scratch between the two kernels
    int64_t n, group, stride, head;
    int frames;
};

__host__ __device__ constexpr int frames_k1(int frames) { return (DS * frames + 2 + 15) / 16 * 16; }

// L2 policies.  The hidden tiles written by the layer-1 kernel are read back by the layer-2/3 kernel moments later: at
// 131,072 rows they are 67 MB and fit the 126 MB L2 if the 67 MB of history that streams through beside them does not
// push them out, which saves their round trip to HBM (two thirds of the traffic of the pair of kernels).
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ void bulk_load_hint(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar, uint64_t policy) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar), "l"(policy)
                 : "memory");
}
__device__ __forceinline__ void st_global_hint(void *p, uint4 v, uint64_t policy) {
    asm volatile("st.global.L2::cache_hint.v4.b32 [%0], {%1, %2, %3, %4}, %5;" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w), "l"(policy)
                 : "memory");
}
// 32 accumulator columns -> ReLU -> bf16 -> four 16-byte chunks of this thread's row of a 128-row tile in global memory
__device__ __forceinline__ void relu_pack_store_global(const uint32_t (&v)[32], uint8_t *dst, uint64_t policy) {
#pragma unroll
    for (int c = 0; c < 4; ++c)
        st_global_hint(dst + c * CHUNK_A,
                       make_uint4(pack_relu_bf16(__uint_as_float(v[c * 8 + 0]), __uint_as_float(v[c * 8 + 1])),
                                  pack_relu_bf16(__uint_as_float(v[c * 8 + 2]), __uint_as_float(v[c * 8 + 3])),
                                  pack_relu_bf16(__uint_as_float(v[c * 8 + 4]), __uint_as_float(v[c * 8 + 5])),
                                  pack_relu_bf16(__uint_as_float(v[c * 8 + 6]), __uint_as_float(v[c * 8 + 7]))),
                       policy);
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}

struct Units {                   // tiles as (noise group, tile in group) pairs, split evenly over the CTAs
    int64_t upg, u0, u1;
    int64_t group, n;
    __device__ Units(const FramesArgs &A) : group(A.group), n(A.n) {
        upg = (A.group + TM - 1) / TM;
        const int64_t units = ((A.n + A.group - 1) / A.group) * upg;
        u0 = units * blockIdx.x / gridDim.x;
        u1 = units * (blockIdx.x + 1) / gridDim.x;
    }
    __device__ int64_t row0(int64_t u) const { const int64_t g = u / upg; return g * group + (u - g * upg) * TM; }
    __device__ int64_t end(int64_t u) const { return min(n, (u / upg + 1) * group); }
};

// ---------------------------------------------------------------------------------------------
// layer 1
// ---------------------------------------------------------------------------------------------
namespace l1 {

constexpr int EPI_WARPS = 4, MMA_W = 4, COPY_W = 5, NTH = 32 * 12;    // warps 6..11 only help to stage the weights
constexpr uint32_t SM_W1 = 0;
constexpr uint32_t SM_X = SM_W1 + W1IMG_BYTES;              // NSTAGE x [8][128][8] fp16
constexpr uint32_t SM_BAR = SM_X + NSTAGE * XSTAGE_BYTES;
constexpr int B_XFULL = 0, B_XFREE = NSTAGE, B_DFULL = 2 * NSTAGE, B_DFREE = 2 * NSTAGE + 2, B_COUNT = 2 * NSTAGE + 4;
constexpr uint32_t SM_TMEM = SM_BAR + B_COUNT * 8;
constexpr uint32_t SM_TOTAL = SM_TMEM + 16;
static_assert(SM_TOTAL <= 227 * 1024, "shared memory budget");

// W1' image [k1 / 8][256][8] fp16.  The history tiles keep their columns in RING order (slot-major), so the
// image's K rows are W1's rows rotated the same way: image row 12 slot + j = W1 row 12 f + j with
// f = (slot - oldest) mod frames, the frame's age rank (0 = oldest).  Rows kx, kx + 1 = b1 high, low.
__device__ __forceinline__ void stage_w1(const float *theta, int frames, int oldest, int k1, uint8_t *img) {
    const int kx = DS * frames, tasks = (k1 / 8) * (H1 / 4);
    // a task = one K chunk (8 rows) of four consecutive units: 8 independent 16-byte loads; two tasks are kept in flight
    auto load = [&](int t, float4 (&v)[8]) {
        const int kc = t / (H1 / 4), n = (t % (H1 / 4)) * 4;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int k = kc * 8 + i;
            v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (k < kx) {
                const int slot = k / DS, j = k - slot * DS;
                int f = slot - oldest;
                if (f < 0) f += frames;
                v[i] = __ldg(reinterpret_cast<const float4 *>(theta + (int64_t)(f * DS + j) * H1 + n));
            } else if (k <= kx + 1) {
                v[i] = __ldg(reinterpret_cast<const float4 *>(theta + (int64_t)kx * H1 + n));      // b1
            }
        }
    };
    auto store = [&](int t, float4 (&v)[8]) {
        const int kc = t / (H1 / 4), n = (t % (H1 / 4)) * 4;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int k = kc * 8 + i;
            if (k == kx || k == kx + 1) {                   // bias pair: hi at kx, lo at kx + 1
                const float b[4] = {v[i].x, v[i].y, v[i].z, v[i].w};
                float o[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float hi = __half2float(__float2half_rn(b[j]));
                    o[j] = k == kx ? hi : b[j] - hi;
                }
                v[i] = make_float4(o[0], o[1], o[2], o[3]);
            }
        }
        uint8_t *dst = img + (uint32_t)(kc * H1 + n) * 16;
        *reinterpret_cast<uint4 *>(dst + 0) = make_uint4(pack_f16(v[0].x, v[1].x), pack_f16(v[2].x, v[3].x), pack_f16(v[4].x, v[5].x), pack_f16(v[6].x, v[7].x));
        *reinterpret_cast<uint4 *>(dst + 16) = make_uint4(pack_f16(v[0].y, v[1].y), pack_f16(v[2].y, v[3].y), pack_f16(v[4].y, v[5].y), pack_f16(v[6].y, v[7].y));
        *reinterpret_cast<uint4 *>(dst + 32) = make_uint4(pack_f16(v[0].z, v[1].z), pack_f16(v[2].z, v[3].z), pack_f16(v[4].z, v[5].z), pack_f16(v[6].z, v[7].z));
        *reinterpret_cast<uint4 *>(dst + 48) = make_uint4(pack_f16(v[0].w, v[1].w), pack_f16(v[2].w, v[3].w), pack_f16(v[4].w, v[5].w), pack_f16(v[6].w, v[7].w));
    };
    for (int t = threadIdx.x; t < tasks; t += 2 * NTH) {
        float4 va[8], vb[8];
        load(t, va);
        if (t + NTH < tasks) load(t + NTH, vb);
        store(t, va);
        if (t + NTH < tasks) store(t + NTH, vb);
    }
}

__global__ void __launch_bounds__(NTH, 1) frames_l1_kernel(const FramesArgs A) {
    extern __shared__ __align__(128) uint8_t smem[];
    const uint32_t sbase = smem_u32(smem);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    auto bar = [&](int idx) -> uint32_t { return sbase + SM_BAR + (uint32_t)idx * 8; };
    const int k1 = frames_k1(A.frames);                     // input columns + bias pair, padded to the MMA K step
    const int nstages = (k1 + KSTAGE - 1) / KSTAGE;         // K stages in use (the last one may be partial)
    const uint32_t tile_bytes = (uint32_t)(k1 / 8) * CHUNK_A;
    const int oldest = (int)((A.head + 1) % A.frames);      // ring slot of the oldest frame

    if (threadIdx.x == 0) {
        for (int s = 0; s < NSTAGE; ++s) {
            mbar_init(bar(B_XFULL + s), 1);
            mbar_init(bar(B_XFREE + s), 1);
        }
        for (int h = 0; h < 2; ++h) {
            mbar_init(bar(B_DFULL + h), 1);
            mbar_init(bar(B_DFREE + h), 32 * EPI_WARPS);
        }
        mbar_fence_init();
    }
    if (warp == MMA_W) tmem_alloc(sbase + SM_TMEM, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *reinterpret_cast<const volatile uint32_t *>(smem + SM_TMEM);

    const Units U(A);
    uint32_t tcount = 0;                                    // tiles this CTA has started: parities derive from it
    for (int64_t u = U.u0; u < U.u1;) {
        const int64_t g = u / U.upg;
        const int64_t seg_end = min(U.u1, (g + 1) * U.upg);
        const uint32_t ntiles = (uint32_t)(seg_end - u);
        stage_w1(A.theta + g * A.stride, A.frames, oldest, k1, smem + SM_W1);
        fence_proxy_async();
        __syncthreads();

        if (warp < EPI_WARPS) {
            // ============ epilogue: D[slot] -> ReLU -> bf16 -> the tile's layer-2 operand image ============
            const int r = warp * 32 + lane;
            const uint32_t tl = tmem + ((uint32_t)(warp * 32) << 16);
            const uint64_t keep = l2_policy_evict_last();
            for (uint32_t i = 0; i < ntiles; ++i) {
                const uint32_t tc = tcount + i, slot = tc & 1;
                uint8_t *out = A.h1 + (u + i) * (int64_t)H1TILE_BYTES + r * 16;
                mbar_wait(bar(B_DFULL + slot), (tc >> 1) & 1);
                tc_fence_after();
                uint32_t va[32], vb[32];
                tmem_ld32(tl + slot * 256, va);
#pragma unroll
                for (int j = 0; j < H1 / 32; j += 2) {
                    tmem_wait_ld();
                    tmem_ld32(tl + slot * 256 + (j + 1) * 32, vb);
                    relu_pack_store_global(va, out + (uint32_t)(j * 4) * CHUNK_A, keep);
                    tmem_wait_ld();
                    if (j + 2 < H1 / 32) tmem_ld32(tl + slot * 256 + (j + 2) * 32, va);
                    else { tc_fence_before(); mbar_arrive(bar(B_DFREE + slot)); }        // D[slot] fully read
                    relu_pack_store_global(vb, out + (uint32_t)((j + 1) * 4) * CHUNK_A, keep);
                }
            }
        } else if (warp == MMA_W) {
            // ============ the MMA-issuing warp ============
            constexpr uint32_t kI = umma_idesc_f16(TM, H1);
            const uint64_t xd = desc_kmajor(sbase + SM_X, CHUNK_A), wd = desc_kmajor(sbase + SM_W1, CHUNK_B1);
            const uint32_t tc0 = __shfl_sync(0xffffffffu, tcount, 0);
            // The tensor pipe queues only a couple of MMAs, so the issuing thread cannot run ahead: whatever it waits for
            // idles the pipe unless MMAs are queued behind it.  Every wait (next stage landed, next accumulator drained) is
            // therefore placed BETWEEN the two halves of a stage's MMAs, and the commits after them.
            mbar_wait(bar(B_DFREE + (tc0 & 1)), ((tc0 >> 1) & 1) ^ 1);
            mbar_wait(bar(B_XFULL + 0), tc0 & 1);
            tc_fence_after();
            for (uint32_t i = 0; i < ntiles; ++i) {
                const uint32_t tc = tc0 + i, slot = tc & 1;
                const uint32_t d = tmem + slot * 256;
#pragma unroll
                for (int sg = 0; sg < NSTAGE; ++sg) {             // unrolled: descriptor offsets and flags fold to constants --
                    if (sg >= nstages) break;                     // a single thread's issue loop must stay a few instructions per MMA
                    const int steps = min(KSTAGE, k1 - sg * KSTAGE) / 16;
                    if (lane == 0) {
#pragma unroll
                        for (int ks = 0; ks < 2; ++ks)
                            if (ks < steps)
                                umma_bf16(d, desc_advance(xd, sg * XSTAGE_BYTES + 2 * CHUNK_A * ks),
                                          desc_advance(wd, (uint32_t)(sg * (KSTAGE / 8) + 2 * ks) * CHUNK_B1), kI, (sg | ks) != 0);
                    }
                    __syncwarp();
                    if (sg + 1 < nstages) {
                        mbar_wait(bar(B_XFULL + sg + 1), tc & 1);
                    } else if (i + 1 < ntiles) {
                        mbar_wait(bar(B_DFREE + (slot ^ 1)), (((tc + 1) >> 1) & 1) ^ 1);      // the epilogue has drained the other D
                        mbar_wait(bar(B_XFULL + 0), (tc + 1) & 1);
                    }
                    tc_fence_after();
                    if (lane == 0) {
#pragma unroll
                        for (int ks = 2; ks < KSTAGE / 16; ++ks)
                            if (ks < steps)
                                umma_bf16(d, desc_advance(xd, sg * XSTAGE_BYTES + 2 * CHUNK_A * ks),
                                          desc_advance(wd, (uint32_t)(sg * (KSTAGE / 8) + 2 * ks) * CHUNK_B1), kI, 1);
                        umma_commit(bar(B_XFREE + sg));
                        if (sg == nstages - 1) umma_commit(bar(B_DFULL + slot));
                    }
                    __syncwarp();
                }
            }
        } else if (warp == COPY_W && lane == 0) {
            // ============ the copy thread: K stages of the history tiles -> X ring ============
            const uint64_t stream_through = l2_policy_evict_first();
            for (uint32_t i = 0; i < ntiles; ++i) {
                const uint32_t tc = tcount + i;
                const uint8_t *src = A.xt + (u + i) * (int64_t)tile_bytes;
                for (int sg = 0; sg < nstages; ++sg) {
                    const uint32_t bytes = (uint32_t)min(KSTAGE, k1 - sg * KSTAGE) / 8 * CHUNK_A;
                    mbar_wait(bar(B_XFREE + sg), (tc & 1) ^ 1);       // the previous tile's MMAs have read this stage
                    mbar_expect_tx(bar(B_XFULL + sg), bytes);
                    bulk_load_hint(sbase + SM_X + sg * XSTAGE_BYTES, src + sg * XSTAGE_BYTES, bytes, bar(B_XFULL + sg), stream_through);
                }
            }
        }
        tcount += ntiles;
        u = seg_end;
        tc_fence_before();
        __syncthreads();                   // every role has finished the segment: the weight image may be replaced
        tc_fence_after();
    }
    if (warp == MMA_W) tmem_dealloc(tmem, 512);
}

}  // namespace l1

// ---------------------------------------------------------------------------------------------
// layers 2 and 3
// ---------------------------------------------------------------------------------------------
namespace l23 {

constexpr int Q_WARPS = 4, MMA_W = 4, NTH = 32 * 6;          // warp 5: the copy thread
constexpr uint32_t SM_B2 = 0;
constexpr uint32_t SM_A1 = SM_B2 + B2_BYTES;                // 2 x [K2/8][128][8] bf16: hidden layer 1 + constant tail
constexpr uint32_t SM_W3 = SM_A1 + 2 * X2_BYTES;
constexpr uint32_t SM_B3 = SM_W3 + H2 * 16;
constexpr uint32_t SM_BAR = SM_B3 + 16;
constexpr int B_AFULL = 0, B_AFREE = 2, B_DFULL = 4, B_DFREE = 6, B_COUNT = 8;
constexpr uint32_t SM_TMEM = SM_BAR + B_COUNT * 8;
constexpr uint32_t SM_TOTAL = SM_TMEM + 16;
static_assert(SM_TOTAL <= 227 * 1024, "shared memory budget");

__global__ void __launch_bounds__(NTH, 1) frames_l23_kernel(const FramesArgs A) {
    extern __shared__ __align__(128) uint8_t smem[];
    const uint32_t sbase = smem_u32(smem);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    auto bar = [&](int idx) -> uint32_t { return sbase + SM_BAR + (uint32_t)idx * 8; };

    if (threadIdx.x == 0) {
        for (int s = 0; s < 2; ++s) {
            mbar_init(bar(B_AFULL + s), 1);
            mbar_init(bar(B_AFREE + s), 1);
            mbar_init(bar(B_DFULL + s), 1);
            mbar_init(bar(B_DFREE + s), 32 * Q_WARPS);
        }
        mbar_fence_init();
    }
    if (warp == MMA_W) tmem_alloc(sbase + SM_TMEM, 256);
    for (uint32_t o = threadIdx.x * 16; o < SM_A1; o += NTH * 16) *reinterpret_cast<uint4 *>(smem + o) = make_uint4(0, 0, 0, 0);
    if (threadIdx.x < TM) {                                 // constant tail chunks of both slots: {1 1 0 ..} | 0
        for (int s = 0; s < 2; ++s) {
            uint8_t *arow = smem + SM_A1 + s * X2_BYTES + threadIdx.x * 16;
            *reinterpret_cast<uint4 *>(arow + (H1 / 8) * CHUNK_A) = tail_chunk_actor();
            *reinterpret_cast<uint4 *>(arow + (H1 / 8 + 1) * CHUNK_A) = make_uint4(0, 0, 0, 0);
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *reinterpret_cast<const volatile uint32_t *>(smem + SM_TMEM);
    // the parameters after W1 are laid out as in the single-frame actor: shift the base so the shared offsets apply
    const int64_t shift = (int64_t)(A.frames - 1) * DS * H1;

    const Units U(A);
    uint32_t tcount = 0;
    for (int64_t u = U.u0; u < U.u1;) {
        const int64_t g = u / U.upg;
        const int64_t seg_end = min(U.u1, (g + 1) * U.upg);
        const uint32_t ntiles = (uint32_t)(seg_end - u);
        stage_weights<NET_ACTOR, NTH, true, false>(Stager{A.theta + g * A.stride + shift, nullptr, smem + SM_B2,
                                                          reinterpret_cast<float4 *>(smem + SM_W3),
                                                          reinterpret_cast<float *>(smem + SM_B3), false, 0.f, 0, 0, 0});
        fence_proxy_async();
        __syncthreads();

        if (warp < Q_WARPS) {
            // ============ output warps: layer 3 + tanh on D[slot] ============
            const int r = warp * 32 + lane;
            const uint32_t tl = tmem + ((uint32_t)(warp * 32) << 16);
            const float4 *w3x = reinterpret_cast<const float4 *>(smem + SM_W3);
            const float *b3 = reinterpret_cast<const float *>(smem + SM_B3);
            const int64_t seg_row = U.row0(u) + r, end = U.end(u);        // a segment stays inside one noise group
            for (uint32_t i = 0; i < ntiles; ++i) {
                const uint32_t tc = tcount + i, slot = tc & 1;
                const int64_t row = seg_row + (int64_t)i * TM;
                mbar_wait(bar(B_DFULL + slot), (tc >> 1) & 1);
                tc_fence_after();
                float acc[2][4] = {{b3[0], 0.f, 0.f, 0.f}, {b3[1], 0.f, 0.f, 0.f}};
                uint32_t va[32], vb[32];
                auto layer3 = [&](const uint32_t (&v)[32], const float4 *w) {
#pragma unroll
                    for (int c = 0; c < 16; ++c) {
                        const float4 ww = w[c];                                  // W3[2c][0..1], W3[2c+1][0..1]
                        const float ha = fmaxf(__uint_as_float(v[c * 2 + 0]), 0.f), hb = fmaxf(__uint_as_float(v[c * 2 + 1]), 0.f);
                        acc[0][(c & 1) * 2 + 0] = fmaf(ha, ww.x, acc[0][(c & 1) * 2 + 0]);
                        acc[1][(c & 1) * 2 + 0] = fmaf(ha, ww.y, acc[1][(c & 1) * 2 + 0]);
                        acc[0][(c & 1) * 2 + 1] = fmaf(hb, ww.z, acc[0][(c & 1) * 2 + 1]);
                        acc[1][(c & 1) * 2 + 1] = fmaf(hb, ww.w, acc[1][(c & 1) * 2 + 1]);
                    }
                };
                tmem_ld32(tl + slot * 128, va);
#pragma unroll
                for (int j = 0; j < H2 / 32; j += 2) {
                    tmem_wait_ld();
                    tmem_ld32(tl + slot * 128 + (j + 1) * 32, vb);
                    layer3(va, w3x + j * 16);
                    tmem_wait_ld();
                    if (j + 2 < H2 / 32) tmem_ld32(tl + slot * 128 + (j + 2) * 32, va);
                    else { tc_fence_before(); mbar_arrive(bar(B_DFREE + slot)); }
                    layer3(vb, w3x + (j + 1) * 16);
                }
                if (row < end)
                    reinterpret_cast<float2 *>(A.act)[row] = make_float2(tanhf((acc[0][0] + acc[0][1]) + (acc[0][2] + acc[0][3])),
                                                                         tanhf((acc[1][0] + acc[1][1]) + (acc[1][2] + acc[1][3])));
            }
        } else if (warp == MMA_W) {
            constexpr uint32_t kI = umma_idesc(TM, H2);
            const uint64_t ad = desc_kmajor(sbase + SM_A1, CHUNK_A), bd = desc_kmajor(sbase + SM_B2, CHUNK_B2);
            const uint32_t tc0 = __shfl_sync(0xffffffffu, tcount, 0);
            for (uint32_t i = 0; i < ntiles; ++i) {
                const uint32_t tc = tc0 + i, slot = tc & 1;
                mbar_wait(bar(B_DFREE + slot), ((tc >> 1) & 1) ^ 1);
                mbar_wait(bar(B_AFULL + slot), (tc >> 1) & 1);
                tc_fence_after();
                if (lane == 0) {
#pragma unroll
                    for (int ks = 0; ks < K2 / 16; ++ks)
                        umma_bf16(tmem + slot * 128, desc_advance(ad, slot * X2_BYTES + 2 * CHUNK_A * ks),
                                  desc_advance(bd, 2 * CHUNK_B2 * ks), kI, ks > 0);
                    umma_commit(bar(B_AFREE + slot));
                    umma_commit(bar(B_DFULL + slot));
                }
                __syncwarp();
            }
        } else if (lane == 0) {
            // ============ the copy thread: operand images of the tiles -> A1 ring ============
            const uint64_t last_use = l2_policy_evict_first();
            for (uint32_t i = 0; i < ntiles; ++i) {
                const uint32_t tc = tcount + i, slot = tc & 1;
                mbar_wait(bar(B_AFREE + slot), ((tc >> 1) & 1) ^ 1);  // the MMAs that read this slot have retired
                mbar_expect_tx(bar(B_AFULL + slot), H1TILE_BYTES);
                const uint8_t *src = A.h1 + (u + i) * (int64_t)H1TILE_BYTES;
#pragma unroll
                for (int p = 0; p < 4; ++p)
                    bulk_load_hint(sbase + SM_A1 + slot * X2_BYTES + p * (H1TILE_BYTES / 4), src + p * (H1TILE_BYTES / 4), H1TILE_BYTES / 4,
                                   bar(B_AFULL + slot), last_use);
            }
        }
        tcount += ntiles;
        u = seg_end;
        tc_fence_before();
        __syncthreads();
        tc_fence_after();
    }
    if (warp == MMA_W) tmem_dealloc(tmem, 256);
}

}  // namespace l23

int64_t frame_units(int64_t n, int64_t group) { return ((n + group - 1) / group) * ((group + TM - 1) / TM); }

// newest observation -> ring slot `slot` of every row's history (fp16, operand layout); a row whose game has just
// restarted gets it in every slot.  Also (re)writes the constant-one pair that multiplies the bias rows.
__global__ void obs_stack_push_tc_kernel(uint8_t *xt, int64_t n_rows, int frames, int slot, uint32_t tile_bytes, const float *obs,
                                         const uint8_t *done, int done_div) {
    const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n_rows) return;
    const float4 *src = reinterpret_cast<const float4 *>(obs + row * DS);
    const float4 a = __ldg(src), b = __ldg(src + 1), c = __ldg(src + 2);
    const uint32_t h[6] = {pack_f16(a.x, a.y), pack_f16(a.z, a.w), pack_f16(b.x, b.y), pack_f16(b.z, b.w), pack_f16(c.x, c.y), pack_f16(c.z, c.w)};
    uint8_t *base = xt + (row / TM) * (int64_t)tile_bytes + (row % TM) * 16;
    auto put = [&](int s) {                                 // columns 12 s .. 12 s + 11: 24 bytes starting 0 or 8 bytes into a chunk
        uint8_t *p = base + (uint32_t)((DS * s) >> 3) * CHUNK_A;
        if ((s & 1) == 0) {
            *reinterpret_cast<uint4 *>(p) = make_uint4(h[0], h[1], h[2], h[3]);
            *reinterpret_cast<uint2 *>(p + CHUNK_A) = make_uint2(h[4], h[5]);
        } else {
            *reinterpret_cast<uint2 *>(p + 8) = make_uint2(h[0], h[1]);
            *reinterpret_cast<uint4 *>(p + CHUNK_A) = make_uint4(h[2], h[3], h[4], h[5]);
        }
    };
    if (done && done[row / done_div]) {
        for (int s = 0; s < frames; ++s) put(s);
    } else {
        put(slot);
    }
    const int kx = DS * frames;                             // {1, 1} at columns kx, kx + 1
    *reinterpret_cast<uint32_t *>(base + (uint32_t)(kx >> 3) * CHUNK_A + (kx & 7) * 2) = 0x3C003C00u;
}

// The learner's history step of a pool tick (ss_obs_stack_push_pool): obs_stack_push_tc_kernel, obs_stack_push_kernel and
// obs_stack_ordered_kernel for the L learner rows in one pass, with each row's restart flag found by the pool row rule.
// Thread (row, f, part) owns float4 `part` of frame f of the row's ordered output (oldest first), i.e. ring slot
// (newest + 1 + f) % frames: it takes the newest observation when that slot is the newest one or the game restarted (and then
// stores it in both histories), the float32 history's value otherwise, and writes it to the ordered row(s).  So every
// history slot is read at most once and the ordered rows are written straight from registers.  blockIdx.y selects a chunk
// of PUSH_CHUNK rows, so the index arithmetic within a chunk is 32-bit; `newest` = head % frames comes from the host.
constexpr int64_t PUSH_CHUNK = 1 << 20;

__global__ void obs_stack_push_pool_kernel(uint8_t *xt, float *stack32, int64_t n_rows, int64_t S, int frames, int newest,
                                           uint32_t tile_bytes, const float *obs, const uint8_t *done, float *rows_out,
                                           float *rows_out2) {
    const uint32_t w4 = 3 * frames, t = blockIdx.x * blockDim.x + threadIdx.x, local = t / w4;
    const int64_t row = (int64_t)blockIdx.y * PUSH_CHUNK + local;
    if (local >= PUSH_CHUNK || row >= n_rows) return;
    const int q = (int)(t - local * w4), f = q / 3, part = q - 3 * f;
    int slot = newest + 1 + f;
    if (slot >= frames) slot -= frames;
    const int64_t env = row < 2 * S ? row >> 1 : row - S;
    const bool restart = done && done[env];
    float4 *h = reinterpret_cast<float4 *>(stack32) + (row * frames + slot) * 3 + part;
    float4 v;
    if (restart || slot == newest) {
        v = __ldg(reinterpret_cast<const float4 *>(obs) + row * 3 + part);
        *h = v;
        if (xt) {                                           // the same 8 bytes obs_stack_push_tc_kernel's put() stores
            const int c = DS * slot + 4 * part;
            *reinterpret_cast<uint2 *>(xt + (row / TM) * (int64_t)tile_bytes + (row % TM) * 16 + (uint32_t)(c >> 3) * CHUNK_A +
                                       (c & 7) * 2) = make_uint2(pack_f16(v.x, v.y), pack_f16(v.z, v.w));
        }
    } else {
        v = *h;
    }
    if (xt && q == 0) {
        const int kx = DS * frames;
        *reinterpret_cast<uint32_t *>(xt + (row / TM) * (int64_t)tile_bytes + (row % TM) * 16 + (uint32_t)(kx >> 3) * CHUNK_A +
                                      (kx & 7) * 2) = 0x3C003C00u;
    }
    const int64_t e = row * w4 + q;
    reinterpret_cast<float4 *>(rows_out)[e] = v;
    if (rows_out2) reinterpret_cast<float4 *>(rows_out2)[e] = v;
}

}  // namespace

int sstc::frames_layer1_tc(const float *params, const void *xt, int frames, int64_t n, void *h1, cudaStream_t st) {
    FramesArgs A{params, (const uint8_t *)xt, nullptr, (uint8_t *)h1, n, n, 0, frames - 1, frames};
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return SS_ERR_CUDA;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return SS_ERR_CUDA;
    const int64_t units = frame_units(n, n);
    if (cudaFuncSetAttribute(l1::frames_l1_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)l1::SM_TOTAL) != cudaSuccess)
        return SS_ERR_CUDA;
    l1::frames_l1_kernel<<<(int)(units < sms ? units : sms), l1::NTH, l1::SM_TOTAL, st>>>(A);
    return cudaGetLastError() == cudaSuccess ? SS_OK : SS_ERR_CUDA;
}

extern "C" int64_t ss_obs_stack_tc_bytes(int64_t n_rows, int frames) {
    if (n_rows <= 0 || frames < 1 || frames > MAXF) return -1;
    return (n_rows + TM - 1) / TM * (int64_t)(frames_k1(frames) / 8) * CHUNK_A;
}

extern "C" int ss_obs_stack_push_tc(void *stack_tc, int64_t n_rows, int frames, int64_t head, const float *obs, const uint8_t *done,
                                    int done_div, void *stream) {
    if (!stack_tc || !obs || n_rows <= 0 || frames < 1 || frames > MAXF || head < 0 || done_div < 1) return SS_ERR_INVALID_ARG;
    if (((uintptr_t)stack_tc | (uintptr_t)obs) & 15) return SS_ERR_INVALID_ARG;
    obs_stack_push_tc_kernel<<<(unsigned)((n_rows + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        (uint8_t *)stack_tc, n_rows, frames, (int)(head % frames), (uint32_t)(frames_k1(frames) / 8) * CHUNK_A, obs, done, done_div);
    return cudaGetLastError() == cudaSuccess ? SS_OK : SS_ERR_CUDA;
}

extern "C" int ss_obs_stack_push_pool(void *stack_tc, float *stack32, int64_t n_envs, int64_t pool_envs, int frames, int64_t head,
                                      const float *obs, const uint8_t *done, float *rows_out, float *rows_out2, void *stream) {
    if (!stack32 || !obs || !rows_out || n_envs <= 0 || pool_envs < 0 || pool_envs > n_envs || frames < 1 || frames > MAXF || head < 0)
        return SS_ERR_INVALID_ARG;
    if (((uintptr_t)stack_tc | (uintptr_t)stack32 | (uintptr_t)obs | (uintptr_t)rows_out | (uintptr_t)rows_out2) & 15)
        return SS_ERR_INVALID_ARG;
    const int64_t S = n_envs - pool_envs, L = 2 * S + pool_envs, threads = 3 * frames * (L < PUSH_CHUNK ? L : PUSH_CHUNK);
    const dim3 grid((unsigned)((threads + 255) / 256), (unsigned)((L + PUSH_CHUNK - 1) / PUSH_CHUNK));
    obs_stack_push_pool_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((uint8_t *)stack_tc, stack32, L, S, frames, (int)(head % frames),
                                                                       (uint32_t)(frames_k1(frames) / 8) * CHUNK_A, obs, done, rows_out,
                                                                       rows_out2);
    return cudaGetLastError() == cudaSuccess ? SS_OK : SS_ERR_CUDA;
}

extern "C" int64_t ss_actor_frames_tc_workspace_bytes(int64_t n_rows, int64_t noise_group) {
    if (n_rows <= 0) return -1;
    const int64_t group = noise_group > 0 && noise_group < n_rows ? noise_group : n_rows;
    return frame_units(n_rows, group) * (int64_t)H1TILE_BYTES;
}

extern "C" int ss_actor_forward_frames_tc(const float *params, int64_t param_stride, int64_t noise_group, const void *stack_tc,
                                          int frames, int64_t head, float *act_out, int64_t n_rows, void *workspace,
                                          int64_t workspace_bytes, void *stream) {
    if (!params || !stack_tc || !act_out || !workspace || n_rows <= 0 || frames < 1 || frames > MAXF || head < 0 || param_stride < 0)
        return SS_ERR_INVALID_ARG;
    if (param_stride > 0 && (noise_group <= 0 || noise_group % TM != 0)) return SS_ERR_INVALID_ARG;
    if ((((uintptr_t)params | (uintptr_t)stack_tc | (uintptr_t)workspace) & 15) || (param_stride & 3) || ((uintptr_t)act_out & 7))
        return SS_ERR_INVALID_ARG;
    FramesArgs A{params, (const uint8_t *)stack_tc, act_out, (uint8_t *)workspace, n_rows,
                 param_stride > 0 ? noise_group : n_rows, param_stride, head, frames};
    if (A.group > n_rows) A.group = n_rows;
    const int64_t units = frame_units(n_rows, A.group);
    if (workspace_bytes < units * (int64_t)H1TILE_BYTES) return SS_ERR_INVALID_ARG;
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return SS_ERR_CUDA;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return SS_ERR_CUDA;
    const int64_t n_groups = (n_rows + A.group - 1) / A.group;
    int grid = (int)(units < sms ? units : sms);
    if (A.group < n_rows && n_groups <= sms) grid = (int)n_groups;       // one noise group per CTA: weights staged once
    if (cudaFuncSetAttribute(l1::frames_l1_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)l1::SM_TOTAL) != cudaSuccess ||
        cudaFuncSetAttribute(l23::frames_l23_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)l23::SM_TOTAL) != cudaSuccess)
        return SS_ERR_CUDA;
    l1::frames_l1_kernel<<<grid, l1::NTH, l1::SM_TOTAL, (cudaStream_t)stream>>>(A);
    l23::frames_l23_kernel<<<grid, l23::NTH, l23::SM_TOTAL, (cudaStream_t)stream>>>(A);
    return cudaGetLastError() == cudaSuccess ? SS_OK : SS_ERR_CUDA;
}
