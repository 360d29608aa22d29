// ss_frames_grad_tc.cu -- the learner of the frame-stacked networks on the tensor cores (tcgen05.mma, sm_100a):
// TD targets, critic gradient and actor gradient for a first layer of 12 * frames inputs (readme.md:18-20).
//
// ss_mlp_grad_tc.cu keeps every weight-gradient accumulator of the 12-input networks resident in tensor memory.  With
// 20 frames dW1'^T alone is 256 units x 256 columns of fp32, all 512 tensor-memory columns, so layer 1 leaves that
// scheme and every call is a chain of kernels that pass 128-row tiles through global memory (and mostly the L2):
//
//   frames_pack_kernel   dense fp32 rows [n][12 F] -> the fp16 layer-1 operand tiles of ss_obs_stack_push_tc (ring
//                        head = F - 1: columns in frame order) and, for the gradients, bf16 high / low halves of the
//                        same tiles with a constant-one column behind the inputs (db1 falls out of dW1)
//   frames_l1_kernel     (ss_frames_tc.cu) H1 = relu(X . W1' + b1) -> bf16 tiles; both networks' first layers
//   frames_mid_kernel    from H1 tiles: layer 2 (the critic's action and both biases as K columns, like the 12-input
//                        kernel), the output layer and
//                          FWD     q, -dQ/da, y = r + gamma (1 - done) q
//                          CRITIC  inverted dropout on H1 as it is loaded, mse loss, G3, G2, dx2 -> dz1 tiles
//                          ACTOR   tanh, upstream -dQ/da, G3, G2, dx2 -> dz1 tiles
//                        dz1 overwrites the H1 tile it came from: a tile is read and written by one CTA only
//   frames_dw1_kernel    dW1'^T[256 units][K1] += dZ1^T . X_hi + dZ1^T . X_lo over the CTA's tiles: both operands
//                        MN-major from the chunked tiles, the accumulator takes all of tensor memory
//
// The middle and dW1 kernels run on the same grid over the same tiles (CTA b: tiles b, b + grid, ..), so CTA b's
// partial gradient is one slice of n_params + 1 floats written half by each: the slices feed reduce_parts_kernel,
// ss_reduce_adam_tf and ss_peer_reduce_push like every other gradient entry point's.  No atomics: fixed-order sums.
//
// Each kernel keeps one tile in flight and runs its phases one after another.  At 65,536 rows every kernel has three or
// four tiles per SM; the chain is bound by its launches and the weight staging, not by overlap inside a kernel.
#include "ss_tc_common.cuh"

namespace {

using namespace sstc;

constexpr int MAXF = SS_MAX_FRAMES;
constexpr uint32_t H1TILE_BYTES = (H1 / 8) * CHUNK_A;       // 65,536: hidden layer 1 (or dz1) of one tile

__host__ __device__ constexpr int frames_k1(int frames) { return (DS * frames + 2 + 15) / 16 * 16; }
__host__ __device__ constexpr int64_t frames_shift(int frames) { return (int64_t)(frames - 1) * DS * H1; }
int64_t actor_n(int frames) { return (int64_t)DS * frames * H1 + H1 + H1 * H2 + H2 + H2 * DA + DA; }
int64_t critic_n(int frames) { return (int64_t)DS * frames * H1 + H1 + (H1 + DA) * H2 + H2 + H2 + 1; }

// ---------------------------------------------------------------------------------------------
// pack: one thread per (tile, 8-column chunk, row); thread e writes byte 16 e of each image
// ---------------------------------------------------------------------------------------------
__global__ void frames_pack_kernel(const float *x, int64_t n, int frames, int64_t tiles, uint8_t *xf16, uint8_t *xhi,
                                   uint8_t *xlo) {
    const int chunks = frames_k1(frames) / 8, kx = DS * frames;
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= tiles * chunks * TM) return;
    const int r = (int)(e % TM), c = (int)((e / TM) % chunks);
    const int64_t row = (e / TM / chunks) * TM + r;
    float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    float one[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};          // the constant-one columns kx, kx + 1
    if (row < n) {
        const float4 *src = reinterpret_cast<const float4 *>(x + row * kx + c * 8);
        if (c * 8 < kx) { const float4 a = __ldg(src); v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; }
        if (c * 8 + 4 < kx) { const float4 b = __ldg(src + 1); v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w; }
#pragma unroll
        for (int i = 0; i < 8; ++i) one[i] = (c * 8 + i == kx || c * 8 + i == kx + 1) ? 1.f : 0.f;
    }
    float f[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) f[i] = v[i] + one[i];
    reinterpret_cast<uint4 *>(xf16)[e] = make_uint4(pack_f16(f[0], f[1]), pack_f16(f[2], f[3]), pack_f16(f[4], f[5]), pack_f16(f[6], f[7]));
    if (!xhi) return;
    float hi[8], lo[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        hi[i] = bf16_round(v[i]);
        lo[i] = v[i] - hi[i];
        if (c * 8 + i == kx) hi[i] = one[i];                            // one bias column for the gradient: db1
    }
    reinterpret_cast<uint4 *>(xhi)[e] = make_uint4(pack_bf16(hi[0], hi[1]), pack_bf16(hi[2], hi[3]), pack_bf16(hi[4], hi[5]), pack_bf16(hi[6], hi[7]));
    reinterpret_cast<uint4 *>(xlo)[e] = make_uint4(pack_bf16(lo[0], lo[1]), pack_bf16(lo[2], lo[3]), pack_bf16(lo[4], lo[5]), pack_bf16(lo[6], lo[7]));
}

// ---------------------------------------------------------------------------------------------
// the middle: layers 2 and 3 forward (+ backward) from H1 tiles
// ---------------------------------------------------------------------------------------------
namespace mid {

constexpr int MODE_FWD = 0, MODE_CRITIC = 1, MODE_ACTOR = 2;
// eight epilogue warps as in ss_mlp_grad_tc.cu: warps w and w + 4 share lane quadrant w & 3 and split the columns
constexpr int EPI_WARPS = 8, NSLICE = 2, MMA_WARP = EPI_WARPS, NTH = 32 * (EPI_WARPS + 1);

constexpr uint32_t SM_B2 = 0;
constexpr uint32_t SM_X2 = SM_B2 + B2_BYTES;                // [K2/8][128][8]: h1 (after dropout) | tail
constexpr uint32_t SM_DZ2 = SM_X2 + X2_BYTES;               // [16][128][8]
constexpr uint32_t SM_H2 = SM_DZ2 + 16 * CHUNK_A;           // [16][128][8]
constexpr uint32_t SM_DZ3 = SM_H2 + 16 * CHUNK_A;           // [2][128][8]: {d0 hi, d1 hi, d0 lo, d1 lo, 0..}, chunk 1 = 0
constexpr uint32_t SM_W3 = SM_DZ3 + 2 * CHUNK_A;            // [128] float4
constexpr uint32_t SM_B3 = SM_W3 + H2 * 16;
constexpr uint32_t SM_BAR = SM_B3 + 16;
constexpr uint32_t SM_TMEM = SM_BAR + 16;
constexpr uint32_t SM_RED = SM_TMEM + 16;                   // 4 warps x 4 floats
constexpr uint32_t SM_ZP = SM_RED + 64;                     // [NSLICE][128] float4: partial output-layer sums per column slice
constexpr uint32_t SM_TOTAL = SM_ZP + NSLICE * TM * 16;
static_assert(SM_TOTAL <= 227 * 1024, "shared memory budget");

constexpr uint32_t T_W2T = 0;        // dW2'^T  [128 units][272]
constexpr uint32_t T_W3T = 272;      // dW3^T   [128 units][16]
constexpr uint32_t T_WORK = 384;     // z2, dx2 halves  [128 rows][128]

struct MidArgs {
    const float *params;             // the network's flat vector (frames layout)
    uint8_t *h1;                     // [tiles][H1TILE_BYTES]: H1 in; dz1 out (gradient modes)
    const float *act;                // critic: actions [n][2]
    const float *target;             // CRITIC: regression target [n]
    const float *up, *q;             // ACTOR: -dQ/da [n][2], Q [n]
    const uint8_t *keep;             // CRITIC: injected dropout mask [n][256] or NULL (Philox)
    float rate;
    uint64_t seed, counter;
    int64_t n, n_global, row_offset;
    float *work;                     // [gridDim.x][pn + 1] gradient slices
    int64_t pn;
    float *q_out, *up_out, *y_out;   // FWD
    const float *reward;
    const uint8_t *done;
    float gamma;
    int frames;
};

// the keep bits of 8 consecutive hidden-1 units of one row: ss_mlp_grad_tc.cu's keep8, the same Philox draw
__device__ __forceinline__ uint32_t keep8(const MidArgs &A, int64_t grow, int chunk, uint32_t thresh16) {
    const U4 u = draw4(A.seed, kTagDropout, (uint32_t)grow, (uint32_t)chunk | ((uint32_t)(grow >> 32) << 8), A.counter);
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
    uint32_t bits = 0;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        const uint32_t v = (e & 1) ? (w[e >> 1] >> 16) : (w[e >> 1] & 0xFFFFu);
        bits |= (v >= thresh16 ? 1u : 0u) << e;
    }
    return bits;
}

template <class F>
__device__ __forceinline__ void sweep_work(uint32_t taddr, int cs, F &&f) {
    constexpr int kSteps = 8 / NSLICE;
    uint32_t va[16], vb[16];
    tmem_ld16(taddr + cs * 16, va);
#pragma unroll
    for (int k = 0; k < kSteps; k += 2) {
        const int j = cs + k * NSLICE;
        tmem_wait_ld();
        if (k + 1 < kSteps) tmem_ld16(taddr + (j + NSLICE) * 16, vb);
        f(va, j);
        if (k + 1 < kSteps) {
            tmem_wait_ld();
            if (k + 2 < kSteps) tmem_ld16(taddr + (j + 2 * NSLICE) * 16, va);
            f(vb, j + NSLICE);
        }
    }
}

template <int MODE>
__global__ void __launch_bounds__(NTH, 1) frames_mid_kernel(const MidArgs A) {
    constexpr int NET = MODE == MODE_ACTOR ? NET_ACTOR : NET_CRITIC;
    constexpr bool GRAD = MODE != MODE_FWD;
    extern __shared__ __align__(128) uint8_t smem[];
    const uint32_t sbase = smem_u32(smem);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t bar_mma = sbase + SM_BAR, bar_epi = sbase + SM_BAR + 8;
    if (threadIdx.x == 0) {
        mbar_init(bar_mma, 32 * EPI_WARPS);
        mbar_init(bar_epi, 1);
        mbar_fence_init();
    }
    if (warp == MMA_WARP) tmem_alloc(sbase + SM_TMEM, 512);
    for (uint32_t o = threadIdx.x * 16; o < CHUNK_B2; o += NTH * 16)
        *reinterpret_cast<uint4 *>(smem + SM_B2 + (K2 / 8 - 1) * CHUNK_B2 + o) = make_uint4(0, 0, 0, 0);
    for (uint32_t o = threadIdx.x * 16; o < 2 * CHUNK_A; o += NTH * 16) {
        *reinterpret_cast<uint4 *>(smem + SM_DZ3 + o) = make_uint4(0, 0, 0, 0);
        *reinterpret_cast<uint4 *>(smem + SM_X2 + (H1 / 8) * CHUNK_A + o) = make_uint4(0, 0, 0, 0);
    }
    __syncthreads();
    if (warp < 4 && NET == NET_ACTOR)
        *reinterpret_cast<uint4 *>(smem + SM_X2 + (H1 / 8) * CHUNK_A + threadIdx.x * 16) = tail_chunk_actor();
    // the parameters after W1 are laid out as in the 12-input networks: shift the base so the shared offsets apply
    const int64_t shift = frames_shift(A.frames);
    stage_weights<NET, NTH, false, false>(Stager{A.params + shift, nullptr, smem + SM_B2, reinterpret_cast<float4 *>(smem + SM_W3),
                                                 reinterpret_cast<float *>(smem + SM_B3), false, 0.f, 0, 0, 0});
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *reinterpret_cast<const volatile uint32_t *>(smem + SM_TMEM);

    const int64_t tiles = (A.n + TM - 1) / TM;

    if (warp < EPI_WARPS) {
        // ======================= epilogue warps: thread r owns row r of the tile =======================
        const int r = (warp & 3) * 32 + lane;
        const int cs = warp >> 2;
        const uint32_t tl = tmem + ((uint32_t)((warp & 3) * 32) << 16);
        uint8_t *x2row = smem + SM_X2 + r * 16, *dz2row = smem + SM_DZ2 + r * 16, *h2row = smem + SM_H2 + r * 16;
        const float4 *w3x = reinterpret_cast<const float4 *>(smem + SM_W3);      // critic layout
        const float2 *w3a = reinterpret_cast<const float2 *>(smem + SM_W3);      // actor layout: W3[128][2] as stored
        const float *b3 = reinterpret_cast<const float *>(smem + SM_B3);
        const bool dropout = MODE == MODE_CRITIC && A.rate > 0.f;
        const float inv_keep = dropout ? 1.0f / (1.0f - A.rate) : 1.0f;
        const uint32_t thresh16 = (uint32_t)(A.rate * 65536.0f);
        uint32_t ph = 0;
        float stat = 0.f, dsum0 = 0.f, dsum1 = 0.f;
        auto to_mma = [&]() { fence_proxy_async(); tc_fence_before(); mbar_arrive(bar_mma); };
        auto from_mma = [&]() { mbar_wait(bar_epi, ph); ph ^= 1; tc_fence_after(); };

        // back through hidden layer 1, one half: WORK = dx2 -> mask of the (dropped-out) activation -> bf16 -> dz1 tile
        auto back1 = [&](int half, uint8_t *g1row) {
            sweep_work(tl + T_WORK, cs, [&](const uint32_t (&v)[16], int j) {
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    const uint32_t off = (uint32_t)(half * 16 + j * 2 + c) * CHUNK_A;
                    const uint4 x = *reinterpret_cast<const uint4 *>(x2row + off);
                    const uint32_t xw[4] = {x.x, x.y, x.z, x.w};
                    float d[8];
#pragma unroll
                    for (int e = 0; e < 8; ++e) {
                        const float act = (e & 1) ? bf16_hi(xw[e >> 1]) : bf16_lo(xw[e >> 1]);
                        d[e] = act > 0.f ? __uint_as_float(v[c * 8 + e]) * inv_keep : 0.f;
                    }
                    __stcg(reinterpret_cast<uint4 *>(g1row + off),
                           make_uint4(pack_bf16(d[0], d[1]), pack_bf16(d[2], d[3]), pack_bf16(d[4], d[5]), pack_bf16(d[6], d[7])));
                }
            });
        };

        for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
            const int64_t row = tile * TM + r;
            const bool valid = row < A.n;
            uint8_t *g1row = A.h1 + tile * (int64_t)H1TILE_BYTES + r * 16;
            // ---- H1 of this row (this warp's 16 chunks) -> X2, with inverted dropout; critic: action -> tail chunk ----
#pragma unroll 4
            for (int k = 0; k < 16; ++k) {
                const int c = cs * 16 + k;
                uint4 h = __ldcg(reinterpret_cast<const uint4 *>(g1row + (uint32_t)c * CHUNK_A));
                if (dropout) {
                    uint32_t kb = 0;
                    if (A.keep) {
                        if (valid) {
                            const uint2 m = __ldg(reinterpret_cast<const uint2 *>(A.keep + row * H1 + c * 8));
                            const uint32_t mw[2] = {m.x, m.y};
#pragma unroll
                            for (int e = 0; e < 8; ++e) kb |= (((mw[e >> 2] >> ((e & 3) * 8)) & 0xFFu) ? 1u : 0u) << e;
                        }
                    } else {
                        kb = keep8(A, A.row_offset + row, c, thresh16);
                    }
                    uint32_t hw[4] = {h.x, h.y, h.z, h.w};
#pragma unroll
                    for (int p = 0; p < 4; ++p) {
                        const float lo = (kb >> (2 * p)) & 1u ? bf16_lo(hw[p]) * inv_keep : 0.f;
                        const float hi = (kb >> (2 * p + 1)) & 1u ? bf16_hi(hw[p]) * inv_keep : 0.f;
                        hw[p] = pack_bf16(lo, hi);
                    }
                    h = make_uint4(hw[0], hw[1], hw[2], hw[3]);
                }
                *reinterpret_cast<uint4 *>(x2row + (uint32_t)c * CHUNK_A) = h;
            }
            float2 side = make_float2(0.f, 0.f);          // critic: action; actor: upstream gradient
            float tgt = 0.f;
            if (valid) {
                if (NET == NET_CRITIC) side = __ldg(reinterpret_cast<const float2 *>(A.act) + row);
                else side = __ldg(reinterpret_cast<const float2 *>(A.up) + row);
                if (MODE == MODE_CRITIC) tgt = __ldg(A.target + row);
                if (MODE == MODE_ACTOR) tgt = __ldg(A.q + row);
            }
            if (NET == NET_CRITIC && cs == 0)
                *reinterpret_cast<uint4 *>(x2row + (H1 / 8) * CHUNK_A) = tail_chunk_critic(side.x, side.y);
            to_mma();                                     // -> L2
            from_mma();
            // ---- output layer (fp32) ----
            float z0 = 0.f, z1 = 0.f, z2 = 0.f;          // actor: two outputs; critic: q, dQ/da0, dQ/da1
            sweep_work(tl + T_WORK, cs, [&](const uint32_t (&v)[16], int j) {
#pragma unroll
                for (int c = 0; c < 16; ++c) {
                    const float zz = __uint_as_float(v[c]), h = fmaxf(zz, 0.f);
                    if (NET == NET_ACTOR) {
                        const float2 w = w3a[j * 16 + c];
                        z0 = fmaf(h, w.x, z0);
                        z1 = fmaf(h, w.y, z1);
                    } else {
                        const float4 w = w3x[j * 16 + c];
                        z0 = fmaf(h, w.x, z0);
                        if (MODE == MODE_FWD && zz > 0.f) { z1 += w.y; z2 += w.z; }
                    }
                }
            });
            {
                float4 *zp = reinterpret_cast<float4 *>(smem + SM_ZP);
                zp[cs * TM + r] = make_float4(z0, z1, z2, 0.f);
                asm volatile("bar.sync 1, 256;" ::: "memory");
                const float4 pa = zp[r], pb = zp[TM + r];
                z0 = pa.x + pb.x;
                z1 = pa.y + pb.y;
                z2 = pa.z + pb.z;
            }
            if (MODE == MODE_FWD) {
                if (valid && cs == 0) {
                    const float q = z0 + b3[0];
                    if (A.q_out) A.q_out[row] = q;
                    if (A.up_out) reinterpret_cast<float2 *>(A.up_out)[row] = make_float2(-z1, -z2);
                    if (A.y_out) A.y_out[row] = A.reward[row] + A.gamma * ((A.done && A.done[row]) ? 0.f : 1.f) * q;
                }
                continue;
            }
            float d0 = 0.f, d1 = 0.f;
            if (MODE == MODE_CRITIC) {
                if (valid) {                              // loss "mse": mean over the global batch
                    const float e = (z0 + b3[0]) - tgt;
                    stat += e * e;
                    d0 = 2.0f * e / (float)A.n_global;
                }
            } else if (valid) {                           // through tanh, upstream = -dQ/da
                stat += tgt;
                const float a0 = tanhf(z0 + b3[0]), a1 = tanhf(z1 + b3[1]);
                d0 = side.x * (1.0f - a0 * a0);
                d1 = side.y * (1.0f - a1 * a1);
            }
            if (cs == 0) {
                dsum0 += d0;
                dsum1 += d1;
                const float h0 = bf16_round(d0), h1 = bf16_round(d1);
                *reinterpret_cast<uint4 *>(smem + SM_DZ3 + r * 16) = make_uint4(pack_bf16(h0, h1), pack_bf16(d0 - h0, d1 - h1), 0u, 0u);
            }
            // ---- h2 and dz2 tiles (second sweep over z2) ----
            sweep_work(tl + T_WORK, cs, [&](const uint32_t (&v)[16], int j) {
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    float gz[8];
#pragma unroll
                    for (int e = 0; e < 8; ++e) {
                        float up;
                        if (NET == NET_ACTOR) {
                            const float2 w = w3a[j * 16 + c * 8 + e];
                            up = fmaf(d1, w.y, d0 * w.x);
                        } else {
                            up = d0 * w3x[j * 16 + c * 8 + e].x;
                        }
                        gz[e] = __uint_as_float(v[c * 8 + e]) > 0.f ? up : 0.f;
                    }
                    *reinterpret_cast<uint4 *>(h2row + (uint32_t)(j * 2 + c) * CHUNK_A) = make_uint4(
                        pack_relu_bf16(__uint_as_float(v[c * 8 + 0]), __uint_as_float(v[c * 8 + 1])),
                        pack_relu_bf16(__uint_as_float(v[c * 8 + 2]), __uint_as_float(v[c * 8 + 3])),
                        pack_relu_bf16(__uint_as_float(v[c * 8 + 4]), __uint_as_float(v[c * 8 + 5])),
                        pack_relu_bf16(__uint_as_float(v[c * 8 + 6]), __uint_as_float(v[c * 8 + 7])));
                    *reinterpret_cast<uint4 *>(dz2row + (uint32_t)(j * 2 + c) * CHUNK_A) =
                        make_uint4(pack_bf16(gz[0], gz[1]), pack_bf16(gz[2], gz[3]), pack_bf16(gz[4], gz[5]), pack_bf16(gz[6], gz[7]));
                }
            });
            to_mma();                                     // -> G2 (first half), BXa | G2 (second half), G3
            from_mma();
            back1(0, g1row);
            to_mma();                                     // -> BXb
            from_mma();                                   // ... which also retires G2 / G3
            back1(1, g1row);
        }

        if (GRAD) {
            // ======================= this CTA's partial gradient: layers 2 and 3 of its slice =======================
            float *g = A.work + (int64_t)blockIdx.x * (A.pn + 1) + shift;        // 12-input offsets apply from here
#pragma unroll 1
            for (int j = cs; j < H1 / 16; j += NSLICE) {
                uint32_t v[16];
                tmem_ld16(tl + T_W2T + j * 16, v);
                tmem_wait_ld();
#pragma unroll
                for (int c = 0; c < 16; ++c) __stcg(g + P_W2 + (j * 16 + c) * H2 + r, __uint_as_float(v[c]));
            }
            if (cs == 0) {
                uint32_t t[16];
                tmem_ld16(tl + T_W2T + H1, t);
                tmem_wait_ld();
                if (NET == NET_ACTOR) {
                    __stcg(g + A_B2 + r, __uint_as_float(t[0]));
                } else {
                    __stcg(g + P_W2 + H1 * H2 + r, __uint_as_float(t[0]) + __uint_as_float(t[2]));
                    __stcg(g + P_W2 + (H1 + 1) * H2 + r, __uint_as_float(t[1]) + __uint_as_float(t[3]));
                    __stcg(g + C_B2 + r, __uint_as_float(t[4]));
                }
                tmem_ld16(tl + T_W3T, t);
                tmem_wait_ld();
                if (NET == NET_ACTOR) {
                    __stcg(g + A_W3 + r * DA + 0, __uint_as_float(t[0]) + __uint_as_float(t[2]));
                    __stcg(g + A_W3 + r * DA + 1, __uint_as_float(t[1]) + __uint_as_float(t[3]));
                } else {
                    __stcg(g + C_W3 + r, __uint_as_float(t[0]) + __uint_as_float(t[2]));
                }
                float s0 = dsum0, s1 = dsum1, s2 = stat;
                for (int o = 16; o > 0; o >>= 1) {
                    s0 += __shfl_xor_sync(0xffffffffu, s0, o);
                    s1 += __shfl_xor_sync(0xffffffffu, s1, o);
                    s2 += __shfl_xor_sync(0xffffffffu, s2, o);
                }
                float *red = reinterpret_cast<float *>(smem + SM_RED);
                if (lane == 0) { red[warp * 4 + 0] = s0; red[warp * 4 + 1] = s1; red[warp * 4 + 2] = s2; }
                asm volatile("bar.sync 2, 128;" ::: "memory");
                if (r == 0) {
                    const float t0 = (red[0] + red[4]) + (red[8] + red[12]), t1 = (red[1] + red[5]) + (red[9] + red[13]);
                    const float t2 = (red[2] + red[6]) + (red[10] + red[14]);
                    if (NET == NET_ACTOR) { g[A_B3] = t0; g[A_B3 + 1] = t1; g[A_N] = t2; }
                    else { g[C_B3] = t0; g[C_N] = t2; }
                }
            }
        }
        tc_fence_before();
    } else {
        // ======================= the MMA-issuing warp =======================
        uint32_t ph = 0;
        const uint32_t work = tmem + T_WORK;
        const uint32_t b2 = sbase + SM_B2, x2 = sbase + SM_X2, dz2 = sbase + SM_DZ2, h2 = sbase + SM_H2, dz3 = sbase + SM_DZ3;
        constexpr uint32_t kFwd = umma_idesc(TM, 128);
        constexpr uint32_t kBx = umma_idesc(TM, 128, 0, 1);
        constexpr uint32_t kG128 = umma_idesc(TM, 128, 1, 1), kG16 = umma_idesc(TM, 16, 1, 1);
        auto wait_epi = [&]() { mbar_wait(bar_mma, ph); ph ^= 1; tc_fence_after(); };
        uint32_t acc = 0;
        for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x, acc = 1) {
            wait_epi();                                               // L2
            if (lane == 0) {
                const uint64_t ad = desc_kmajor(x2, CHUNK_A), bd = desc_kmajor(b2, CHUNK_B2);
#pragma unroll
                for (int ks = 0; ks < K2 / 16; ++ks)
                    umma_bf16(work, desc_advance(ad, 2 * CHUNK_A * ks), desc_advance(bd, 2 * CHUNK_B2 * ks), kFwd, ks > 0);
                umma_commit(bar_epi);
            }
            __syncwarp();
            if (!GRAD) continue;
            wait_epi();                                               // G2, BXa, G3
            if (lane == 0) {
                const uint64_t h2t = desc_mnmajor(h2, CHUNK_A), dz3t = desc_mnmajor(dz3, CHUNK_A);
                const uint64_t dz2t = desc_mnmajor(dz2, CHUNK_A), x2t = desc_mnmajor(x2, CHUNK_A);
                const uint64_t x2hi = desc_mnmajor(x2 + 16 * CHUNK_A, CHUNK_A);
                const uint64_t x2tail = desc_mnmajor(x2 + (H1 / 8) * CHUNK_A, CHUNK_A);
#pragma unroll
                for (int ks = 0; ks < TM / 16; ++ks) {
                    const uint32_t off = 2 * CORE * ks;
                    umma_bf16(tmem + T_W2T, desc_advance(dz2t, off), desc_advance(x2t, off), kG128, acc | (ks > 0));
                }
                const uint64_t ad = desc_kmajor(dz2, CHUNK_A), bd = desc_mnmajor(b2, CHUNK_B2);
#pragma unroll
                for (int ks = 0; ks < H2 / 16; ++ks)
                    umma_bf16(work, desc_advance(ad, 2 * CHUNK_A * ks), desc_advance(bd, 2 * CORE * ks), kBx, ks > 0);
                umma_commit(bar_epi);
#pragma unroll
                for (int ks = 0; ks < TM / 16; ++ks) {
                    const uint32_t off = 2 * CORE * ks, a = acc | (ks > 0);
                    umma_bf16(tmem + T_W2T + 128, desc_advance(dz2t, off), desc_advance(x2hi, off), kG128, a);
                    umma_bf16(tmem + T_W2T + H1, desc_advance(dz2t, off), desc_advance(x2tail, off), kG16, a);
                    umma_bf16(tmem + T_W3T, desc_advance(h2t, off), desc_advance(dz3t, off), kG16, a);
                }
            }
            __syncwarp();
            wait_epi();                                               // BXb; its commit also retires the G group above
            if (lane == 0) {
                const uint64_t ad = desc_kmajor(dz2, CHUNK_A), bd = desc_mnmajor(b2 + 16 * CHUNK_B2, CHUNK_B2);
#pragma unroll
                for (int ks = 0; ks < H2 / 16; ++ks)
                    umma_bf16(work, desc_advance(ad, 2 * CHUNK_A * ks), desc_advance(bd, 2 * CORE * ks), kBx, ks > 0);
                umma_commit(bar_epi);
            }
            __syncwarp();
        }
    }

    __syncthreads();
    if (warp == MMA_WARP) {
        tc_fence_after();
        tmem_dealloc(tmem, 512);
    }
}

}  // namespace mid

// ---------------------------------------------------------------------------------------------
// dW1: the layer-1 weight gradient, a reduction over the rows of the CTA's tiles
// ---------------------------------------------------------------------------------------------
namespace dw1 {

constexpr int NTH = 128;                                    // warp w drains tensor-memory lanes 32 w ..
constexpr uint32_t XTILE_MAX = (frames_k1(MAXF) / 8) * CHUNK_A;
constexpr uint32_t SM_DZ = 0;                               // [32][128][8] bf16: dz1
constexpr uint32_t SM_XH = SM_DZ + H1TILE_BYTES;            // [K1/8][128][8] bf16: X high half (+ the one column)
constexpr uint32_t SM_XL = SM_XH + XTILE_MAX;               // X low half
constexpr uint32_t SM_BAR = SM_XL + XTILE_MAX;
constexpr uint32_t SM_TMEM = SM_BAR + 8;
constexpr uint32_t SM_TOTAL = SM_TMEM + 8;
static_assert(SM_TOTAL <= 227 * 1024, "shared memory budget");

struct Dw1Args {
    const uint8_t *dz1, *xhi, *xlo;  // tiles
    int64_t n;
    float *work;                     // [gridDim.x][pn + 1]
    int64_t pn;
    int frames;
};

__device__ __forceinline__ void copy_tile(uint8_t *dst, const uint8_t *src, uint32_t bytes) {
    for (uint32_t o = threadIdx.x * 16; o < bytes; o += NTH * 16)
        *reinterpret_cast<uint4 *>(dst + o) = __ldcg(reinterpret_cast<const uint4 *>(src + o));
}

__global__ void __launch_bounds__(NTH, 1) frames_dw1_kernel(const Dw1Args A) {
    extern __shared__ __align__(128) uint8_t smem[];
    const uint32_t sbase = smem_u32(smem);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t bar = sbase + SM_BAR;
    const int k1 = frames_k1(A.frames), kx = DS * A.frames;
    const uint32_t xbytes = (uint32_t)(k1 / 8) * CHUNK_A;
    if (threadIdx.x == 0) {
        mbar_init(bar, 1);
        mbar_fence_init();
    }
    if (warp == 0) tmem_alloc(sbase + SM_TMEM, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *reinterpret_cast<const volatile uint32_t *>(smem + SM_TMEM);
    // M = 128 units of one half, N = the K1 input columns, K = 16 rows per step; both operands MN-major
    const uint32_t kG = umma_idesc(TM, k1, 1, 1);

    const int64_t tiles = (A.n + TM - 1) / TM;
    uint32_t ph = 0, acc = 0;
    for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x, acc = 1) {
        copy_tile(smem + SM_DZ, A.dz1 + tile * (int64_t)H1TILE_BYTES, H1TILE_BYTES);
        copy_tile(smem + SM_XH, A.xhi + tile * (int64_t)xbytes, xbytes);
        copy_tile(smem + SM_XL, A.xlo + tile * (int64_t)xbytes, xbytes);
        fence_proxy_async();
        __syncthreads();
        if (threadIdx.x == 0) {
            tc_fence_after();
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const uint64_t dzt = desc_mnmajor(sbase + SM_DZ + half * 16 * CHUNK_A, CHUNK_A);
#pragma unroll
                for (int part = 0; part < 2; ++part) {
                    const uint64_t xt = desc_mnmajor(sbase + (part ? SM_XL : SM_XH), CHUNK_A);
#pragma unroll
                    for (int ks = 0; ks < TM / 16; ++ks)
                        umma_bf16(tmem + half * 256, desc_advance(dzt, 2 * CORE * ks), desc_advance(xt, 2 * CORE * ks), kG,
                                  acc | (uint32_t)(part | ks));
                }
            }
            umma_commit(bar);
        }
        mbar_wait(bar, ph);                                   // the MMAs have read the tiles: they may be replaced
        ph ^= 1;
        tc_fence_after();
    }

    // thread r = hidden-1 unit 128 half + r; column c < 12 F: W1 row c, column 12 F: b1
    float *g = A.work + (int64_t)blockIdx.x * (A.pn + 1);
    const int r = warp * 32 + lane;
    const uint32_t tl = tmem + ((uint32_t)(warp * 32) << 16);
#pragma unroll 1
    for (int half = 0; half < 2; ++half) {
        const int unit = half * 128 + r;
#pragma unroll 1
        for (int j = 0; j * 16 <= kx; ++j) {
            uint32_t v[16];
            tmem_ld16(tl + half * 256 + j * 16, v);
            tmem_wait_ld();
#pragma unroll
            for (int c = 0; c < 16; ++c) {
                const int col = j * 16 + c;
                if (col <= kx) __stcg(g + (int64_t)col * H1 + unit, __uint_as_float(v[c]));     // row kx of W1' = b1
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        tmem_dealloc(tmem, 512);
    }
}

}  // namespace dw1

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
int64_t align16(int64_t b) { return (b + 15) / 16 * 16; }

// workspace: [slices][X fp16][X hi][X lo][H1 a][H1 b][act][up][q]
struct Lay {
    int64_t tiles, parts, pn, slices, xf, xhi, xlo, h1a, h1b, act, up, q, total;
};
Lay lay_of(int frames, int64_t n) {
    Lay L{};
    L.tiles = (n + TM - 1) / TM;
    L.parts = L.tiles < SS_LEARNER_MAX_PARTS ? L.tiles : SS_LEARNER_MAX_PARTS;
    const int64_t an = actor_n(frames), cn = critic_n(frames);
    L.pn = an > cn ? an : cn;
    const int64_t xb = L.tiles * (frames_k1(frames) / 8) * (int64_t)CHUNK_A, hb = L.tiles * (int64_t)H1TILE_BYTES;
    L.slices = 0;
    L.xf = align16(L.parts * (L.pn + 1) * 4);
    L.xhi = L.xf + xb;
    L.xlo = L.xhi + xb;
    L.h1a = L.xlo + xb;
    L.h1b = L.h1a + hb;
    L.act = L.h1b + hb;
    L.up = L.act + align16(n * 8);
    L.q = L.up + align16(n * 8);
    L.total = L.q + align16(n * 4);
    return L;
}

struct Ctx {
    Lay L;
    uint8_t *ws;
    cudaStream_t st;
    int sms;
    template <class T = uint8_t>
    T *at(int64_t off) const { return reinterpret_cast<T *>(ws + off); }
};

// the checks every entry point shares; SS_OK and a filled context, or SS_ERR_INVALID_ARG before any device call
int prepare(int frames, int64_t n, void *workspace, int64_t workspace_bytes, void *stream, Ctx &C) {
    if (frames < 1 || frames > MAXF || n <= 0 || !workspace || ((uintptr_t)workspace & 15)) return SS_ERR_INVALID_ARG;
    C.L = lay_of(frames, n);
    if (workspace_bytes < C.L.total) return SS_ERR_INVALID_ARG;
    C.ws = (uint8_t *)workspace;
    C.st = (cudaStream_t)stream;
    return SS_OK;
}

int device_sms(int &sms) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return SS_ERR_CUDA;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return SS_ERR_CUDA;
    return SS_OK;
}

int pack(const Ctx &C, const float *x, int frames, int64_t n, bool with_grad_images) {
    const int64_t threads = C.L.tiles * (frames_k1(frames) / 8) * TM;
    frames_pack_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, C.st>>>(x, n, frames, C.L.tiles, C.at(C.L.xf),
                                                                          with_grad_images ? C.at(C.L.xhi) : nullptr,
                                                                          with_grad_images ? C.at(C.L.xlo) : nullptr);
    return cudaGetLastError() == cudaSuccess ? SS_OK : SS_ERR_CUDA;
}

template <int MODE>
int launch_mid(const mid::MidArgs &A, int grid, cudaStream_t st) {
    if (cudaFuncSetAttribute(mid::frames_mid_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)mid::SM_TOTAL) !=
        cudaSuccess)
        return SS_ERR_CUDA;
    mid::frames_mid_kernel<MODE><<<grid, mid::NTH, mid::SM_TOTAL, st>>>(A);
    return cudaGetLastError() == cudaSuccess ? SS_OK : SS_ERR_CUDA;
}

int grid_of(const Ctx &C, int sms) {
    const int64_t g = C.L.parts < sms ? C.L.parts : sms;
    return (int)g;
}

// q / -dQ/da / y of `critic_params` at (packed X, act): critic layer 1 into H1 region b, then the middle in FWD mode
int critic_forward(const Ctx &C, const float *critic_params, int frames, int64_t n, const float *act, float *q_out, float *up_out,
                   const float *reward, const uint8_t *done, float gamma, float *y_out, int sms) {
    int rc = frames_layer1_tc(critic_params, C.at(C.L.xf), frames, n, C.at(C.L.h1b), C.st);
    if (rc != SS_OK) return rc;
    mid::MidArgs A{};
    A.params = critic_params; A.h1 = C.at(C.L.h1b); A.act = act; A.n = n; A.n_global = n; A.frames = frames;
    A.q_out = q_out; A.up_out = up_out; A.y_out = y_out; A.reward = reward; A.done = done; A.gamma = gamma;
    return launch_mid<mid::MODE_FWD>(A, grid_of(C, sms), C.st);
}

// the middle in a gradient mode (its dz1 overwrites the H1 tiles at h1), dW1, then the reduction unless slices only
template <int MODE>
int gradient(const Ctx &C, mid::MidArgs A, int frames, int64_t n, int64_t pn, float *grad_out, float *aux_out, int sms) {
    const int grid = grid_of(C, sms);
    A.work = C.at<float>(C.L.slices); A.pn = pn; A.n = n; A.frames = frames;
    int rc = launch_mid<MODE>(A, grid, C.st);
    if (rc != SS_OK) return rc;
    if (cudaFuncSetAttribute(dw1::frames_dw1_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dw1::SM_TOTAL) != cudaSuccess)
        return SS_ERR_CUDA;
    dw1::frames_dw1_kernel<<<grid, dw1::NTH, dw1::SM_TOTAL, C.st>>>(
        dw1::Dw1Args{A.h1, C.at(C.L.xhi), C.at(C.L.xlo), n, C.at<float>(C.L.slices), pn, frames});
    if (cudaGetLastError() != cudaSuccess) return SS_ERR_CUDA;
    if (!grad_out) return grid;                               // slices only (ss_reduce_adam_tf / ss_peer_reduce_push follow)
    return reduce_slices(C.at<float>(C.L.slices), grid, (int)pn, grad_out, aux_out, C.st);
}

}  // namespace

extern "C" {

int64_t ss_learner_frames_tc_workspace_bytes(int frames, int64_t n) {
    if (frames < 1 || frames > MAXF || n <= 0) return -1;
    return lay_of(frames, n).total;
}

int ss_critic_forward_frames_tc(const float *critic_params, int frames, const float *obs, const float *act, float *q_out,
                                float *neg_dq_da_out, int64_t n, void *workspace, int64_t workspace_bytes, void *stream) {
    Ctx C{};
    if (!critic_params || !obs || !act || (!q_out && !neg_dq_da_out)) return SS_ERR_INVALID_ARG;
    if (((uintptr_t)critic_params | (uintptr_t)obs) & 15 || (((uintptr_t)act | (uintptr_t)neg_dq_da_out) & 7)) return SS_ERR_INVALID_ARG;
    if (prepare(frames, n, workspace, workspace_bytes, stream, C) != SS_OK) return SS_ERR_INVALID_ARG;
    int sms = 0, rc = device_sms(sms);
    if (rc == SS_OK) rc = pack(C, obs, frames, n, false);
    if (rc == SS_OK) rc = critic_forward(C, critic_params, frames, n, act, q_out, neg_dq_da_out, nullptr, nullptr, 0.f, nullptr, sms);
    return rc;
}

int ss_ddpg_targets_frames_tc(const float *target_actor_params, const float *target_critic_params, int frames,
                              const float *reward, const float *next_obs, const uint8_t *done, float gamma, float *y_out,
                              int64_t n, void *workspace, int64_t workspace_bytes, void *stream) {
    Ctx C{};
    if (!target_actor_params || !target_critic_params || !reward || !next_obs || !y_out) return SS_ERR_INVALID_ARG;
    if (((uintptr_t)target_actor_params | (uintptr_t)target_critic_params | (uintptr_t)next_obs) & 15) return SS_ERR_INVALID_ARG;
    if (prepare(frames, n, workspace, workspace_bytes, stream, C) != SS_OK) return SS_ERR_INVALID_ARG;
    int sms = 0, rc = device_sms(sms);
    if (rc == SS_OK) rc = pack(C, next_obs, frames, n, false);
    // a' = actor'(s'): layers 1 and 2/3 of the frame-stacked actor, its hidden layer in region b
    if (rc == SS_OK)
        rc = ss_actor_forward_frames_tc(target_actor_params, 0, 0, C.at(C.L.xf), frames, frames - 1, C.at<float>(C.L.act), n,
                                        C.at(C.L.h1b), C.L.act - C.L.h1b, stream);
    if (rc == SS_OK)
        rc = critic_forward(C, target_critic_params, frames, n, C.at<float>(C.L.act), nullptr, nullptr, reward, done, gamma, y_out, sms);
    return rc;
}

// ss_ddpg_targets_frames_tc with the smoothing on a' and, with a second critic, both critics' q (in the q and -dQ/da
// regions of the workspace) -> td3_min_target
int ss_td3_targets_frames_tc(const float *target_actor_params, const float *target_critic_params, const float *target_critic2_params,
                             int frames, const float *reward, const float *next_obs, const uint8_t *done, float gamma, float noise_sd,
                             float noise_clip, uint64_t seed, uint64_t counter, int64_t row_offset, float *y_out, int64_t n,
                             void *workspace, int64_t workspace_bytes, void *stream) {
    Ctx C{};
    if (!target_actor_params || !target_critic_params || !reward || !next_obs || !y_out) return SS_ERR_INVALID_ARG;
    if (frames < 2 || !(noise_sd >= 0.f) || !(noise_clip >= 0.f) || row_offset < 0) return SS_ERR_INVALID_ARG;
    if (((uintptr_t)target_actor_params | (uintptr_t)target_critic_params | (uintptr_t)target_critic2_params | (uintptr_t)next_obs) & 15)
        return SS_ERR_INVALID_ARG;
    if (prepare(frames, n, workspace, workspace_bytes, stream, C) != SS_OK) return SS_ERR_INVALID_ARG;
    int sms = 0, rc = device_sms(sms);
    if (rc == SS_OK) rc = pack(C, next_obs, frames, n, false);
    if (rc == SS_OK)
        rc = ss_actor_forward_frames_tc(target_actor_params, 0, 0, C.at(C.L.xf), frames, frames - 1, C.at<float>(C.L.act), n,
                                        C.at(C.L.h1b), C.L.act - C.L.h1b, stream);
    if (rc == SS_OK && noise_sd > 0.f)
        rc = td3_smooth_actions(C.at<float>(C.L.act), n, noise_sd, noise_clip, seed, counter, row_offset, C.st);
    if (rc != SS_OK) return rc;
    if (!target_critic2_params)
        return critic_forward(C, target_critic_params, frames, n, C.at<float>(C.L.act), nullptr, nullptr, reward, done, gamma, y_out, sms);
    float *q1 = C.at<float>(C.L.q), *q2 = C.at<float>(C.L.up);
    rc = critic_forward(C, target_critic_params, frames, n, C.at<float>(C.L.act), q1, nullptr, nullptr, nullptr, 0.f, nullptr, sms);
    if (rc == SS_OK)
        rc = critic_forward(C, target_critic2_params, frames, n, C.at<float>(C.L.act), q2, nullptr, nullptr, nullptr, 0.f, nullptr, sms);
    if (rc != SS_OK) return rc;
    return td3_min_target(q1, q2, reward, done, gamma, y_out, n, C.st);
}

int ss_critic_grad_frames_tc(const float *critic_params, int frames, const float *obs, const float *act, const float *target,
                             const uint8_t *dropout_keep, float dropout_rate, uint64_t seed, uint64_t counter,
                             int64_t n, int64_t n_global, int64_t row_offset, float *grad_out, float *sse_out,
                             void *workspace, int64_t workspace_bytes, void *stream) {
    Ctx C{};
    if (!critic_params || !obs || !act || !target) return SS_ERR_INVALID_ARG;
    if (dropout_rate < 0.f || dropout_rate >= 1.f) return SS_ERR_INVALID_ARG;
    if (((uintptr_t)critic_params | (uintptr_t)obs) & 15 || ((uintptr_t)act & 7) || ((uintptr_t)dropout_keep & 7))
        return SS_ERR_INVALID_ARG;
    if (prepare(frames, n, workspace, workspace_bytes, stream, C) != SS_OK) return SS_ERR_INVALID_ARG;
    int sms = 0, rc = device_sms(sms);
    if (rc == SS_OK) rc = pack(C, obs, frames, n, true);
    if (rc == SS_OK) rc = frames_layer1_tc(critic_params, C.at(C.L.xf), frames, n, C.at(C.L.h1a), C.st);
    if (rc != SS_OK) return rc;
    mid::MidArgs A{};
    A.params = critic_params; A.h1 = C.at(C.L.h1a); A.act = act; A.target = target; A.keep = dropout_keep; A.rate = dropout_rate;
    A.seed = seed; A.counter = counter; A.n_global = n_global > 0 ? n_global : n; A.row_offset = row_offset;
    return gradient<mid::MODE_CRITIC>(C, A, frames, n, critic_n(frames), grad_out, sse_out, sms);
}

int ss_actor_grad_frames_tc(const float *actor_params, const float *critic_params, int frames, const float *obs, int64_t n,
                            float *grad_out, float *q_sum_out, void *workspace, int64_t workspace_bytes, void *stream) {
    Ctx C{};
    if (!actor_params || !critic_params || !obs) return SS_ERR_INVALID_ARG;
    if (((uintptr_t)actor_params | (uintptr_t)critic_params | (uintptr_t)obs) & 15) return SS_ERR_INVALID_ARG;
    if (prepare(frames, n, workspace, workspace_bytes, stream, C) != SS_OK) return SS_ERR_INVALID_ARG;
    int sms = 0, rc = device_sms(sms);
    if (rc == SS_OK) rc = pack(C, obs, frames, n, true);
    // a = actor(s), its hidden layer kept in region a; q, -dQ/da = critic(s, a) with dropout off (region b)
    if (rc == SS_OK)
        rc = ss_actor_forward_frames_tc(actor_params, 0, 0, C.at(C.L.xf), frames, frames - 1, C.at<float>(C.L.act), n, C.at(C.L.h1a),
                                        C.L.h1b - C.L.h1a, stream);
    if (rc == SS_OK)
        rc = critic_forward(C, critic_params, frames, n, C.at<float>(C.L.act), C.at<float>(C.L.q), C.at<float>(C.L.up), nullptr, nullptr,
                            0.f, nullptr, sms);
    if (rc != SS_OK) return rc;
    mid::MidArgs A{};
    A.params = actor_params; A.h1 = C.at(C.L.h1a); A.up = C.at<float>(C.L.up); A.q = C.at<float>(C.L.q); A.n_global = n;
    return gradient<mid::MODE_ACTOR>(C, A, frames, n, actor_n(frames), grad_out, q_sum_out, sms);
}

}  // extern "C"
