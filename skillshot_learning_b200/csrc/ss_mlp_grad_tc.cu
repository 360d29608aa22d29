// ss_mlp_grad_tc.cu -- forward + backward pass of the actor / critic MLP on the tensor cores
// (tcgen05.mma, sm_100a): the gradient half of model_critic.fit (SkillshotLearner.py:434) and of
// model_actor_fit_step (SkillshotLearner.py:386-417) for large batches.
//
// Per 128-row tile the dense work is seven GEMM groups, all bf16 x bf16 -> fp32 in tensor memory:
//
//   L1a/L1b  z1[:, half]   = X0 . W1'                 128 x 128 x 32     (bias row included)
//   L2       z2            = X2 . W2'                 128 x 128 x 272    (bias / action rows included)
//   G3       dW3^T        += H2^T . DZ3               128 x 16  x 128 rows
//   G2       dW2'^T       += DZ2^T . X2               128 x 272 x 128 rows
//   BXa/BXb  dx2[:, half]  = DZ2 . W2^T               128 x 128 x 128
//   G1       dW1'^T[half] += DZ1[:, half]^T . X0      128 x 32  x 128 rows
//
// The weight-gradient GEMMs reduce over the ROWS of the tile.  Their operands are the very
// activation tiles the forward pass wrote, read MN-major instead of K-major (ss_tc_common.cuh),
// and their accumulators (272 + 64 + 16 tensor-memory columns) stay resident for every tile the
// CTA processes: nothing but the final sums ever leaves the SM.  Because the bias rows are part of
// W1' / W2' (constant-one columns in X0 / X2), db1 and db2 fall out of G1 / G2 for free, as do the
// gradients of the critic's two action rows.  The element-wise steps between the GEMMs (ReLU,
// inverted dropout, the 128 -> 1|2 output layer, loss / upstream gradient, ReLU masks) run on eight
// epilogue warps (two per tensor-memory lane quadrant, splitting the columns of every sweep), one
// thread per row and column slice, between tcgen05.ld and the shared-memory tile stores.
// One tile is in flight per CTA (its activations take 136 KB of shared memory beside 86 KB of
// weight images; the accumulators take 352 of the 512 tensor-memory columns).
//
// Order of issue within a tile (round 2): L1a, L1b, L2 one by one (each output is consumed before
// the next can overwrite the work columns); then G2's first half and BXa behind ONE commit -- the
// epilogue warps wait for dx2 only, and its first half may overwrite h1[:, :128] as soon as G2 has
// consumed it -- with the rest of G2, its bias / action columns and G3 running beside back1(0) and
// retiring with BXb's commit; G1 has no commit of its own and retires with the next tile's L1a
// (X0 of the next tile is staged into the head of the H2 buffer meanwhile).
//
// Gradients are therefore computed from bf16 operands (products exact, fp32 accumulation):
// relative error ~1e-3 against the float32 path of ss_learner.cu, which remains the exact one.
// Per-CTA partial gradients go to the same workspace layout and fixed-order reduction as there.
#include "ss_tc_common.cuh"

namespace {

using namespace sstc;

// eight epilogue warps: warps w and w + 4 share tensor-memory lane quadrant w & 3 (rows 32 (w & 3) ..) and split the
// columns of every element-wise sweep between them; MMAs and sweeps alternate in this kernel, so the extra tcgen05.ld
// traffic does not compete with the tensor pipe (unlike in the forward kernel)
constexpr int EPI_WARPS = 8, NSLICE = EPI_WARPS / 4, MMA_WARP = EPI_WARPS, NTHREADS = 32 * (EPI_WARPS + 1);

// shared-memory map (bytes)
constexpr uint32_t SM_B1 = 0;
constexpr uint32_t SM_B2 = SM_B1 + B1_BYTES;
constexpr uint32_t SM_X2 = SM_B2 + B2_BYTES;                // [K2/8][128][8]: h1 | tail, later dz1
constexpr uint32_t SM_DZ2 = SM_X2 + X2_BYTES;               // [16][128][8]: dz2; its head holds X0 (4 chunks) before / after
constexpr uint32_t SM_H2 = SM_DZ2 + 16 * CHUNK_A;           // [16][128][8]: h2
constexpr uint32_t SM_DZ3 = SM_H2 + 16 * CHUNK_A;           // [2][128][8]: {d0 hi, d1 hi, d0 lo, d1 lo, 0..}, chunk 1 = 0
constexpr uint32_t SM_W3 = SM_DZ3 + 2 * CHUNK_A;            // [128] float4
constexpr uint32_t SM_B3 = SM_W3 + H2 * 16;
constexpr uint32_t SM_BAR = SM_B3 + 16;                     // {epilogue -> MMA (128 arrivals), MMA -> epilogue (commit)}
constexpr uint32_t SM_TMEM = SM_BAR + 16;
constexpr uint32_t SM_RED = SM_TMEM + 16;                   // 4 warps x 4 floats
constexpr uint32_t SM_ZP = SM_RED + 64;                     // [NSLICE][128] float2: partial output-layer sums per column slice
constexpr uint32_t SM_TOTAL = SM_ZP + NSLICE * TM * 8;
static_assert(SM_TOTAL <= 227 * 1024, "shared memory budget");

// tensor-memory columns
constexpr uint32_t T_W2T = 0;        // dW2'^T  [128 units][272]
constexpr uint32_t T_W1T = 272;      // dW1'^T  2 x [128 units][32]
constexpr uint32_t T_W3T = 336;      // dW3^T   [128 units][16]
constexpr uint32_t T_WORK = 384;     // z1 halves, z2, dx2 halves  [128 rows][128]

struct GradArgs {
    const float *params, *obs;
    const float *act, *target;       // critic: actions [n][2], regression target [n]
    const float *up;                 // actor: upstream gradient on the action [n][2] (= -dQ/da)
    const float *q;                  // actor: Q(s, actor(s)) per row [n] or NULL; its sum goes out through the slices' extra slot
    const uint8_t *keep;             // critic: injected dropout mask [n][256] or NULL (Philox)
    float rate;
    uint64_t seed, counter;
    int64_t n, n_global, row_offset;
    float *work;                     // [gridDim.x][params + 1]
    int early_weights;               // ss_launch.cuh: the parameters may be staged ahead of griddepcontrol.wait (set by launch_grad)
};

// inverted-dropout keep bits of 8 consecutive hidden-1 units of one row: one Philox draw, 16 bits per unit
__device__ __forceinline__ uint32_t keep8(const GradArgs &A, int64_t grow, int chunk, uint32_t thresh16) {
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

// The 128 work columns in steps of 16, this warp's steps only (j = cs, cs + NSLICE, ..), tensor-memory loads
// double-buffered: f(v, j) gets columns 16 j .. 16 j + 15 of this thread's lane while the next step's load is in flight.
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

template <int NET>
__global__ void __launch_bounds__(NTHREADS, 1) mlp_grad_tc_kernel(const GradArgs A) {
    constexpr int PN = NET == NET_ACTOR ? A_N : C_N;
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
    // zero what is only partly rewritten: the padding chunk of the layer-2 weight image (stage_weights writes every other
    // byte of both images), DZ3 (chunk 1), X2 tail chunks
    for (uint32_t o = threadIdx.x * 16; o < CHUNK_B2; o += NTHREADS * 16)
        *reinterpret_cast<uint4 *>(smem + SM_B2 + (K2 / 8 - 1) * CHUNK_B2 + o) = make_uint4(0, 0, 0, 0);
    for (uint32_t o = threadIdx.x * 16; o < 2 * CHUNK_A; o += NTHREADS * 16) {
        *reinterpret_cast<uint4 *>(smem + SM_DZ3 + o) = make_uint4(0, 0, 0, 0);
        *reinterpret_cast<uint4 *>(smem + SM_X2 + (H1 / 8) * CHUNK_A + o) = make_uint4(0, 0, 0, 0);
    }
    __syncthreads();
    if (warp < 4 && NET == NET_ACTOR)
        *reinterpret_cast<uint4 *>(smem + SM_X2 + (H1 / 8) * CHUNK_A + threadIdx.x * 16) = tail_chunk_actor();
    // dependent launch (ss_launch.cuh): the set-up above ran beside the previous grid's tail; the weights are staged ahead of
    // the wait too when the caller knows that grid does not write them
    if (!A.early_weights) { sslaunch::griddep_wait(); sslaunch::griddep_launch(); }
    stage_weights<NET, NTHREADS>(Stager{A.params, smem + SM_B1, smem + SM_B2, reinterpret_cast<float4 *>(smem + SM_W3),
                                        reinterpret_cast<float *>(smem + SM_B3), false, 0.f, 0, 0, 0});
    if (A.early_weights) { sslaunch::griddep_wait(); sslaunch::griddep_launch(); }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *reinterpret_cast<const volatile uint32_t *>(smem + SM_TMEM);

    const int64_t tiles = (A.n + TM - 1) / TM;
    float *g = A.work + (int64_t)blockIdx.x * (PN + 1);

    if (warp < EPI_WARPS) {
        // ======================= epilogue warps: thread r owns row r of the tile =======================
        const int r = (warp & 3) * 32 + lane;           // row of the tile = tensor-memory lane
        const int cs = warp >> 2;                       // column slice of this warp
        const uint32_t tl = tmem + ((uint32_t)((warp & 3) * 32) << 16);
        uint8_t *x2row = smem + SM_X2 + r * 16, *dz2row = smem + SM_DZ2 + r * 16, *h2row = smem + SM_H2 + r * 16;
        const float4 *w3x = reinterpret_cast<const float4 *>(smem + SM_W3);      // critic layout
        const float2 *w3a = reinterpret_cast<const float2 *>(smem + SM_W3);      // actor layout: W3[128][2] as stored
        const float *b3 = reinterpret_cast<const float *>(smem + SM_B3);
        const float inv_keep = (NET == NET_CRITIC && A.rate > 0.f) ? 1.0f / (1.0f - A.rate) : 1.0f;
        const uint32_t thresh16 = (uint32_t)(A.rate * 65536.0f);
        uint32_t ph = 0;
        float stat = 0.f, dsum0 = 0.f, dsum1 = 0.f;      // sum of squared errors; db3 partials
        int tl_i = 0;                                   // tiles done by this CTA
        auto to_mma = [&]() { fence_proxy_async(); tc_fence_before(); mbar_arrive(bar_mma); };
        auto from_mma = [&]() { mbar_wait(bar_epi, ph); ph ^= 1; tc_fence_after(); };

        // hidden layer 1, one 128-unit half: WORK -> ReLU (+ dropout) -> bf16 -> X2 chunks 16 * half ..
        // Inverted-dropout keep bits of this thread's row for the columns its warp handles: 2 halves x 4 steps x 16
        // units = 128 bits.  They are generated one tile AHEAD, in four parts, while the warp would otherwise idle in the waits
        // for the three long MMA phases (32 Philox draws per row and tile cost ~5 k cycles when computed inside hidden1).
        uint32_t kb_cur[4] = {~0u, ~0u, ~0u, ~0u}, kb_next[4] = {~0u, ~0u, ~0u, ~0u};
        // part = 0, 1: the first / second pair of this warp's four 16-unit steps of the half (4 of the row's 16 draws)
        auto make_keep = [&](int64_t tile, int half, int part) {
            if (!(NET == NET_CRITIC && A.rate > 0.f) || tile >= tiles) return;
            const int64_t row = tile * TM + r;
            kb_next[half * 2 + part] = 0u;
            {
#pragma unroll
                for (int k = 2 * part; k < 2 * part + 2; ++k) {
                    const int c0 = half * 16 + (cs + k * NSLICE) * 2;          // first of the step's two 8-unit chunks
                    uint32_t kb = 0;
                    if (A.keep) {
                        if (row < A.n) {
                            const uint4 m = __ldg(reinterpret_cast<const uint4 *>(A.keep + row * H1 + c0 * 8));
                            const uint32_t mw[4] = {m.x, m.y, m.z, m.w};
#pragma unroll
                            for (int e = 0; e < 16; ++e) kb |= (((mw[e >> 2] >> ((e & 3) * 8)) & 0xFFu) ? 1u : 0u) << e;
                        }
                    } else {
                        kb = keep8(A, A.row_offset + row, c0, thresh16) | (keep8(A, A.row_offset + row, c0 + 1, thresh16) << 8);
                    }
                    kb_next[half * 2 + (k >> 1)] |= kb << ((k & 1) * 16);
                }
            }
        };
        // hidden layer 1, one 128-unit half: WORK -> ReLU (+ dropout) -> bf16 -> X2 chunks 16 * half ..
        auto hidden1 = [&](int half) {
            sweep_work(tl + T_WORK, cs, [&](const uint32_t (&v)[16], int j) {      // 16 columns = 2 chunks per step
                const int k = (j - cs) / NSLICE;
                const uint32_t kb = (kb_cur[half * 2 + (k >> 1)] >> ((k & 1) * 16)) & 0xFFFFu;
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    float h[8];
#pragma unroll
                    for (int e = 0; e < 8; ++e)
                        h[e] = ((kb >> (c * 8 + e)) & 1u) ? __uint_as_float(v[c * 8 + e]) * inv_keep : 0.f;
                    *reinterpret_cast<uint4 *>(x2row + (uint32_t)(half * 16 + j * 2 + c) * CHUNK_A) = make_uint4(
                        pack_relu_bf16(h[0], h[1]), pack_relu_bf16(h[2], h[3]), pack_relu_bf16(h[4], h[5]), pack_relu_bf16(h[6], h[7]));
                }
            });
        };
        // back through hidden layer 1, one half: WORK = dx2 -> mask of the stored activation -> bf16 -> same chunks
        auto back1 = [&](int half) {
            sweep_work(tl + T_WORK, cs, [&](const uint32_t (&v)[16], int j) {
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    uint4 *p = reinterpret_cast<uint4 *>(x2row + (uint32_t)(half * 16 + j * 2 + c) * CHUNK_A);
                    const uint4 x = *p;
                    const uint32_t xw[4] = {x.x, x.y, x.z, x.w};
                    float d[8];
#pragma unroll
                    for (int e = 0; e < 8; ++e) {
                        const float act = (e & 1) ? bf16_hi(xw[e >> 1]) : bf16_lo(xw[e >> 1]);
                        d[e] = act > 0.f ? __uint_as_float(v[c * 8 + e]) * inv_keep : 0.f;
                    }
                    *p = make_uint4(pack_bf16(d[0], d[1]), pack_bf16(d[2], d[3]), pack_bf16(d[4], d[5]), pack_bf16(d[6], d[7]));
                }
            });
        };

        // this row's inputs of the NEXT tile are fetched while the current tile is processed
        float4 xnext[3];
        float2 side_next = make_float2(0.f, 0.f);        // critic: action; actor: upstream gradient
        float tgt_next = 0.f;
        auto fetch = [&](int64_t tile) {
            const int64_t row = tile * TM + r;
            load_obs(A.obs, row, tile < tiles ? A.n : 0, xnext);
            side_next = make_float2(0.f, 0.f);
            tgt_next = 0.f;
            if (tile < tiles && row < A.n) {
                side_next = __ldg(reinterpret_cast<const float2 *>(NET == NET_CRITIC ? A.act : A.up) + row);
                if (NET == NET_CRITIC) tgt_next = __ldg(A.target + row);
                else if (A.q) tgt_next = __ldg(A.q + row);
            }
        };
        fetch(blockIdx.x);
        for (int q = 0; q < 4; ++q) make_keep(blockIdx.x, q >> 1, q & 1);
        for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
            const int64_t row = tile * TM + r;
            const bool valid = row < A.n;
#pragma unroll
            for (int w = 0; w < 4; ++w) kb_cur[w] = kb_next[w];
            // ---- stage: X0 -> head of the DZ2 buffer; critic: action -> tail chunk of X2 ----
            float4 xin[3] = {xnext[0], xnext[1], xnext[2]};
            const float2 side = side_next;
            const float tgt = tgt_next;
            fetch(tile + gridDim.x);
            store_obs_half(xin, h2row, cs);               // (G1 of the previous tile may still be reading its X0 in the DZ2 buffer)
            if (NET == NET_CRITIC && cs == 0)
                *reinterpret_cast<uint4 *>(x2row + (H1 / 8) * CHUNK_A) = tail_chunk_critic(side.x, side.y);
            // every warp has arrived for the previous tile's G1 before any arrives for this tile's L1a (no wait lies between
            // the two arrivals, and a warp that arrived twice in one phase would complete it without the slowest one)
            if (tl_i > 0) asm volatile("bar.sync 1, 256;" ::: "memory");
            to_mma();                                     // -> L1a
            from_mma();                                   // (the commit behind L1a also retires the previous tile's G1)
            hidden1(0);
            to_mma();                                     // -> L1b
            from_mma();
            hidden1(1);
            to_mma();                                     // -> L2
            make_keep(tile + gridDim.x, 0, 0);            // in the shadow of the 17-step layer-2 chain
            make_keep(tile + gridDim.x, 0, 1);
            from_mma();
            // ---- output layer, loss / upstream gradient (fp32) ----
            float z0 = 0.f, z1 = 0.f;
            sweep_work(tl + T_WORK, cs, [&](const uint32_t (&v)[16], int j) {
#pragma unroll
                for (int c = 0; c < 16; ++c) {
                    const float h = fmaxf(__uint_as_float(v[c]), 0.f);
                    if (NET == NET_ACTOR) {
                        const float2 w = w3a[j * 16 + c];
                        z0 = fmaf(h, w.x, z0);
                        z1 = fmaf(h, w.y, z1);
                    } else {
                        z0 = fmaf(h, w3x[j * 16 + c].x, z0);
                    }
                }
            });
            {   // the row's output-layer sums: combine the column slices (slice 0 + slice 1: same order in every warp)
                float2 *zp = reinterpret_cast<float2 *>(smem + SM_ZP);
                zp[cs * TM + r] = make_float2(z0, z1);
                asm volatile("bar.sync 1, 256;" ::: "memory");
                const float2 pa = zp[r], pb = zp[TM + r];
                z0 = pa.x + pb.x;
                z1 = pa.y + pb.y;
            }
            float d0 = 0.f, d1 = 0.f;
            if (NET == NET_CRITIC) {
                if (valid) {                              // loss "mse": mean over the global batch
                    const float e = (z0 + b3[0]) - tgt;
                    stat += e * e;
                    d0 = 2.0f * e / (float)A.n_global;
                }
            } else if (valid) {                           // through tanh, upstream = -dQ/da (SkillshotLearner.py:408-410)
                stat += tgt;                              // Q of the row (reported sum)
                const float a0 = tanhf(z0 + b3[0]), a1 = tanhf(z1 + b3[1]);
                d0 = side.x * (1.0f - a0 * a0);
                d1 = side.y * (1.0f - a1 * a1);
            }
            if (cs != 0) stat = 0.f;                      // statistics and db3 are kept by slice 0 only
            else { dsum0 += d0; dsum1 += d1; }
            if (cs == 0) {
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
            make_keep(tile + gridDim.x, 1, 0);            // ... of G2's first half and BXa
            from_mma();                                   // dx2[:, :128] is there and h1[:, :128] has been consumed
            back1(0);                                     // (beside the rest of G2 and G3)
            to_mma();                                     // -> BXb
            make_keep(tile + gridDim.x, 1, 1);            // ... and of the rest of the weight-gradient group and BXb
            from_mma();                                   // ... which also retires G2 / G3: h1[:, 128:], h2, dz2 are free
            back1(1);
            store_obs_half(xin, dz2row, cs);              // X0 for G1 (the DZ2 buffer is free: BXb has retired)
            to_mma();                                     // -> G1, not waited for: it retires with the next tile's L1a
            ++tl_i;
        }
        from_mma();                                       // the last tile's G1

        // ======================= write this CTA's partial gradient =======================
        // thread r = hidden-2 unit r for dW2'^T and dW3^T, = hidden-1 unit 128 h + r for dW1'^T; columns split by slice
        {
#pragma unroll 1
            for (int j = cs; j < H1 / 16; j += NSLICE) {
                uint32_t v[16];
                tmem_ld16(tl + T_W2T + j * 16, v);
                tmem_wait_ld();
#pragma unroll
                for (int c = 0; c < 16; ++c) __stcg(g + P_W2 + (j * 16 + c) * H2 + r, __uint_as_float(v[c]));
            }
            uint32_t t[16];
            if (cs == 0) {
                tmem_ld16(tl + T_W2T + H1, t);
                tmem_wait_ld();
                if (NET == NET_ACTOR) {
                    __stcg(g + A_B2 + r, __uint_as_float(t[0]));
                } else {                                  // action rows (hi + lo parts of the action), then b2
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
            }
            {
                const int h = cs;                         // each slice dumps one half of dW1'^T
                uint32_t a[16], b[16];
                tmem_ld16(tl + T_W1T + h * 32, a);
                tmem_ld16(tl + T_W1T + h * 32 + 16, b);
                tmem_wait_ld();
#pragma unroll
                for (int i = 0; i < DS; ++i)
                    __stcg(g + P_W1 + i * H1 + h * 128 + r, __uint_as_float(a[i]) + __uint_as_float(b[i]));
                __stcg(g + P_B1 + h * 128 + r, __uint_as_float(a[12]));
            }
            // db3 and the loss statistic: sums over the rows (slice 0 holds them)
            if (cs == 0) {
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
                    if (NET == NET_ACTOR) { g[A_B3] = t0; g[A_B3 + 1] = t1; g[PN] = t2; }
                    else { g[C_B3] = t0; g[PN] = t2; }
                }
            }
        }
        tc_fence_before();
    } else {
        // ======================= the MMA-issuing warp =======================
        uint32_t ph = 0;
        const uint32_t work = tmem + T_WORK;
        const uint32_t b1 = sbase + SM_B1, b2 = sbase + SM_B2, x2 = sbase + SM_X2, dz2 = sbase + SM_DZ2;
        const uint32_t h2 = sbase + SM_H2, dz3 = sbase + SM_DZ3;
        constexpr uint32_t kFwd = umma_idesc(TM, 128);                // K-major x K-major
        constexpr uint32_t kBx = umma_idesc(TM, 128, 0, 1);           // dz2 (K-major) x W2 image (MN-major)
        constexpr uint32_t kG128 = umma_idesc(TM, 128, 1, 1), kG16 = umma_idesc(TM, 16, 1, 1), kG32 = umma_idesc(TM, 32, 1, 1);
        auto wait_epi = [&]() { mbar_wait(bar_mma, ph); ph ^= 1; tc_fence_after(); };
        uint32_t acc = 0;                                             // 0 on the CTA's first tile: accumulators start fresh
        for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x, acc = 1) {
            for (int half = 0; half < 2; ++half) {                    // L1a, L1b (X0 sits in the head of the H2 buffer)
                wait_epi();
                if (lane == 0) {
                    const uint64_t ad = desc_kmajor(h2, CHUNK_A), bd = desc_kmajor(b1 + half * 128 * 16, CHUNK_B1);
#pragma unroll
                    for (int ks = 0; ks < K1 / 16; ++ks)
                        umma_bf16(work, desc_advance(ad, 2 * CHUNK_A * ks), desc_advance(bd, 2 * CHUNK_B1 * ks), kFwd, ks > 0);
                    umma_commit(bar_epi);
                }
                __syncwarp();
            }
            wait_epi();                                               // L2
            if (lane == 0) {
                const uint64_t ad = desc_kmajor(x2, CHUNK_A), bd = desc_kmajor(b2, CHUNK_B2);
#pragma unroll
                for (int ks = 0; ks < K2 / 16; ++ks)
                    umma_bf16(work, desc_advance(ad, 2 * CHUNK_A * ks), desc_advance(bd, 2 * CHUNK_B2 * ks), kFwd, ks > 0);
                umma_commit(bar_epi);
            }
            __syncwarp();
            // The epilogue warps wait for nothing but dx2: what they need first goes first.  The first half of G2 consumes
            // h1[:, :128] (the chunks back1(0) overwrites with dz1), BXa delivers dx2[:, :128]; the commit behind those two
            // releases back1(0), which then runs beside the second half of G2, its bias / action columns and G3.
            wait_epi();                                               // G2, BXa, G3
            if (lane == 0) {
                const uint64_t h2t = desc_mnmajor(h2, CHUNK_A), dz3t = desc_mnmajor(dz3, CHUNK_A);
                const uint64_t dz2t = desc_mnmajor(dz2, CHUNK_A), x2t = desc_mnmajor(x2, CHUNK_A);
                const uint64_t x2hi = desc_mnmajor(x2 + 16 * CHUNK_A, CHUNK_A);
                const uint64_t x2tail = desc_mnmajor(x2 + (H1 / 8) * CHUNK_A, CHUNK_A);
#pragma unroll
                for (int ks = 0; ks < TM / 16; ++ks) {                // reduction over the 128 rows, 16 per step
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
            wait_epi();                                               // G1: no commit of its own, the next L1a's covers it
            if (lane == 0) {
                const uint64_t x0t = desc_mnmajor(dz2, CHUNK_A);
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                    const uint64_t dz1t = desc_mnmajor(x2 + half * 16 * CHUNK_A, CHUNK_A);
#pragma unroll
                    for (int ks = 0; ks < TM / 16; ++ks)
                        umma_bf16(tmem + T_W1T + half * 32, desc_advance(dz1t, 2 * CORE * ks), desc_advance(x0t, 2 * CORE * ks),
                                  kG32, acc | (ks > 0));
                }
            }
            __syncwarp();
        }
        if (lane == 0) umma_commit(bar_epi);                          // the last tile's G1
        __syncwarp();
    }

    __syncthreads();
    if (warp == MMA_WARP) {
        tc_fence_after();
        tmem_dealloc(tmem, 512);
    }
}

// grad[p] = sum over CTA slices in a fixed order (bit-identical from run to run): four interleaved
// groups of slices are summed by four threads per parameter and combined 0+1+2+3 through shared memory;
// aux[0] = the same sum of the slices' extra slot
__global__ void reduce_parts_kernel(const float *work, int parts, int n_params, float *grad, float *aux) {
    __shared__ float red[4][64];
    const int p = blockIdx.x * 64 + threadIdx.x, q = threadIdx.y;
    float s = 0.f;
    if (p <= n_params) {
#pragma unroll 10        // ten independent loads in flight per thread; the additions keep their order
        for (int c = q; c < parts; c += 4) s += __ldcg(work + (int64_t)c * (n_params + 1) + p);
    }
    red[q][threadIdx.x] = s;
    __syncthreads();
    if (q == 0 && p <= n_params) {
        const float t = ((red[0][threadIdx.x] + red[1][threadIdx.x]) + red[2][threadIdx.x]) + red[3][threadIdx.x];
        if (p < n_params) grad[p] = t;
        else if (aux) aux[0] = t;
    }
}

template <int NET>
int launch_grad(const GradArgs &A0, float *grad_out, float *aux_out, int64_t workspace_bytes, void *stream) {
    constexpr int PN = NET == NET_ACTOR ? A_N : C_N;
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return SS_ERR_CUDA;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return SS_ERR_CUDA;
    if (cudaFuncSetAttribute(mlp_grad_tc_kernel<NET>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SM_TOTAL) != cudaSuccess)
        return SS_ERR_CUDA;
    const int64_t tiles = (A0.n + TM - 1) / TM;
    int64_t cap = workspace_bytes / ((int64_t)(PN + 1) * 4);
    if (cap > sms) cap = sms;
    if (cap < 1) return SS_ERR_INVALID_ARG;
    // No more CTAs than the rounds need: 512 tiles on 148 SMs are four rounds whichever way, and 128 CTAs of four tiles stage
    // the weights 128 times instead of 148 (the staging is L2-bandwidth bound) and leave 128 gradient slices to reduce.
    const int64_t rounds = (tiles + cap - 1) / cap;
    const int grid = (int)((tiles + rounds - 1) / rounds);
    cudaStream_t st = (cudaStream_t)stream;
    GradArgs A1 = A0;
    A1.early_weights = sslaunch::take_early_weights();
    if (sslaunch::launch(mlp_grad_tc_kernel<NET>, dim3(grid), dim3(NTHREADS), SM_TOTAL, st, A1) != cudaSuccess) return SS_ERR_CUDA;
    if (!grad_out) return cudaGetLastError() == cudaSuccess ? grid : SS_ERR_CUDA;   // slices only (ss_peer_reduce_push follows)
    reduce_parts_kernel<<<(PN + 1 + 63) / 64, dim3(64, 4), 0, st>>>(A0.work, grid, PN, grad_out, aux_out);
    return cudaGetLastError() == cudaSuccess ? SS_OK : SS_ERR_CUDA;
}

// TD3 target policy smoothing of the target actions, one thread per row (ss_rng.cuh td3_smooth)
__global__ void td3_smooth_kernel(float2 *act, int64_t n, float sigma, float clip, uint64_t seed, uint64_t counter,
                                  int64_t row_offset) {
    const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n) return;
    float2 a = act[row];
    ss::td3_smooth(seed, counter, row_offset + row, sigma, clip, &a.x, &a.y);
    act[row] = a;
}

// the TD3 target from the two target critics' values: the TD epilogue of the forward kernels on min(q1, q2)
__global__ void td3_min_target_kernel(const float *q1, const float *q2, const float *reward, const uint8_t *done, float gamma,
                                      float *y, int64_t n) {
    const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n) return;
    y[row] = reward[row] + gamma * (done && done[row] ? 0.f : 1.f) * fminf(q1[row], q2[row]);
}

}  // namespace

int sstc::reduce_slices(const float *work, int parts, int n_params, float *grad, float *aux, cudaStream_t st) {
    reduce_parts_kernel<<<(n_params + 1 + 63) / 64, dim3(64, 4), 0, st>>>(work, parts, n_params, grad, aux);
    return cudaGetLastError() == cudaSuccess ? SS_OK : SS_ERR_CUDA;
}

int sstc::td3_smooth_actions(float *act, int64_t n, float sigma, float clip, uint64_t seed, uint64_t counter, int64_t row_offset,
                             cudaStream_t st) {
    td3_smooth_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>((float2 *)act, n, sigma, clip, seed, counter, row_offset);
    return cudaGetLastError() == cudaSuccess ? SS_OK : SS_ERR_CUDA;
}

int sstc::td3_min_target(const float *q1, const float *q2, const float *reward, const uint8_t *done, float gamma, float *y, int64_t n,
                         cudaStream_t st) {
    td3_min_target_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(q1, q2, reward, done, gamma, y, n);
    return cudaGetLastError() == cudaSuccess ? SS_OK : SS_ERR_CUDA;
}

extern "C" {

int ss_critic_grad_tc(const float *critic_params, const float *obs, const float *act, const float *target,
                      const uint8_t *dropout_keep, float dropout_rate, uint64_t seed, uint64_t counter,
                      int64_t n, int64_t n_global, int64_t row_offset, float *grad_out, float *sse_out,
                      void *workspace, int64_t workspace_bytes, void *stream) {
    if (!critic_params || !obs || !act || !target || !workspace || n <= 0) return SS_ERR_INVALID_ARG;
    if (dropout_rate < 0.f || dropout_rate >= 1.f) return SS_ERR_INVALID_ARG;
    if (((uintptr_t)critic_params | (uintptr_t)obs | (uintptr_t)dropout_keep) & 15 || ((uintptr_t)act & 7))
        return SS_ERR_INVALID_ARG;
    GradArgs A{};
    A.params = critic_params; A.obs = obs; A.act = act; A.target = target; A.keep = dropout_keep; A.rate = dropout_rate;
    A.seed = seed; A.counter = counter; A.n = n; A.n_global = n_global > 0 ? n_global : n; A.row_offset = row_offset;
    A.work = (float *)workspace;
    return launch_grad<NET_CRITIC>(A, grad_out, sse_out, workspace_bytes, stream);
}

// stage: 0 = the whole actor step; 1 = only a = actor(s) (it depends on neither network's pending update: a sharded update
// runs it while the critic's gradient exchange is in flight); 2 = the rest, with stage 1's actions in the scratch area
int ss_actor_grad_tc_staged(const float *actor_params, const float *critic_params, const float *obs, int64_t n,
                            float *grad_out, float *q_sum_out, void *workspace, int64_t workspace_bytes, int stage,
                            void *stream) {
    return ss_actor_grad_tc_paired(actor_params, critic_params, obs, n, grad_out, q_sum_out, workspace, workspace_bytes, stage,
                                   nullptr, stream);
}

// pair_mail != NULL (stage 0 only): a = actor(s) and critic([s, a]) run as one launch (ss_actor_critic_forward_tc)
int ss_actor_grad_tc_paired(const float *actor_params, const float *critic_params, const float *obs, int64_t n,
                            float *grad_out, float *q_sum_out, void *workspace, int64_t workspace_bytes, int stage,
                            void *pair_mail, void *stream) {
    if (!actor_params || !critic_params || !obs || !workspace || n <= 0 || stage < 0 || stage > 2) return SS_ERR_INVALID_ARG;
    if (((uintptr_t)actor_params | (uintptr_t)critic_params | (uintptr_t)obs | (uintptr_t)workspace) & 15)
        return SS_ERR_INVALID_ARG;
    // scratch behind the gradient slices: the actor's actions, -dQ/da and Q per row
    const int64_t scratch = ((n * 2 + 3) / 4 * 4) * 2 + (n + 3) / 4 * 4;
    const int64_t slice_bytes = workspace_bytes - scratch * 4;
    if (slice_bytes < (int64_t)(A_N + 1) * 4) return SS_ERR_INVALID_ARG;
    float *act = (float *)((char *)workspace + slice_bytes / 16 * 16);
    float *up = act + (n * 2 + 3) / 4 * 4;
    float *q = up + (n * 2 + 3) / 4 * 4;
    // a = actor(s);  q, -dq/da = critic([s, a]) with Dropout off;  then the actor's backward pass
    int rc;
    if (stage == 0 && pair_mail) {
        rc = ss_actor_critic_forward_tc(actor_params, critic_params, obs, act, n, q, up, nullptr, nullptr, 0.f, nullptr, pair_mail,
                                        stream);
        if (rc != SS_OK) return rc;
    } else {
        if (stage != 2) {
            rc = ss_actor_forward_tc(actor_params, obs, act, n, 0.f, 0, 0.f, 0, 0, stream);
            if (rc != SS_OK || stage == 1) return rc;
        }
        rc = ss_critic_forward_tc(critic_params, obs, act, n, q, up, nullptr, nullptr, 0.f, nullptr, stream);
        if (rc != SS_OK) return rc;
    }
    GradArgs A{};
    A.params = actor_params; A.obs = obs; A.up = up; A.q = q; A.n = n; A.n_global = n; A.work = (float *)workspace;
    // the rows' Q values are summed by the gradient kernel's row owners into the slices' extra slot: the fixed-order
    // reduction that follows (here or in ss_peer_reduce_push / ss_reduce_adam_tf) delivers sum Q without a kernel of its own
    return launch_grad<NET_ACTOR>(A, grad_out, q_sum_out, slice_bytes / 16 * 16, stream);
}

int ss_actor_grad_tc(const float *actor_params, const float *critic_params, const float *obs, int64_t n,
                     float *grad_out, float *q_sum_out, void *workspace, int64_t workspace_bytes, void *stream) {
    return ss_actor_grad_tc_staged(actor_params, critic_params, obs, n, grad_out, q_sum_out, workspace, workspace_bytes, 0, stream);
}

int ss_ddpg_targets_tc(const float *target_actor_params, const float *target_critic_params, const float *reward,
                       const float *next_obs, const uint8_t *done, float gamma, float *y_out, int64_t n,
                       void *workspace, int64_t workspace_bytes, void *stream) {
    return ss_ddpg_targets_tc_paired(target_actor_params, target_critic_params, reward, next_obs, done, gamma, y_out, n, workspace,
                                     workspace_bytes, nullptr, stream);
}

// pair_mail != NULL: actor'(s2) and critic'(s2, a2) run as one launch (ss_actor_critic_forward_tc)
int ss_ddpg_targets_tc_paired(const float *target_actor_params, const float *target_critic_params, const float *reward,
                              const float *next_obs, const uint8_t *done, float gamma, float *y_out, int64_t n,
                              void *workspace, int64_t workspace_bytes, void *pair_mail, void *stream) {
    if (!target_actor_params || !target_critic_params || !reward || !next_obs || !y_out || !workspace || n <= 0)
        return SS_ERR_INVALID_ARG;
    if (workspace_bytes < n * 8 || ((uintptr_t)workspace & 15)) return SS_ERR_INVALID_ARG;
    float *act = (float *)workspace;
    if (pair_mail)
        return ss_actor_critic_forward_tc(target_actor_params, target_critic_params, next_obs, act, n, nullptr, nullptr, reward, done,
                                          gamma, y_out, pair_mail, stream);
    int rc = ss_actor_forward_tc(target_actor_params, next_obs, act, n, 0.f, 0, 0.f, 0, 0, stream);
    if (rc != SS_OK) return rc;
    return ss_critic_forward_tc(target_critic_params, next_obs, act, n, nullptr, nullptr, reward, done, gamma, y_out, stream);
}

// actor'(s') -> [smoothing] -> critic'(s', a~) with the TD epilogue (one critic: ss_ddpg_targets_tc's two launches), or both
// critics' q -> td3_min_target.  workspace: [act n x 2 | q1 n | q2 n], each 16-byte aligned.
int ss_td3_targets_tc(const float *target_actor_params, const float *target_critic_params, const float *target_critic2_params,
                      const float *reward, const float *next_obs, const uint8_t *done, float gamma, float noise_sd, float noise_clip,
                      uint64_t seed, uint64_t counter, int64_t row_offset, float *y_out, int64_t n, void *workspace,
                      int64_t workspace_bytes, void *stream) {
    if (!target_actor_params || !target_critic_params || !reward || !next_obs || !y_out || !workspace || n <= 0 ||
        !(noise_sd >= 0.f) || !(noise_clip >= 0.f) || row_offset < 0)
        return SS_ERR_INVALID_ARG;
    if (((uintptr_t)target_actor_params | (uintptr_t)target_critic_params | (uintptr_t)target_critic2_params | (uintptr_t)next_obs |
         (uintptr_t)workspace) & 15)
        return SS_ERR_INVALID_ARG;
    const int64_t act_bytes = (n * 8 + 15) / 16 * 16, q_bytes = (n * 4 + 15) / 16 * 16;
    if (workspace_bytes < (target_critic2_params ? SS_TD3_TC_WORKSPACE_BYTES(n) : act_bytes)) return SS_ERR_INVALID_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    float *act = (float *)workspace;
    int rc = ss_actor_forward_tc(target_actor_params, next_obs, act, n, 0.f, 0, 0.f, 0, 0, stream);
    if (rc == SS_OK && noise_sd > 0.f) rc = td3_smooth_actions(act, n, noise_sd, noise_clip, seed, counter, row_offset, st);
    if (rc != SS_OK) return rc;
    if (!target_critic2_params)
        return ss_critic_forward_tc(target_critic_params, next_obs, act, n, nullptr, nullptr, reward, done, gamma, y_out, stream);
    float *q1 = (float *)((char *)workspace + act_bytes), *q2 = (float *)((char *)workspace + act_bytes + q_bytes);
    rc = ss_critic_forward_tc(target_critic_params, next_obs, act, n, q1, nullptr, nullptr, nullptr, 0.f, nullptr, stream);
    if (rc == SS_OK)
        rc = ss_critic_forward_tc(target_critic2_params, next_obs, act, n, q2, nullptr, nullptr, nullptr, 0.f, nullptr, stream);
    if (rc != SS_OK) return rc;
    return td3_min_target(q1, q2, reward, done, gamma, y_out, n, st);
}

}  // extern "C"
