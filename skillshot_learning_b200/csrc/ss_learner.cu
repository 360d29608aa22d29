// ss_learner.cu -- float32 kernels of the learner path and their C ABI
// (include/skillshot_b200.h): actor / critic forward, the critic's MSE gradient,
// the actor's deterministic-policy-gradient step, tf.keras Adam (+ soft target
// update), the replay ring, Philox parameter noise.
//
// This translation unit is the EXACT path: float32 everywhere, the arithmetic the
// reference's Keras graph does (SkillshotLearner.py:70-121, 245-281, 386-443).
// It serves the reference's own configuration (batches of 16, per-call parameter
// noise) and is the numerical yardstick for the bf16 tensor-core kernels of
// ss_mlp_tc.cu, which take over the large rollout batches.
//
// Scheme: a CTA of 256 threads owns a tile of 32 samples.  Activations live in
// shared memory TRANSPOSED, [feature][sample] with a row pitch of 36 floats, so a
// thread that owns one output unit sweeps the reduction dimension reading one
// coalesced weight (Keras kernels are [in][out], out contiguous) and broadcast
// float4s of the 32 samples.  Weight gradients are accumulated per CTA in a
// private slice of an L2-resident workspace and summed in a fixed order by
// reduce_kernel, so the result does not depend on scheduling (deterministic, and
// identical whatever the number of CTAs that took part).
#include <cuda_runtime.h>
#include <stdint.h>

#include <cmath>

#include "../../include/skillshot_b200.h"
#include "ss_launch.cuh"
#include "ss_rng.cuh"

namespace sstc {   // the tensor-core families of ss_critic_grad_weighted (ss_tc_common.cuh)
int critic_grad_tc_weighted(const float *critic_params, const float *obs, const float *act, const float *target,
                            const float *row_weight, float *td_abs_out, const uint8_t *dropout_keep, float dropout_rate,
                            uint64_t seed, uint64_t counter, int64_t n, int64_t n_global, int64_t row_offset, float *grad_out,
                            float *sse_out, void *workspace, int64_t workspace_bytes, cudaStream_t stream);
int critic_grad_frames_tc_weighted(const float *critic_params, int frames, const float *obs, const float *act, const float *target,
                                   const float *row_weight, float *td_abs_out, const uint8_t *dropout_keep, float dropout_rate,
                                   uint64_t seed, uint64_t counter, int64_t n, int64_t n_global, int64_t row_offset,
                                   float *grad_out, float *sse_out, void *workspace, int64_t workspace_bytes, cudaStream_t stream);
}  // namespace sstc

namespace {

using namespace ss;

constexpr int TB = 32;        // samples per tile
constexpr int PITCH = 36;     // floats per shared-memory row: conflict-free float4 row stores
constexpr int NT = 256;       // threads per CTA

constexpr int DS = SS_DIM_STATE, DA = SS_DIM_ACTION, H1 = SS_HIDDEN1, H2 = SS_HIDDEN2;
// flat parameter vectors in Keras get_weights() order
constexpr int A_W1 = 0, A_B1 = A_W1 + DS * H1, A_W2 = A_B1 + H1, A_B2 = A_W2 + H1 * H2, A_W3 = A_B2 + H2,
              A_B3 = A_W3 + H2 * DA, A_N = A_B3 + DA;
constexpr int C_W1 = 0, C_B1 = C_W1 + DS * H1, C_W2 = C_B1 + H1, C_B2 = C_W2 + (H1 + DA) * H2,
              C_W3 = C_B2 + H2, C_B3 = C_W3 + H2, C_N = C_B3 + 1;
static_assert(A_N == SS_ACTOR_PARAMS && C_N == SS_CRITIC_PARAMS, "parameter counts");

// The same two networks with a first layer of `ds` inputs instead of 12 (the frame-stacked "planning" networks of
// readme.md:18-20, ds = 12 * frames; ds = 12 is the reference): offsets of the six Keras arrays in the flat vectors.
struct Lay {
    int ds;
    int a_b1, a_w2, a_b2, a_w3, a_b3, a_n;       // actor:  W1[ds][256] b1 W2[256][128] b2 W3[128][2] b3
    int c_b1, c_w2, c_b2, c_w3, c_b3, c_n;       // critic: W1[ds][256] b1 W2[258][128] b2 W3[128][1] b3
};
__host__ __device__ inline Lay lay_of(int ds) {
    Lay L;
    L.ds = ds;
    L.a_b1 = ds * H1; L.a_w2 = L.a_b1 + H1; L.a_b2 = L.a_w2 + H1 * H2; L.a_w3 = L.a_b2 + H2; L.a_b3 = L.a_w3 + H2 * DA;
    L.a_n = L.a_b3 + DA;
    L.c_b1 = ds * H1; L.c_w2 = L.c_b1 + H1; L.c_b2 = L.c_w2 + (H1 + DA) * H2; L.c_w3 = L.c_b2 + H2; L.c_b3 = L.c_w3 + H2;
    L.c_n = L.c_b3 + 1;
    return L;
}

enum { ACT_NONE = 0, ACT_RELU = 1 };

__device__ __forceinline__ float4 ld4(const float *p) { return *reinterpret_cast<const float4 *>(p); }
__device__ __forceinline__ void st4(float *p, float4 v) { *reinterpret_cast<float4 *>(p) = v; }

// outT[j][t] = act(b[j] + sum_i W[i*N + j] * inT[i][t])        Dense, x @ W[in,out] + b
template <int N, int ACT>
__device__ __forceinline__ void dense_fwd(const float *W, const float *b, const float *inT, int K, float *outT) {
    constexpr int TPC = NT / N;       // threads per output unit (1 or 2)
    constexpr int TS = TB / TPC;      // samples per thread
    const int j = threadIdx.x % N, t0 = (threadIdx.x / N) * TS;
    float acc[TS];
    const float bias = b[j];
#pragma unroll
    for (int t = 0; t < TS; ++t) acc[t] = bias;
#pragma unroll 4
    for (int i = 0; i < K; ++i) {
        const float w = W[i * N + j];
        const float *row = inT + i * PITCH + t0;
#pragma unroll
        for (int q = 0; q < TS / 4; ++q) {
            const float4 x = ld4(row + 4 * q);
            acc[4 * q + 0] = fmaf(x.x, w, acc[4 * q + 0]);
            acc[4 * q + 1] = fmaf(x.y, w, acc[4 * q + 1]);
            acc[4 * q + 2] = fmaf(x.z, w, acc[4 * q + 2]);
            acc[4 * q + 3] = fmaf(x.w, w, acc[4 * q + 3]);
        }
    }
    float *o = outT + j * PITCH + t0;
#pragma unroll
    for (int q = 0; q < TS / 4; ++q) {
        float4 v = make_float4(acc[4 * q], acc[4 * q + 1], acc[4 * q + 2], acc[4 * q + 3]);
        if (ACT == ACT_RELU) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
        st4(o + 4 * q, v);
    }
}

// Back-propagation to a hidden layer of H1 units through a [.., H2] kernel whose
// first H1 rows are W:  d[i][t] = sum_k W[i*H2 + k] * doutT[k][t], then the ReLU
// (and inverted-dropout) mask of the layer's own output held in ioT:
// ioT[i][t] = ioT[i][t] > 0 ? d * scale : 0.   Thread i owns row i.
__device__ __forceinline__ void dense_bwd_input(const float *W, const float *doutT, float *ioT, float scale) {
    const int i = threadIdx.x;
    float acc[TB];
#pragma unroll
    for (int t = 0; t < TB; ++t) acc[t] = 0.f;
    const float *wrow = W + i * H2;
#pragma unroll 1
    for (int k4 = 0; k4 < H2 / 4; ++k4) {
        const float4 w = ld4(wrow + 4 * k4);
        const float wk[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
            const float *row = doutT + (4 * k4 + kk) * PITCH;
#pragma unroll
            for (int q = 0; q < TB / 4; ++q) {
                const float4 x = ld4(row + 4 * q);
                acc[4 * q + 0] = fmaf(x.x, wk[kk], acc[4 * q + 0]);
                acc[4 * q + 1] = fmaf(x.y, wk[kk], acc[4 * q + 1]);
                acc[4 * q + 2] = fmaf(x.z, wk[kk], acc[4 * q + 2]);
                acc[4 * q + 3] = fmaf(x.w, wk[kk], acc[4 * q + 3]);
            }
        }
    }
    float *o = ioT + i * PITCH;
#pragma unroll
    for (int q = 0; q < TB / 4; ++q) {
        const float4 h = ld4(o + 4 * q);
        st4(o + 4 * q, make_float4(h.x > 0.f ? acc[4 * q] * scale : 0.f, h.y > 0.f ? acc[4 * q + 1] * scale : 0.f,
                                   h.z > 0.f ? acc[4 * q + 2] * scale : 0.f, h.w > 0.f ? acc[4 * q + 3] * scale : 0.f));
    }
}

// CTA-private gradient slice in the workspace: first tile overwrites, later tiles add.
__device__ __forceinline__ void accum(float *p, float v, bool first) {
    __stcg(p, first ? v : __ldcg(p) + v);
}

// gW[i*N + k] += sum_t inT[i][t] * doutT[k][t]  (i < K);   gb[k] += sum_t doutT[k][t]
template <int N>
__device__ __forceinline__ void dense_bwd_weight(const float *inT, int K, const float *doutT, float *gW, float *gb,
                                                 bool first) {
    constexpr int TPC = NT / N;
    const int k = threadIdx.x % N, part = threadIdx.x / N;
    float dz[TB];
#pragma unroll
    for (int q = 0; q < TB / 4; ++q) {
        const float4 x = ld4(doutT + k * PITCH + 4 * q);
        dz[4 * q] = x.x; dz[4 * q + 1] = x.y; dz[4 * q + 2] = x.z; dz[4 * q + 3] = x.w;
    }
    if (part == 0) {
        float s = 0.f;
#pragma unroll
        for (int t = 0; t < TB; ++t) s += dz[t];
        accum(gb + k, s, first);
    }
#pragma unroll 2
    for (int i = part; i < K; i += TPC) {
        const float *row = inT + i * PITCH;
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
        for (int q = 0; q < TB / 4; ++q) {
            const float4 x = ld4(row + 4 * q);
            a0 = fmaf(x.x, dz[4 * q + 0], a0);
            a1 = fmaf(x.y, dz[4 * q + 1], a1);
            a2 = fmaf(x.z, dz[4 * q + 2], a2);
            a3 = fmaf(x.w, dz[4 * q + 3], a3);
        }
        accum(gW + i * N + k, (a0 + a1) + (a2 + a3), first);
    }
}

// rows of a [n][W] float32 matrix -> transposed tile dstT[c][t], zero beyond n
template <int W>
__device__ __forceinline__ void load_tile_T(const float *src, int64_t base, int64_t n, float *dstT) {
    for (int e = threadIdx.x; e < TB * W; e += NT) {
        const int t = e / W, c = e - t * W;
        dstT[c * PITCH + t] = (base + t < n) ? src[(base + t) * W + c] : 0.f;
    }
}

// the same with a run-time row width (frame-stacked inputs)
__device__ __forceinline__ void load_tile_rt(const float *src, int64_t base, int64_t n, float *dstT, int w) {
    for (int e = threadIdx.x; e < TB * w; e += NT) {
        const int t = e / w, c = e - t * w;
        dstT[c * PITCH + t] = (base + t < n) ? src[(base + t) * w + c] : 0.f;
    }
}

// actor output layer: aT[m][t] = tanh(b3[m] + sum_k W3[k*2 + m] * h2T[k][t])
__device__ __forceinline__ void actor_out(const float *W3, const float *b3, const float *h2T, float *aT) {
    if (threadIdx.x < TB * DA) {
        const int t = threadIdx.x & (TB - 1), m = threadIdx.x / TB;
        float z = b3[m];
#pragma unroll 8
        for (int k = 0; k < H2; ++k) z = fmaf(W3[k * DA + m], h2T[k * PITCH + t], z);
        aT[m * PITCH + t] = tanhf(z);
    }
}
// critic output layer: q[t] = b3 + sum_k W3[k] * h2T[k][t]
__device__ __forceinline__ void critic_out(const float *W3, const float *b3, const float *h2T, float *q) {
    if (threadIdx.x < TB) {
        const int t = threadIdx.x;
        float z = b3[0];
#pragma unroll 8
        for (int k = 0; k < H2; ++k) z = fmaf(W3[k], h2T[k * PITCH + t], z);
        q[t] = z;
    }
}

// ---------------------------------------------------------------------------
// actor forward (+ parameter noise, + action noise)
// ---------------------------------------------------------------------------
struct ActorFwdArgs {
    const float *theta, *obs;
    float *act;
    int64_t n, group;           // samples; samples per parameter-noise draw
    float param_sd, action_sd;
    uint64_t seed, counter;
};

// model_act / model_act_action_noise / model_act_param_noise (SkillshotLearner.py:215-281)
// without the env side effects.  NOISY: the CTA keeps a private perturbed copy of
// the 36,482 actor parameters in shared memory, w + w * (sd * eps), eps ~ N(0,1) from
// Philox keyed by (parameter index, noise group, counter): group size 1 is the
// reference's fresh draw per call, larger groups share one draw between
// consecutive samples.
template <bool NOISY>
__global__ void __launch_bounds__(NT) actor_fwd_kernel(const ActorFwdArgs A) {
    extern __shared__ __align__(16) float smem[];
    float *sT = smem, *h1T = sT + DS * PITCH, *h2T = h1T + H1 * PITCH, *aT = h2T + H2 * PITCH;
    float *wS = aT + DA * PITCH;
    const float *P = NOISY ? wS : A.theta;

    // work units never straddle a noise group
    const int64_t group = NOISY ? A.group : A.n;
    const int64_t upg = (group + TB - 1) / TB;
    const int64_t n_groups = (A.n + group - 1) / group;
    const int64_t units = n_groups * upg;
    const int64_t u0 = units * blockIdx.x / gridDim.x, u1 = units * (blockIdx.x + 1) / gridDim.x;
    int64_t have_group = -1;
    for (int64_t u = u0; u < u1; ++u) {
        const int64_t g = u / upg, base = g * group + (u - g * upg) * TB;
        const int64_t end = min(A.n, (g + 1) * group);
        if (base >= end) continue;
        __syncthreads();                                  // previous unit done with smem
        if (NOISY && g != have_group) {
            for (int q = threadIdx.x; q < (A_N + 3) / 4; q += NT) {
                float z[4];
                normal4(A.seed, kTagParamNoise, (uint32_t)q, (uint32_t)g, A.counter, z);
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int p = 4 * q + e;
                    if (p < A_N) { const float w = A.theta[p]; wS[p] = w + w * (A.param_sd * z[e]); }
                }
            }
            have_group = g;
        }
        load_tile_T<DS>(A.obs, base, end, sT);
        __syncthreads();
        dense_fwd<H1, ACT_RELU>(P + A_W1, P + A_B1, sT, DS, h1T);
        __syncthreads();
        dense_fwd<H2, ACT_RELU>(P + A_W2, P + A_B2, h1T, H1, h2T);
        __syncthreads();
        actor_out(P + A_W3, P + A_B3, h2T, aT);
        __syncthreads();
        if (threadIdx.x < TB && base + threadIdx.x < end) {
            const int64_t row = base + threadIdx.x;
            float a0 = aT[threadIdx.x], a1 = aT[PITCH + threadIdx.x];
            if (A.action_sd > 0.f) {                      // predictions += N(0, sd), SkillshotLearner.py:238
                float z[4];
                normal4(A.seed, kTagActionNoise, (uint32_t)row, (uint32_t)(row >> 32), A.counter, z);
                a0 += A.action_sd * z[0];
                a1 += A.action_sd * z[1];
            }
            reinterpret_cast<float2 *>(A.act)[row] = make_float2(a0, a1);
        }
    }
}

// ---------------------------------------------------------------------------
// frame-stacked ("planning") actor: readme.md:18-20 -- no reference code, parity unpinned
// ---------------------------------------------------------------------------
// The actor sees the last `frames` observations of a player instead of one: first layer 12 * frames -> 256, the rest
// unchanged.  Parameters: one flat vector [W1[12 F][256] b1 W2 b2 W3 b3] in the same Keras order; frames = 1 IS the
// reference actor.  The observation history is a ring per row, stack[row][slot][12]; `head` is the slot of the newest
// frame and the network input is ordered oldest -> newest.  Parameter noise comes as ready-made vectors, one per
// noise group (ss_param_noise_groups): group g of `group` consecutive rows uses theta + g * stride.
struct FramesFwdArgs {
    const float *theta, *stack;
    float *act;
    int64_t n, group, stride, head;
    int frames;
};

__global__ void __launch_bounds__(NT) actor_frames_fwd_kernel(const FramesFwdArgs A) {
    extern __shared__ __align__(16) float smem[];
    const int dsf = DS * A.frames;
    float *sT = smem, *h1T = sT + dsf * PITCH, *h2T = h1T + H1 * PITCH, *aT = h2T + H2 * PITCH;
    const int w1 = 0, b1 = dsf * H1, w2 = b1 + H1, b2 = w2 + H1 * H2, w3 = b2 + H2, b3 = w3 + H2 * DA;
    const int64_t upg = (A.group + TB - 1) / TB, n_groups = (A.n + A.group - 1) / A.group, units = n_groups * upg;
    for (int64_t u = blockIdx.x; u < units; u += gridDim.x) {
        const int64_t g = u / upg, base = g * A.group + (u - g * upg) * TB;
        const int64_t end = min(A.n, (g + 1) * A.group);
        if (base >= end) continue;
        const float *P = A.theta + g * A.stride;
        __syncthreads();
        for (int e = threadIdx.x; e < TB * dsf; e += NT) {
            const int t = e / dsf, c = e - t * dsf, f = c / DS, j = c - f * DS;
            const int slot = (int)((A.head + 1 + f) % A.frames);                  // oldest frame first
            sT[c * PITCH + t] = (base + t < end) ? A.stack[((base + t) * A.frames + slot) * DS + j] : 0.f;
        }
        __syncthreads();
        dense_fwd<H1, ACT_RELU>(P + w1, P + b1, sT, dsf, h1T);
        __syncthreads();
        dense_fwd<H2, ACT_RELU>(P + w2, P + b2, h1T, H1, h2T);
        __syncthreads();
        actor_out(P + w3, P + b3, h2T, aT);
        __syncthreads();
        if (threadIdx.x < TB && base + threadIdx.x < end)
            reinterpret_cast<float2 *>(A.act)[base + threadIdx.x] = make_float2(aT[threadIdx.x], aT[PITCH + threadIdx.x]);
    }
}

// stack[row][head % frames] = obs[row]; a row whose game has just restarted gets the new observation in every slot
__global__ void obs_stack_push_kernel(float *stack, int64_t n_rows, int frames, int64_t head, const float *obs,
                                      const uint8_t *done, int done_div) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= 3 * n_rows) return;
    const int64_t row = e / 3, part = e - row * 3;
    const float4 v = reinterpret_cast<const float4 *>(obs)[e];
    float4 *dst = reinterpret_cast<float4 *>(stack) + row * frames * 3 + part;
    if (done && done[row / done_div]) {
        for (int f = 0; f < frames; ++f) dst[f * 3] = v;
    } else {
        dst[(head % frames) * 3] = v;
    }
}

// out[row][f][12] = stack[row][(head + 1 + f) % frames][12]: the network input, oldest frame first, as dense rows
__global__ void obs_stack_ordered_kernel(const float *stack, int64_t n_rows, int frames, int64_t head, float *out) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int w4 = 3 * frames;
    if (e >= w4 * n_rows) return;
    const int64_t row = e / w4;
    const int q = (int)(e - row * w4), f = q / 3, part = q - 3 * f;
    const int slot = (int)((head + 1 + f) % frames);
    reinterpret_cast<float4 *>(out)[e] = reinterpret_cast<const float4 *>(stack)[(row * frames + slot) * 3 + part];
}

__global__ void param_noise_groups_kernel(const float *theta, float *out, int64_t n_params, int64_t stride, float sd,
                                          uint64_t seed, uint64_t counter) {
    const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (4 * q >= n_params) return;
    float z[4];
    normal4_fast(seed, kTagParamNoise, (uint32_t)q, (uint32_t)blockIdx.y, counter, z);
    float *dst = out + (int64_t)blockIdx.y * stride;
    if (4 * q + 3 < n_params) {          // parameter vectors are 16-byte aligned and stride % 4 == 0
        const float4 w = __ldg(reinterpret_cast<const float4 *>(theta) + q);
        reinterpret_cast<float4 *>(dst)[q] = make_float4(w.x + w.x * (sd * z[0]), w.y + w.y * (sd * z[1]), w.z + w.z * (sd * z[2]),
                                                         w.w + w.w * (sd * z[3]));
    } else {
        for (int e = 0; e < 4; ++e) {
            const int64_t p = 4 * q + e;
            if (p < n_params) { const float w = theta[p]; dst[p] = w + w * (sd * z[e]); }
        }
    }
}

// The perturbed parameter vector itself (tests, and the host facade's introspection).
__global__ void param_noise_kernel(const float *theta, float *out, int64_t n_params, float sd, uint64_t seed,
                                   uint64_t group, uint64_t counter) {
    const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (4 * q >= n_params) return;
    float z[4];
    normal4(seed, kTagParamNoise, (uint32_t)q, (uint32_t)group, counter, z);
    for (int e = 0; e < 4; ++e) {
        const int64_t p = 4 * q + e;
        if (p < n_params) { const float w = theta[p]; out[p] = w + w * (sd * z[e]); }
    }
}

// ---------------------------------------------------------------------------
// critic forward, optionally on the actor's own action, optionally as TD target
// ---------------------------------------------------------------------------
struct CriticFwdArgs {
    const float *theta;      // actor parameters, or NULL: use `act`
    const float *phi, *obs, *act;
    const float *reward;     // NULL: out = q;  else out = reward + gamma * (1 - done) * q
    const uint8_t *done;
    float gamma;
    float *out;
    int64_t n;
    int ds;                  // input width: 12 (reference) or 12 * frames
};

template <bool WITH_ACTOR>
__global__ void __launch_bounds__(NT) critic_fwd_kernel(const CriticFwdArgs A) {
    extern __shared__ __align__(16) float smem[];
    const Lay L = lay_of(A.ds);
    float *sT = smem, *x2T = sT + L.ds * PITCH, *c2T = x2T + (H1 + DA) * PITCH, *qv = c2T + H2 * PITCH;
    float *h1T = qv + TB, *h2T = h1T + H1 * PITCH;       // WITH_ACTOR only
    const int64_t tiles = (A.n + TB - 1) / TB;
    for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        const int64_t base = tile * TB;
        __syncthreads();
        load_tile_rt(A.obs, base, A.n, sT, L.ds);
        if (!WITH_ACTOR) load_tile_T<DA>(A.act, base, A.n, x2T + H1 * PITCH);
        __syncthreads();
        if (WITH_ACTOR) {
            dense_fwd<H1, ACT_RELU>(A.theta, A.theta + L.a_b1, sT, L.ds, h1T);
            __syncthreads();
            dense_fwd<H2, ACT_RELU>(A.theta + L.a_w2, A.theta + L.a_b2, h1T, H1, h2T);
            __syncthreads();
            actor_out(A.theta + L.a_w3, A.theta + L.a_b3, h2T, x2T + H1 * PITCH);
        }
        dense_fwd<H1, ACT_RELU>(A.phi, A.phi + L.c_b1, sT, L.ds, x2T);
        __syncthreads();
        dense_fwd<H2, ACT_RELU>(A.phi + L.c_w2, A.phi + L.c_b2, x2T, H1 + DA, c2T);
        __syncthreads();
        critic_out(A.phi + L.c_w3, A.phi + L.c_b3, c2T, qv);
        __syncthreads();
        if (threadIdx.x < TB && base + threadIdx.x < A.n) {
            const int64_t row = base + threadIdx.x;
            float q = qv[threadIdx.x];
            if (A.reward) q = A.reward[row] + A.gamma * (A.done && A.done[row] ? 0.f : 1.f) * q;
            A.out[row] = q;
        }
    }
}

// ---------------------------------------------------------------------------
// TD3 target (no reference code, DESIGN.md section 6.14):
//   a~ = clamp(mu'(s') + clamp(sigma eps, -c, c), -1, 1);  y = r + gamma (1 - d) min(Q1'(s', a~), Q2'(s', a~))
// critic_fwd_kernel<true>'s tile loop with the smoothing between the actor and the critic and a second critic pass;
// with phi2 == NULL and sigma == 0 every operation is that kernel's, so y is ss_ddpg_targets_frames' bit for bit.
// ---------------------------------------------------------------------------
struct Td3TargetArgs {
    const float *theta, *phi, *phi2;     // target actor, target critics (phi2 NULL: one critic)
    const float *reward, *obs;           // obs = s'
    const uint8_t *done;
    float gamma, sigma, clip;
    uint64_t seed, counter;
    int64_t row_offset;                  // global index of row 0 (the smoothing draw of a shard)
    float *out;
    int64_t n;
    int ds;
};

__global__ void __launch_bounds__(NT) td3_target_kernel(const Td3TargetArgs A) {
    extern __shared__ __align__(16) float smem[];
    const Lay L = lay_of(A.ds);
    float *sT = smem, *x2T = sT + L.ds * PITCH, *c2T = x2T + (H1 + DA) * PITCH, *qv = c2T + H2 * PITCH;
    float *h1T = qv + TB, *h2T = h1T + H1 * PITCH, *qv2 = h2T + H2 * PITCH;
    const int64_t tiles = (A.n + TB - 1) / TB;
    for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        const int64_t base = tile * TB;
        __syncthreads();
        load_tile_rt(A.obs, base, A.n, sT, L.ds);
        __syncthreads();
        dense_fwd<H1, ACT_RELU>(A.theta, A.theta + L.a_b1, sT, L.ds, h1T);
        __syncthreads();
        dense_fwd<H2, ACT_RELU>(A.theta + L.a_w2, A.theta + L.a_b2, h1T, H1, h2T);
        __syncthreads();
        actor_out(A.theta + L.a_w3, A.theta + L.a_b3, h2T, x2T + H1 * PITCH);
        if (A.sigma > 0.f) {                      // (uniform over the CTA) one thread per row smooths both actions
            __syncthreads();
            if (threadIdx.x < TB && base + threadIdx.x < A.n) {
                float *a = x2T + H1 * PITCH + threadIdx.x;
                td3_smooth(A.seed, A.counter, A.row_offset + base + threadIdx.x, A.sigma, A.clip, a, a + PITCH);
            }
        }
        dense_fwd<H1, ACT_RELU>(A.phi, A.phi + L.c_b1, sT, L.ds, x2T);
        __syncthreads();
        dense_fwd<H2, ACT_RELU>(A.phi + L.c_w2, A.phi + L.c_b2, x2T, H1 + DA, c2T);
        __syncthreads();
        critic_out(A.phi + L.c_w3, A.phi + L.c_b3, c2T, qv);
        if (A.phi2) {
            dense_fwd<H1, ACT_RELU>(A.phi2, A.phi2 + L.c_b1, sT, L.ds, x2T);
            __syncthreads();
            dense_fwd<H2, ACT_RELU>(A.phi2 + L.c_w2, A.phi2 + L.c_b2, x2T, H1 + DA, c2T);
            __syncthreads();
            critic_out(A.phi2 + L.c_w3, A.phi2 + L.c_b3, c2T, qv2);
        }
        __syncthreads();
        if (threadIdx.x < TB && base + threadIdx.x < A.n) {
            const int64_t row = base + threadIdx.x;
            float q = qv[threadIdx.x];
            if (A.phi2) q = fminf(q, qv2[threadIdx.x]);
            q = A.reward[row] + A.gamma * (A.done && A.done[row] ? 0.f : 1.f) * q;
            A.out[row] = q;
        }
    }
}

// ---------------------------------------------------------------------------
// critic MSE gradient (one Keras fit batch, SkillshotLearner.py:434)
// ---------------------------------------------------------------------------
struct CriticGradArgs {
    const float *phi, *obs, *act, *target;
    const uint8_t *keep;     // injected dropout mask [n][256] (1 = keep), or NULL: Philox
    float rate;              // dropout rate (0 = off)
    uint64_t seed, counter;
    int64_t n, n_global, row_offset;   // row_offset: global index of row 0 (Philox dropout of a shard)
    float *work;             // [gridDim.x][c_n + 1]
    int ds;                  // input width: 12 (reference) or 12 * frames
    const float *row_weight; // WEIGHTED: the loss weight of each row [n] or NULL (1)
    float *td_abs;           // WEIGHTED: |q - target| of each row [n] or NULL
};

// critic_grad_kernel's body; WEIGHTED (critic_grad_weighted_kernel, ss_critic_grad_weighted) multiplies each row's loss
// gradient by its weight and stores |e|
template <bool WEIGHTED>
__device__ __forceinline__ void critic_grad_tiles(const CriticGradArgs &A) {
    extern __shared__ __align__(16) float smem[];
    const Lay L = lay_of(A.ds);
    const int C_B1 = L.c_b1, C_W2 = L.c_w2, C_B2 = L.c_b2, C_W3 = L.c_w3, C_B3 = L.c_b3, C_N = L.c_n, C_W1 = 0;
    float *sT = smem, *x2T = sT + L.ds * PITCH, *h2T = x2T + (H1 + DA) * PITCH, *qv = h2T + H2 * PITCH, *dq = qv + TB;
    float *g = A.work + (int64_t)blockIdx.x * (C_N + 1);
    const float inv_keep = A.rate > 0.f ? 1.0f / (1.0f - A.rate) : 1.0f;
    const int64_t tiles = (A.n + TB - 1) / TB;
    float sse = 0.f;
    bool first = true;
    for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x, first = false) {
        const int64_t base = tile * TB;
        __syncthreads();
        load_tile_rt(A.obs, base, A.n, sT, L.ds);
        load_tile_T<DA>(A.act, base, A.n, x2T + H1 * PITCH);
        __syncthreads();
        dense_fwd<H1, ACT_RELU>(A.phi + C_W1, A.phi + C_B1, sT, L.ds, x2T);
        if (A.rate > 0.f) {                                 // Dropout(0.2), training=True: h * keep / (1 - rate)
            const int j = threadIdx.x;                      // this thread wrote row j
            float *row = x2T + j * PITCH;
            if (A.keep) {
                for (int t = 0; t < TB; ++t)
                    row[t] = (base + t < A.n && A.keep[(base + t) * H1 + j]) ? row[t] * inv_keep : 0.f;
            } else {
                // one Philox draw per (global row, 8 units): 16 bits per unit, this thread's unit is lane j % 8
                // (the keying of the tensor-core kernel, where a thread owns a row: ss_mlp_grad_tc.cu)
                const uint32_t thresh16 = (uint32_t)(A.rate * 65536.0f);
                for (int t = 0; t < TB; ++t) {
                    const uint64_t grow = (uint64_t)(A.row_offset + base + t);
                    const U4 u = draw4(A.seed, kTagDropout, (uint32_t)grow, (uint32_t)(j >> 3) | ((uint32_t)(grow >> 32) << 8),
                                       A.counter);
                    const int e = j & 7;
                    const uint32_t w = (e >> 1) == 0 ? u.x : (e >> 1) == 1 ? u.y : (e >> 1) == 2 ? u.z : u.w;
                    const uint32_t v = (e & 1) ? (w >> 16) : (w & 0xFFFFu);
                    row[t] = v >= thresh16 ? row[t] * inv_keep : 0.f;
                }
            }
        }
        __syncthreads();
        dense_fwd<H2, ACT_RELU>(A.phi + C_W2, A.phi + C_B2, x2T, H1 + DA, h2T);
        __syncthreads();
        critic_out(A.phi + C_W3, A.phi + C_B3, h2T, qv);
        __syncthreads();
        if (threadIdx.x < TB) {                             // loss "mse": mean over the (global) batch
            const int t = threadIdx.x;
            float d = 0.f;
            if (base + t < A.n) {
                const float e = qv[t] - A.target[base + t];
                sse += e * e;
                d = 2.0f * e / (float)A.n_global;
                if (WEIGHTED) {                             // (the weight last: w = 1 leaves d as it is)
                    if (A.row_weight) d = d * A.row_weight[base + t];
                    if (A.td_abs) A.td_abs[base + t] = fabsf(e);
                }
            }
            dq[t] = d;
        }
        __syncthreads();
        if (threadIdx.x < H2) {                             // output layer gradients; then dz2 in place
            const int k = threadIdx.x;
            float *row = h2T + k * PITCH;
            const float w3 = A.phi[C_W3 + k];
            float s = 0.f;
#pragma unroll
            for (int t = 0; t < TB; ++t) {
                const float h = row[t], d = dq[t];
                s = fmaf(h, d, s);
                row[t] = h > 0.f ? d * w3 : 0.f;
            }
            accum(g + C_W3 + k, s, first);
        } else if (threadIdx.x == H2) {
            float s = 0.f;
            for (int t = 0; t < TB; ++t) s += dq[t];
            accum(g + C_B3, s, first);
        }
        __syncthreads();
        dense_bwd_weight<H2>(x2T, H1 + DA, h2T, g + C_W2, g + C_B2, first);
        __syncthreads();
        dense_bwd_input(A.phi + C_W2, h2T, x2T, inv_keep);
        __syncthreads();
        dense_bwd_weight<H1>(sT, L.ds, x2T, g + C_W1, g + C_B1, first);
    }
    // sum of squared errors of this CTA's tiles (threads 0..31 hold the partial sums)
    if (threadIdx.x < 32) {
        for (int o = 16; o > 0; o >>= 1) sse += __shfl_xor_sync(0xffffffffu, sse, o);
        if (threadIdx.x == 0) g[C_N] = sse;
    }
    if (first) {   // this CTA had no tile: its slice must still read as zero
        for (int p = threadIdx.x; p < C_N; p += NT) g[p] = 0.f;
    }
}

__global__ void __launch_bounds__(NT) critic_grad_kernel(const CriticGradArgs A) { critic_grad_tiles<false>(A); }
__global__ void __launch_bounds__(NT) critic_grad_weighted_kernel(const CriticGradArgs A) { critic_grad_tiles<true>(A); }

// ---------------------------------------------------------------------------
// actor deterministic-policy-gradient (model_actor_fit_step, SkillshotLearner.py:386-417)
// ---------------------------------------------------------------------------
struct ActorGradArgs {
    const float *theta, *phi, *obs;
    int64_t n;
    float *work;             // [gridDim.x][a_n + 1]
    int ds;                  // input width: 12 (reference) or 12 * frames
};

__global__ void __launch_bounds__(NT) actor_grad_kernel(const ActorGradArgs A) {
    extern __shared__ __align__(16) float smem[];
    const Lay L = lay_of(A.ds);
    const int A_W1 = 0, A_B1 = L.a_b1, A_W2 = L.a_w2, A_B2 = L.a_b2, A_W3 = L.a_w3, A_B3 = L.a_b3, A_N = L.a_n;
    const int C_W1 = 0, C_B1 = L.c_b1, C_W2 = L.c_w2, C_B2 = L.c_b2, C_W3 = L.c_w3, C_B3 = L.c_b3;
    float *sT = smem, *h1T = sT + L.ds * PITCH, *h2T = h1T + H1 * PITCH, *aT = h2T + H2 * PITCH;
    float *x2T = aT + DA * PITCH, *c2T = x2T + (H1 + DA) * PITCH, *dz3T = c2T + H2 * PITCH, *qv = dz3T + DA * PITCH;
    float *g = A.work + (int64_t)blockIdx.x * (A_N + 1);
    const int64_t tiles = (A.n + TB - 1) / TB;
    float qsum = 0.f;
    bool first = true;
    for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x, first = false) {
        const int64_t base = tile * TB;
        __syncthreads();
        load_tile_rt(A.obs, base, A.n, sT, L.ds);
        __syncthreads();
        // a = actor(s)
        dense_fwd<H1, ACT_RELU>(A.theta + A_W1, A.theta + A_B1, sT, L.ds, h1T);
        // critic's first layer depends on s only (model called directly: Dropout off)
        dense_fwd<H1, ACT_RELU>(A.phi + C_W1, A.phi + C_B1, sT, L.ds, x2T);
        __syncthreads();
        dense_fwd<H2, ACT_RELU>(A.theta + A_W2, A.theta + A_B2, h1T, H1, h2T);
        __syncthreads();
        actor_out(A.theta + A_W3, A.theta + A_B3, h2T, aT);
        __syncthreads();
        if (threadIdx.x < TB * DA) {
            const int t = threadIdx.x & (TB - 1), m = threadIdx.x / TB;
            x2T[(H1 + m) * PITCH + t] = aT[m * PITCH + t];
        }
        __syncthreads();
        // q = critic([s, a])
        dense_fwd<H2, ACT_RELU>(A.phi + C_W2, A.phi + C_B2, x2T, H1 + DA, c2T);
        __syncthreads();
        critic_out(A.phi + C_W3, A.phi + C_B3, c2T, qv);
        __syncthreads();
        if (threadIdx.x < TB && base + threadIdx.x < A.n) qsum += qv[threadIdx.x];
        // dq/da: only the two action rows of the critic's second kernel matter
        if (threadIdx.x < TB * DA) {
            const int t = threadIdx.x & (TB - 1), m = threadIdx.x / TB;
            const float *w = A.phi + C_W2 + (H1 + m) * H2;
            float da = 0.f;
#pragma unroll 8
            for (int k = 0; k < H2; ++k) da = fmaf(c2T[k * PITCH + t] > 0.f ? A.phi[C_W3 + k] : 0.f, w[k], da);
            const float a = aT[m * PITCH + t];
            // output_gradients = -dq/da (SkillshotLearner.py:410), through tanh
            dz3T[m * PITCH + t] = (base + t < A.n) ? -da * (1.0f - a * a) : 0.f;
        }
        __syncthreads();
        if (threadIdx.x < H2) {                             // actor output layer gradients; dz2 -> c2T
            const int k = threadIdx.x;
            const float w0 = A.theta[A_W3 + k * DA], w1 = A.theta[A_W3 + k * DA + 1];
            const float *hrow = h2T + k * PITCH;
            float *orow = c2T + k * PITCH;
            float s0 = 0.f, s1 = 0.f;
#pragma unroll
            for (int t = 0; t < TB; ++t) {
                const float h = hrow[t], d0 = dz3T[t], d1 = dz3T[PITCH + t];
                s0 = fmaf(h, d0, s0);
                s1 = fmaf(h, d1, s1);
                orow[t] = h > 0.f ? fmaf(d0, w0, d1 * w1) : 0.f;
            }
            accum(g + A_W3 + k * DA, s0, first);
            accum(g + A_W3 + k * DA + 1, s1, first);
        } else if (threadIdx.x < H2 + DA) {
            const int m = threadIdx.x - H2;
            float s = 0.f;
            for (int t = 0; t < TB; ++t) s += dz3T[m * PITCH + t];
            accum(g + A_B3 + m, s, first);
        }
        __syncthreads();
        dense_bwd_weight<H2>(h1T, H1, c2T, g + A_W2, g + A_B2, first);
        __syncthreads();
        dense_bwd_input(A.theta + A_W2, c2T, h1T, 1.0f);
        __syncthreads();
        dense_bwd_weight<H1>(sT, L.ds, h1T, g + A_W1, g + A_B1, first);
    }
    if (threadIdx.x < 32) {
        for (int o = 16; o > 0; o >>= 1) qsum += __shfl_xor_sync(0xffffffffu, qsum, o);
        if (threadIdx.x == 0) g[A_N] = qsum;
    }
    if (first) {
        for (int p = threadIdx.x; p < A_N; p += NT) g[p] = 0.f;
    }
}

// grad[p] = sum over CTA slices in a fixed order (bit-identical from run to run): four interleaved
// groups of slices are summed by four threads per parameter and combined 0+1+2+3 through shared memory;
// aux[0] = the same sum of the slices' extra slot
__global__ void reduce_kernel(const float *work, int parts, int n_params, float *grad, float *aux) {
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

// tf.keras.optimizers.Adam.apply_gradients (SkillshotLearner.py:68, 118, 417) and the
// DDPG soft target update (tau = 1 copies; target == NULL skips it).
__global__ void adam_kernel(float *params, const float *grads, float *m, float *v, float *target, int64_t n,
                            float lr_t, float beta1, float beta2, float eps, float tau, float grad_scale) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const float gr = grads[p] * grad_scale;
    const float mm = beta1 * m[p] + (1.0f - beta1) * gr;
    const float vv = beta2 * v[p] + (1.0f - beta2) * gr * gr;
    m[p] = mm;
    v[p] = vv;
    const float w = params[p] - lr_t * mm / (sqrtf(vv) + eps);
    params[p] = w;
    if (target) target[p] = tau * w + (1.0f - tau) * target[p];
}

// reduce_kernel and adam_kernel in one pass (single GPU: nothing sits between the two): the thread that holds a
// parameter's summed gradient applies Adam and the soft target update to it.
__global__ void reduce_adam_kernel(const float *work, int parts, int n_params, float *aux, float *grad_out, float *params,
                                   float *m, float *v, float *target, float lr_t, float beta1, float beta2, float eps, float tau,
                                   float grad_scale) {
    __shared__ float red[4][64];
    const int p = blockIdx.x * 64 + threadIdx.x, q = threadIdx.y;
    sslaunch::griddep_wait();            // ss_launch.cuh: placed beside the gradient kernel's last CTAs, held here until it is done
    sslaunch::griddep_launch();
    float s = 0.f;
    if (p <= n_params) {
#pragma unroll 10        // ten independent loads in flight per thread; the additions keep their order
        for (int c = q; c < parts; c += 4) s += __ldcg(work + (int64_t)c * (n_params + 1) + p);
    }
    red[q][threadIdx.x] = s;
    __syncthreads();
    if (q != 0 || p > n_params) return;
    const float t = ((red[0][threadIdx.x] + red[1][threadIdx.x]) + red[2][threadIdx.x]) + red[3][threadIdx.x];
    if (p == n_params) {
        if (aux) aux[0] = t;
        return;
    }
    if (grad_out) grad_out[p] = t;
    const float gr = t * grad_scale;
    const float mm = beta1 * m[p] + (1.0f - beta1) * gr;
    const float vv = beta2 * v[p] + (1.0f - beta2) * gr * gr;
    m[p] = mm;
    v[p] = vv;
    const float w = params[p] - lr_t * mm / (sqrtf(vv) + eps);
    params[p] = w;
    if (target) target[p] = tau * w + (1.0f - tau) * target[p];
}

// ---------------------------------------------------------------------------
// replay ring: SoA of (s[12], a[2], r, s'[12], done) rows
// ---------------------------------------------------------------------------
struct Ring {
    float *s, *a, *r, *s2;
    uint8_t *done;
    int64_t capacity;
};

// w4 = float4 per observation row: 3 (12 floats, the reference) or 3 * frames
__global__ void replay_push_kernel(Ring R, int64_t pos, const float *s, const float *a, const float *r,
                                   const float *s2, const uint8_t *done, int done_div, int64_t n, int w4) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= w4 * n) return;
    const int64_t row = e / w4, part = e - row * w4;
    const int64_t dst = (pos + row) % R.capacity;
    reinterpret_cast<float4 *>(R.s)[dst * w4 + part] = reinterpret_cast<const float4 *>(s)[e];
    if (s2) reinterpret_cast<float4 *>(R.s2)[dst * w4 + part] = reinterpret_cast<const float4 *>(s2)[e];
    if (part == 0) {
        reinterpret_cast<float2 *>(R.a)[dst] = reinterpret_cast<const float2 *>(a)[row];
        R.r[dst] = r[row];
        R.done[dst] = (done && done[row / done_div]) ? 1 : 0;      // any non-zero flag (e.g. winner_id 1 / 2) is stored as 1
    }
}

__device__ __forceinline__ void replay_sample_row(const Ring &R, int64_t size, const int64_t *indices, uint64_t seed,
                                                  uint64_t counter, float *s, float *a, float *r, float *s2, uint8_t *done,
                                                  int64_t *indices_out, int w4, int64_t e) {
    const int64_t b = e / w4, part = e - b * w4;
    int64_t src;
    if (indices) {
        src = indices[b];
    } else {                     // uniform with replacement over the filled part of the ring
        const U4 u = draw4(seed, kTagReplay, (uint32_t)(b / 4), (uint32_t)((b / 4) >> 32), counter);
        const uint32_t x = (b & 3) == 0 ? u.x : (b & 3) == 1 ? u.y : (b & 3) == 2 ? u.z : u.w;
        src = (int64_t)(((uint64_t)x * (uint64_t)size) >> 32);      // size < 2^32 rows
    }
    reinterpret_cast<float4 *>(s)[e] = reinterpret_cast<const float4 *>(R.s)[src * w4 + part];
    reinterpret_cast<float4 *>(s2)[e] = reinterpret_cast<const float4 *>(R.s2)[src * w4 + part];
    if (part == 0) {
        reinterpret_cast<float2 *>(a)[b] = reinterpret_cast<const float2 *>(R.a)[src];
        r[b] = R.r[src];
        done[b] = R.done[src];
        if (indices_out) indices_out[b] = src;
    }
}

// early (ss_launch.cuh, kPdlSampleEarly): gather first, wait afterwards -- the rows are then drawn while the previous
// update's last kernel still runs
__global__ void replay_sample_kernel(Ring R, int64_t size, const int64_t *indices, uint64_t seed, uint64_t counter,
                                     int64_t batch, float *s, float *a, float *r, float *s2, uint8_t *done,
                                     int64_t *indices_out, int w4, int early) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (!early) {                        // (the minibatch buffers may still be read by the previous update's kernels)
        sslaunch::griddep_wait();
        sslaunch::griddep_launch();
    }
    if (e < w4 * batch) replay_sample_row(R, size, indices, seed, counter, s, a, r, s2, done, indices_out, w4, e);
    if (early) {
        sslaunch::griddep_wait();
        sslaunch::griddep_launch();
    }
}

// n-step rows (DESIGN.md section 6.15): the eligible rows are up to SS_REPLAY_MAX_RUNS runs of ring positions; draw j of
// their total length picks the j-th eligible row in run order
struct NstepRuns {
    int64_t start[SS_REPLAY_MAX_RUNS], length[SS_REPLAY_MAX_RUNS];
    int n;
};

// replay_sample_kernel's thread per (row, float4) and draw.  The walk visits src + t * tick_rows (mod capacity) and stops
// after the first row with its done flag set or after n_step rows; every lane of a row walks the done bytes itself (the
// row's other lanes find them in L1) because each needs the walk's last row for its part of next_obs.  The reward sum
// rounds each product and each sum on its own (no FMA), so that a float32 restatement of the recurrence is exact.
__global__ void replay_sample_nstep_kernel(Ring R, NstepRuns runs, int64_t total, int64_t tick_rows, int n_step, float gamma,
                                           uint64_t seed, uint64_t counter, int64_t batch, float *s, float *a, float *r, float *s2,
                                           uint8_t *done, int64_t *indices_out, uint8_t *steps_out, int w4, int early) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (!early) {
        sslaunch::griddep_wait();
        sslaunch::griddep_launch();
    }
    if (e < w4 * batch) {
        const int64_t b = e / w4, part = e - b * w4;
        const U4 u = draw4(seed, kTagReplay, (uint32_t)(b / 4), (uint32_t)((b / 4) >> 32), counter);
        const uint32_t x = (b & 3) == 0 ? u.x : (b & 3) == 1 ? u.y : (b & 3) == 2 ? u.z : u.w;
        int64_t j = (int64_t)(((uint64_t)x * (uint64_t)total) >> 32);      // total < 2^32 rows
        int64_t src = runs.start[0] + j;
        for (int i = 0; i < runs.n; ++i) {
            if (j < runs.length[i]) {
                src = runs.start[i] + j;
                break;
            }
            j -= runs.length[i];
        }
        int64_t last = src;
        int k = 1;
        for (; k < n_step && !R.done[last]; ++k) {
            last += tick_rows;
            if (last >= R.capacity) last -= R.capacity;
        }
        reinterpret_cast<float4 *>(s)[e] = reinterpret_cast<const float4 *>(R.s)[src * w4 + part];
        reinterpret_cast<float4 *>(s2)[e] = reinterpret_cast<const float4 *>(R.s2)[last * w4 + part];
        if (part == 0) {
            float sum = R.r[src], g = 1.0f;
            int64_t row = src;
            for (int t = 1; t < k; ++t) {
                row += tick_rows;
                if (row >= R.capacity) row -= R.capacity;
                g = __fmul_rn(g, gamma);
                sum = __fadd_rn(sum, __fmul_rn(g, R.r[row]));
            }
            reinterpret_cast<float2 *>(a)[b] = reinterpret_cast<const float2 *>(R.a)[src];
            r[b] = sum;
            done[b] = R.done[last];
            if (indices_out) indices_out[b] = src;
            if (steps_out) steps_out[b] = (uint8_t)k;
        }
    }
    if (early) {
        sslaunch::griddep_wait();
        sslaunch::griddep_launch();
    }
}

// ---------------------------------------------------------------------------
// prioritized replay (DESIGN.md section 6.16): one float32 leaf p^alpha per ring position
// ---------------------------------------------------------------------------
constexpr int kPriThreads = 256, kPriItems = 8, kPriChunk = kPriThreads * kPriItems;   // eligible rows per scan block
constexpr int kPriRows = 64;                                                            // minibatch rows per draw block

// the float64 scratch of one prioritized draw over total_n eligible rows (capacity bounds total_n)
struct PriScratch {
    double *prefix;          // [total_n] inclusive prefix of the leaves WITHIN each kPriChunk block
    double *start;           // [blocks + 1] prefix before each block: start[0] = 0, start[k + 1] = start[k] + block k's sum
    float *bmin;             // [blocks] smallest non-zero leaf of each block (+inf: none)
    int64_t *blast;          // [blocks] last eligible row with a non-zero leaf of each block (-1: none)
    float *leaf_min;         // smallest non-zero eligible leaf
    int64_t *last_nz;        // last eligible row with a non-zero leaf (-1: none)
};

inline int64_t pri_blocks(int64_t capacity) { return (capacity + kPriChunk - 1) / kPriChunk; }
inline int64_t pri_scratch_bytes(int64_t capacity) {
    const int64_t nb = pri_blocks(capacity);
    return 8 * capacity + 8 * (nb + 1) + 8 * nb + 8 * nb + 16;
}
inline PriScratch pri_scratch(void *base, int64_t capacity) {
    const int64_t nb = pri_blocks(capacity);
    char *p = (char *)base;
    PriScratch S;
    S.prefix = (double *)p;
    S.start = (double *)(p + 8 * capacity);
    S.blast = (int64_t *)(p + 8 * capacity + 8 * (nb + 1));
    S.bmin = (float *)(p + 8 * capacity + 8 * (nb + 1) + 8 * nb);
    S.last_nz = (int64_t *)(p + 8 * capacity + 8 * (nb + 1) + 16 * nb);
    S.leaf_min = (float *)(p + 8 * capacity + 8 * (nb + 1) + 16 * nb + 8);
    return S;
}

// ring position of eligible row j (the mapping of replay_sample_nstep_kernel)
__device__ __forceinline__ int64_t run_position(const NstepRuns &runs, int64_t j) {
    int64_t src = runs.start[0] + j;
    for (int i = 0; i < runs.n; ++i) {
        if (j < runs.length[i]) {
            src = runs.start[i] + j;
            break;
        }
        j -= runs.length[i];
    }
    return src;
}

// block k: the inclusive prefix of eligible rows [k kPriChunk, (k + 1) kPriChunk) in a fixed order (each thread's eight rows
// in sequence, then the threads' sums by a fixed shuffle / shared-memory scan), its smallest non-zero leaf and its last
// row with a non-zero leaf
__global__ void __launch_bounds__(kPriThreads) priority_scan_kernel(const float *leaf, NstepRuns runs, int64_t total_n, PriScratch S) {
    __shared__ double wsum[kPriThreads / 32];
    __shared__ float wmin[kPriThreads / 32];
    __shared__ long long wlast[kPriThreads / 32];
    sslaunch::griddep_wait();
    sslaunch::griddep_launch();
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int64_t j0 = (int64_t)blockIdx.x * kPriChunk + (int64_t)t * kPriItems;
    double loc[kPriItems], acc = 0.0;
    float mn = INFINITY;
    long long last = -1;
#pragma unroll
    for (int i = 0; i < kPriItems; ++i) {
        const int64_t j = j0 + i;
        const float v = j < total_n ? leaf[run_position(runs, j)] : 0.f;
        acc += (double)v;
        loc[i] = acc;
        if (v > 0.f) {
            mn = fminf(mn, v);
            last = j;
        }
    }
    // inclusive scan of the thread sums: within the warp, then over the warps
    double inc = acc;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double y = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += y;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        last = max(last, __shfl_xor_sync(0xffffffffu, last, o));
    }
    if (lane == 31) wsum[warp] = inc;
    if (lane == 0) {
        wmin[warp] = mn;
        wlast[warp] = last;
    }
    __syncthreads();
    double before = 0.0;                                  // the earlier warps' sums, in order
    for (int w = 0; w < warp; ++w) before += wsum[w];
    const double below = __shfl_up_sync(0xffffffffu, inc, 1);
    const double base = lane == 0 ? before : before + below;
#pragma unroll
    for (int i = 0; i < kPriItems; ++i) {
        const int64_t j = j0 + i;
        if (j < total_n) S.prefix[j] = base + loc[i];
    }
    if (t == kPriThreads - 1) S.start[blockIdx.x + 1] = base + loc[kPriItems - 1];     // this block's sum (start fixed up below)
    if (t == 0) {
        float m = wmin[0];
        long long l = wlast[0];
        for (int w = 1; w < kPriThreads / 32; ++w) {
            m = fminf(m, wmin[w]);
            l = max(l, wlast[w]);
        }
        S.bmin[blockIdx.x] = m;
        S.blast[blockIdx.x] = l;
    }
}

// start[k + 1] = start[k] + sum_k in block order (the blocks' sums are in start[1 ..] on entry), by one thread from shared
// memory, 1,024 blocks at a time (the running sum is a chain of float64 additions; its operands are staged by every thread);
// the smallest non-zero leaf and the last row with one
constexpr int kPriBlocksThreads = 1024;
__global__ void __launch_bounds__(kPriBlocksThreads) priority_blocks_kernel(int64_t nb, PriScratch S) {
    __shared__ double sums[kPriBlocksThreads], starts[kPriBlocksThreads];
    __shared__ float wmin[kPriBlocksThreads / 32];
    __shared__ long long wlast[kPriBlocksThreads / 32];
    sslaunch::griddep_wait();
    sslaunch::griddep_launch();
    const int t = threadIdx.x;
    float mn = INFINITY;
    long long last = -1;
    for (int64_t k = t; k < nb; k += kPriBlocksThreads) {
        mn = fminf(mn, S.bmin[k]);
        last = max(last, (long long)S.blast[k]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        last = max(last, __shfl_xor_sync(0xffffffffu, last, o));
    }
    if ((t & 31) == 0) {
        wmin[t >> 5] = mn;
        wlast[t >> 5] = last;
    }
    double run = 0.0;
    for (int64_t c0 = 0; c0 < nb; c0 += kPriBlocksThreads) {
        const int n = (int)min((int64_t)kPriBlocksThreads, nb - c0);
        if (t < n) sums[t] = S.start[c0 + t + 1];
        __syncthreads();
        if (t == 0) {
#pragma unroll 16
            for (int i = 0; i < n; ++i) {
                run += sums[i];
                starts[i] = run;
            }
        }
        __syncthreads();
        if (t < n) S.start[c0 + t + 1] = starts[t];
        __syncthreads();
    }
    if (t == 0) {
        for (int w = 1; w < kPriBlocksThreads / 32; ++w) {
            mn = fminf(mn, wmin[w]);
            last = max(last, wlast[w]);
        }
        S.start[0] = 0.0;
        *S.leaf_min = mn;
        *S.last_nz = last;
    }
}

// One minibatch row per thread of the first kPriRows: the stratified draw u_b = (b + U_b) / B * total, the smallest eligible
// j with P[j] > u_b (binary search over the blocks' starts, then inside the block), the walk and reward sum of
// replay_sample_nstep_kernel (n_step = 1: the one-step row) and the importance weight; then every thread of the block copies
// the rows' observations, one float4 per (row, part)
__global__ void __launch_bounds__(256) replay_sample_prioritized_kernel(Ring R, NstepRuns runs, int64_t total_n, int64_t nb,
                                                                        PriScratch S, const float *leaf, int64_t tick_rows,
                                                                        int n_step, float gamma, uint64_t seed, uint64_t counter,
                                                                        int64_t batch, float beta, float *s, float *a, float *r,
                                                                        float *s2, uint8_t *done, int64_t *indices_out,
                                                                        uint8_t *steps_out, float *w_out, int w4) {
    __shared__ int64_t src_s[kPriRows], last_s[kPriRows];
    sslaunch::griddep_wait();
    sslaunch::griddep_launch();
    const int64_t b0 = (int64_t)blockIdx.x * kPriRows;
    if (threadIdx.x < kPriRows && b0 + threadIdx.x < batch) {
        const int64_t b = b0 + threadIdx.x;
        const U4 u4 = draw4(seed, kTagPriority, (uint32_t)(b / 4), (uint32_t)((b / 4) >> 32), counter);
        const uint32_t x = (b & 3) == 0 ? u4.x : (b & 3) == 1 ? u4.y : (b & 3) == 2 ? u4.z : u4.w;
        const double total = S.start[nb];
        const double u = ((double)b + (double)x * 0x1p-32) / (double)batch * total;
        int64_t j;
        if (!(u < total)) {
            j = *S.last_nz;                              // (u rounded up to total)
        } else {
            int64_t lo = 0, hi = nb - 1;                 // the first block whose end start[k + 1] exceeds u
            while (lo < hi) {
                const int64_t mid = (lo + hi) >> 1;
                if (S.start[mid + 1] > u) hi = mid;
                else lo = mid + 1;
            }
            const double st = S.start[lo];
            int64_t jl = lo * kPriChunk, jh = min(total_n, jl + kPriChunk) - 1;
            while (jl < jh) {
                const int64_t mid = (jl + jh) >> 1;
                if (st + S.prefix[mid] > u) jh = mid;
                else jl = mid + 1;
            }
            j = jl;
        }
        float w = 1.0f;
        if (j < 0) {
            j = 0;                                       // no non-zero leaf: row 0 of the runs, weight 1
        }
        const int64_t src = run_position(runs, j);
        const float p = leaf[src];
        if (p > 0.f) w = (float)pow((double)*S.leaf_min / (double)p, (double)beta);
        int64_t last = src;
        int k = 1;
        for (; k < n_step && !R.done[last]; ++k) {
            last += tick_rows;
            if (last >= R.capacity) last -= R.capacity;
        }
        float sum = R.r[src], g = 1.0f;
        int64_t row = src;
        for (int t = 1; t < k; ++t) {
            row += tick_rows;
            if (row >= R.capacity) row -= R.capacity;
            g = __fmul_rn(g, gamma);
            sum = __fadd_rn(sum, __fmul_rn(g, R.r[row]));
        }
        reinterpret_cast<float2 *>(a)[b] = reinterpret_cast<const float2 *>(R.a)[src];
        r[b] = sum;
        done[b] = R.done[last];
        w_out[b] = w;
        if (indices_out) indices_out[b] = src;
        if (steps_out) steps_out[b] = (uint8_t)k;
        src_s[threadIdx.x] = src;
        last_s[threadIdx.x] = last;
    }
    __syncthreads();
    const int64_t rows = min((int64_t)kPriRows, batch - b0);
    for (int64_t e = threadIdx.x; e < rows * w4; e += blockDim.x) {
        const int64_t bl = e / w4, part = e - bl * w4, o = (b0 + bl) * w4 + part;
        reinterpret_cast<float4 *>(s)[o] = reinterpret_cast<const float4 *>(R.s)[src_s[bl] * w4 + part];
        reinterpret_cast<float4 *>(s2)[o] = reinterpret_cast<const float4 *>(R.s2)[last_s[bl] * w4 + part];
    }
}

// priority update, in three launches: mark every drawn position, let the largest batch position claim it, and write the
// claimed leaves (and raise priority_max: non-negative floats order as their bit patterns)
__global__ void priority_mark_kernel(const int64_t *idx, int64_t batch, int64_t capacity, int *claim) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    sslaunch::griddep_wait();
    sslaunch::griddep_launch();
    if (b < batch && idx[b] >= 0 && idx[b] < capacity) claim[idx[b]] = -1;
}

__global__ void priority_claim_kernel(const int64_t *idx, int64_t batch, int64_t capacity, int *claim) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    sslaunch::griddep_wait();
    sslaunch::griddep_launch();
    if (b < batch && idx[b] >= 0 && idx[b] < capacity) atomicMax(claim + idx[b], (int)b);
}

__global__ void priority_write_kernel(const int64_t *idx, const float *td_abs, int64_t batch, int64_t capacity, const int *claim,
                                      float alpha, float eps, float *leaf, float *leaf_max) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    sslaunch::griddep_wait();
    sslaunch::griddep_launch();
    if (b < batch) {
        const int64_t i = idx[b];
        if (i >= 0 && i < capacity && claim[i] == (int)b) {
            const float p = powf(__fadd_rn(fabsf(td_abs[b]), eps), alpha);
            leaf[i] = p;
            atomicMax(reinterpret_cast<int *>(leaf_max), __float_as_int(p));
        }
    }
}

__global__ void priority_fill_kernel(float *leaf, const float *leaf_max, int64_t capacity, int64_t pos, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    sslaunch::griddep_wait();
    sslaunch::griddep_launch();
    if (i < n) {
        int64_t dst = pos + i;
        if (dst >= capacity) dst -= capacity;
        leaf[dst] = *leaf_max;
    }
}

// ---------------------------------------------------------------------------
// launch helpers
// ---------------------------------------------------------------------------
constexpr size_t kSmemActorFwd = (size_t)(DS + H1 + H2 + DA) * PITCH * 4;
constexpr size_t kSmemActorFwdNoisy = kSmemActorFwd + (size_t)((A_N + 3) / 4 * 4) * 4;
inline size_t smem_critic_fwd(int ds) { return (size_t)(ds + H1 + DA + H2) * PITCH * 4 + TB * 4; }
inline size_t smem_critic_fwd_actor(int ds) { return smem_critic_fwd(ds) + (size_t)(H1 + H2) * PITCH * 4; }
inline size_t smem_critic_grad(int ds) { return (size_t)(ds + H1 + DA + H2) * PITCH * 4 + 2 * TB * 4; }
inline size_t smem_actor_grad(int ds) { return (size_t)(ds + H1 + H2 + DA + H1 + DA + H2 + DA) * PITCH * 4 + TB * 4; }

inline int check_launch() { return cudaGetLastError() == cudaSuccess ? SS_OK : SS_ERR_CUDA; }

template <class K>
int max_ctas(K kernel, size_t smem) {
    int dev = 0, sms = 0, per_sm = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return -1;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return -1;
    if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return -1;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, NT, smem) != cudaSuccess) return -1;
    return sms * (per_sm > 0 ? per_sm : 1);
}

// persistent grid: one CTA per tile up to the number of resident CTAs
template <class K>
int grid_for(K kernel, size_t smem, int64_t tiles, int cap) {
    int m = max_ctas(kernel, smem);
    if (m <= 0) return -1;
    if (cap > 0 && m > cap) m = cap;
    return (int)(tiles < m ? (tiles > 0 ? tiles : 1) : m);
}

}  // namespace

extern "C" {

int64_t ss_learner_workspace_bytes(void) {
    return (int64_t)SS_LEARNER_MAX_PARTS * (SS_CRITIC_PARAMS + 1) * sizeof(float);
}

int ss_actor_forward(const float *actor_params, const float *obs, float *act_out, int64_t n,
                     float param_noise_sd, int64_t noise_group, float action_noise_sd,
                     uint64_t seed, uint64_t counter, void *stream) {
    if (!actor_params || !obs || !act_out || n <= 0 || param_noise_sd < 0.f || action_noise_sd < 0.f)
        return SS_ERR_INVALID_ARG;
    if (((uintptr_t)actor_params & 15) || ((uintptr_t)act_out & 7)) return SS_ERR_INVALID_ARG;
    const bool noisy = param_noise_sd > 0.f;
    if (noisy && noise_group <= 0) return SS_ERR_INVALID_ARG;
    ActorFwdArgs A{actor_params, obs, act_out, n, noisy ? noise_group : n, param_noise_sd, action_noise_sd, seed, counter};
    cudaStream_t st = (cudaStream_t)stream;
    if (noisy) {
        const int64_t upg = (noise_group + TB - 1) / TB, groups = (n + noise_group - 1) / noise_group;
        const int grid = grid_for(actor_fwd_kernel<true>, kSmemActorFwdNoisy, groups * upg, 0);
        if (grid < 0) return SS_ERR_CUDA;
        actor_fwd_kernel<true><<<grid, NT, kSmemActorFwdNoisy, st>>>(A);
    } else {
        const int grid = grid_for(actor_fwd_kernel<false>, kSmemActorFwd, (n + TB - 1) / TB, 0);
        if (grid < 0) return SS_ERR_CUDA;
        actor_fwd_kernel<false><<<grid, NT, kSmemActorFwd, st>>>(A);
    }
    return check_launch();
}

int ss_param_noise(const float *params, float *out, int64_t n_params, float sd, uint64_t seed,
                   uint64_t group, uint64_t counter, void *stream) {
    if (!params || !out || n_params <= 0) return SS_ERR_INVALID_ARG;
    const int64_t quads = (n_params + 3) / 4;
    param_noise_kernel<<<(unsigned)((quads + 127) / 128), 128, 0, (cudaStream_t)stream>>>(params, out, n_params, sd,
                                                                                          seed, group, counter);
    return check_launch();
}

// ---- critic forward / TD target / gradients with a first layer of 12 * frames inputs (frames = 1: the reference) ----
int64_t ss_critic_frames_params(int frames) { return frames < 1 || frames > SS_MAX_FRAMES ? -1 : (int64_t)lay_of(DS * frames).c_n; }

int64_t ss_learner_frames_workspace_bytes(int frames) {
    if (frames < 1 || frames > SS_MAX_FRAMES) return -1;
    const Lay L = lay_of(DS * frames);
    return (int64_t)SS_LEARNER_MAX_PARTS * ((L.c_n > L.a_n ? L.c_n : L.a_n) + 1) * sizeof(float);
}

int ss_critic_forward_frames(const float *critic_params, int frames, const float *obs, const float *act, float *q_out,
                             int64_t n, void *stream) {
    if (!critic_params || !obs || !act || !q_out || n <= 0 || frames < 1 || frames > SS_MAX_FRAMES) return SS_ERR_INVALID_ARG;
    const int ds = DS * frames;
    CriticFwdArgs A{nullptr, critic_params, obs, act, nullptr, nullptr, 0.f, q_out, n, ds};
    const int grid = grid_for(critic_fwd_kernel<false>, smem_critic_fwd(ds), (n + TB - 1) / TB, 0);
    if (grid < 0) return SS_ERR_CUDA;
    critic_fwd_kernel<false><<<grid, NT, smem_critic_fwd(ds), (cudaStream_t)stream>>>(A);
    return check_launch();
}

int ss_ddpg_targets_frames(const float *target_actor_params, const float *target_critic_params, int frames,
                           const float *reward, const float *next_obs, const uint8_t *done, float gamma, float *y_out,
                           int64_t n, void *stream) {
    if (!target_actor_params || !target_critic_params || !reward || !next_obs || !y_out || n <= 0 || frames < 1 ||
        frames > SS_MAX_FRAMES)
        return SS_ERR_INVALID_ARG;
    const int ds = DS * frames;
    CriticFwdArgs A{target_actor_params, target_critic_params, next_obs, nullptr, reward, done, gamma, y_out, n, ds};
    const int grid = grid_for(critic_fwd_kernel<true>, smem_critic_fwd_actor(ds), (n + TB - 1) / TB, 0);
    if (grid < 0) return SS_ERR_CUDA;
    critic_fwd_kernel<true><<<grid, NT, smem_critic_fwd_actor(ds), (cudaStream_t)stream>>>(A);
    return check_launch();
}

int ss_td3_targets_frames(const float *target_actor_params, const float *target_critic_params, const float *target_critic2_params,
                          int frames, const float *reward, const float *next_obs, const uint8_t *done, float gamma,
                          float noise_sd, float noise_clip, uint64_t seed, uint64_t counter, int64_t row_offset, float *y_out,
                          int64_t n, void *workspace, int64_t workspace_bytes, void *stream) {
    (void)workspace; (void)workspace_bytes;       // (the float32 kernel keeps everything in shared memory)
    if (!target_actor_params || !target_critic_params || !reward || !next_obs || !y_out || n <= 0 || frames < 1 ||
        frames > SS_MAX_FRAMES || !(noise_sd >= 0.f) || !(noise_clip >= 0.f) || row_offset < 0)
        return SS_ERR_INVALID_ARG;
    const int ds = DS * frames;
    const size_t smem = smem_critic_fwd_actor(ds) + TB * 4;
    Td3TargetArgs A{target_actor_params, target_critic_params, target_critic2_params, reward, next_obs, done, gamma, noise_sd,
                    noise_clip, seed, counter, row_offset, y_out, n, ds};
    const int grid = grid_for(td3_target_kernel, smem, (n + TB - 1) / TB, 0);
    if (grid < 0) return SS_ERR_CUDA;
    td3_target_kernel<<<grid, NT, smem, (cudaStream_t)stream>>>(A);
    return check_launch();
}

static int critic_grad_f32(const float *critic_params, int frames, const float *obs, const float *act, const float *target,
                           const float *row_weight, float *td_abs_out, bool weighted, const uint8_t *dropout_keep,
                           float dropout_rate, uint64_t seed, uint64_t counter, int64_t n, int64_t n_global, int64_t row_offset,
                           float *grad_out, float *sse_out, void *workspace, int64_t workspace_bytes, void *stream) {
    if (!critic_params || !obs || !act || !target || !workspace || n <= 0 || frames < 1 || frames > SS_MAX_FRAMES)
        return SS_ERR_INVALID_ARG;
    if (dropout_rate < 0.f || dropout_rate >= 1.f) return SS_ERR_INVALID_ARG;
    if ((uintptr_t)critic_params & 15) return SS_ERR_INVALID_ARG;
    const Lay L = lay_of(DS * frames);
    const int cap = (int)(workspace_bytes / ((int64_t)(L.c_n + 1) * 4));
    if (cap < 1) return SS_ERR_INVALID_ARG;
    auto kernel = weighted ? critic_grad_weighted_kernel : critic_grad_kernel;
    const int grid = grid_for(kernel, smem_critic_grad(L.ds), (n + TB - 1) / TB, cap < SS_LEARNER_MAX_PARTS ? cap : SS_LEARNER_MAX_PARTS);
    if (grid < 0) return SS_ERR_CUDA;
    CriticGradArgs A{critic_params, obs, act, target, dropout_keep, dropout_rate, seed, counter,
                     n, n_global > 0 ? n_global : n, row_offset, (float *)workspace, L.ds, row_weight, td_abs_out};
    cudaStream_t st = (cudaStream_t)stream;
    kernel<<<grid, NT, smem_critic_grad(L.ds), st>>>(A);
    if (!grad_out) return check_launch() == SS_OK ? grid : SS_ERR_CUDA;      // slices only (ss_peer_reduce_push follows)
    reduce_kernel<<<(L.c_n + 1 + 63) / 64, dim3(64, 4), 0, st>>>((const float *)workspace, grid, L.c_n, grad_out, sse_out);
    return check_launch();
}

int ss_critic_grad_frames(const float *critic_params, int frames, const float *obs, const float *act, const float *target,
                          const uint8_t *dropout_keep, float dropout_rate, uint64_t seed, uint64_t counter,
                          int64_t n, int64_t n_global, int64_t row_offset, float *grad_out, float *sse_out,
                          void *workspace, int64_t workspace_bytes, void *stream) {
    return critic_grad_f32(critic_params, frames, obs, act, target, nullptr, nullptr, false, dropout_keep, dropout_rate, seed, counter,
                           n, n_global, row_offset, grad_out, sse_out, workspace, workspace_bytes, stream);
}

int ss_critic_grad_weighted(const float *critic_params, int frames, int tensor_cores, const float *obs, const float *act,
                            const float *target, const float *row_weight, float *td_abs_out, const uint8_t *dropout_keep,
                            float dropout_rate, uint64_t seed, uint64_t counter, int64_t n, int64_t n_global, int64_t row_offset,
                            float *grad_out, float *sse_out, void *workspace, int64_t workspace_bytes, void *stream) {
    if (!critic_params || !obs || !act || !target || !workspace || n <= 0 || frames < 1 || frames > SS_MAX_FRAMES)
        return SS_ERR_INVALID_ARG;
    if (!(dropout_rate >= 0.f && dropout_rate < 1.f) || n_global < 0 || row_offset < 0) return SS_ERR_INVALID_ARG;
    if (((uintptr_t)row_weight | (uintptr_t)td_abs_out) & 3) return SS_ERR_INVALID_ARG;
    if (!tensor_cores)
        return critic_grad_f32(critic_params, frames, obs, act, target, row_weight, td_abs_out, true, dropout_keep, dropout_rate, seed,
                               counter, n, n_global, row_offset, grad_out, sse_out, workspace, workspace_bytes, stream);
    // the checks of ss_critic_grad_tc / ss_critic_grad_frames_tc
    if (((uintptr_t)critic_params | (uintptr_t)obs) & 15 || ((uintptr_t)act & 7)) return SS_ERR_INVALID_ARG;
    if (frames == 1) {
        if ((uintptr_t)dropout_keep & 15) return SS_ERR_INVALID_ARG;
        if (workspace_bytes / ((int64_t)(SS_CRITIC_PARAMS + 1) * 4) < 1) return SS_ERR_INVALID_ARG;
        return sstc::critic_grad_tc_weighted(critic_params, obs, act, target, row_weight, td_abs_out, dropout_keep, dropout_rate, seed,
                                             counter, n, n_global, row_offset, grad_out, sse_out, workspace, workspace_bytes,
                                             (cudaStream_t)stream);
    }
    if (((uintptr_t)dropout_keep & 7) || ((uintptr_t)workspace & 15) || workspace_bytes < ss_learner_frames_tc_workspace_bytes(frames, n))
        return SS_ERR_INVALID_ARG;
    return sstc::critic_grad_frames_tc_weighted(critic_params, frames, obs, act, target, row_weight, td_abs_out, dropout_keep,
                                                dropout_rate, seed, counter, n, n_global, row_offset, grad_out, sse_out, workspace,
                                                workspace_bytes, (cudaStream_t)stream);
}

int ss_actor_grad_frames(const float *actor_params, const float *critic_params, int frames, const float *obs, int64_t n,
                         float *grad_out, float *q_sum_out, void *workspace, int64_t workspace_bytes, void *stream) {
    if (!actor_params || !critic_params || !obs || !workspace || n <= 0 || frames < 1 || frames > SS_MAX_FRAMES)
        return SS_ERR_INVALID_ARG;
    if (((uintptr_t)actor_params | (uintptr_t)critic_params) & 15) return SS_ERR_INVALID_ARG;
    const Lay L = lay_of(DS * frames);
    const int cap = (int)(workspace_bytes / ((int64_t)(L.a_n + 1) * 4));
    if (cap < 1) return SS_ERR_INVALID_ARG;
    const int grid = grid_for(actor_grad_kernel, smem_actor_grad(L.ds), (n + TB - 1) / TB,
                              cap < SS_LEARNER_MAX_PARTS ? cap : SS_LEARNER_MAX_PARTS);
    if (grid < 0) return SS_ERR_CUDA;
    ActorGradArgs A{actor_params, critic_params, obs, n, (float *)workspace, L.ds};
    cudaStream_t st = (cudaStream_t)stream;
    actor_grad_kernel<<<grid, NT, smem_actor_grad(L.ds), st>>>(A);
    if (!grad_out) return check_launch() == SS_OK ? grid : SS_ERR_CUDA;
    reduce_kernel<<<(L.a_n + 1 + 63) / 64, dim3(64, 4), 0, st>>>((const float *)workspace, grid, L.a_n, grad_out, q_sum_out);
    return check_launch();
}

// the reference's own width: 12 inputs
int ss_critic_forward(const float *critic_params, const float *obs, const float *act, float *q_out, int64_t n,
                      void *stream) {
    return ss_critic_forward_frames(critic_params, 1, obs, act, q_out, n, stream);
}

int ss_ddpg_targets(const float *target_actor_params, const float *target_critic_params, const float *reward,
                    const float *next_obs, const uint8_t *done, float gamma, float *y_out, int64_t n, void *stream) {
    return ss_ddpg_targets_frames(target_actor_params, target_critic_params, 1, reward, next_obs, done, gamma, y_out, n, stream);
}

int ss_critic_grad(const float *critic_params, const float *obs, const float *act, const float *target,
                   const uint8_t *dropout_keep, float dropout_rate, uint64_t seed, uint64_t counter,
                   int64_t n, int64_t n_global, int64_t row_offset, float *grad_out, float *sse_out,
                   void *workspace, int64_t workspace_bytes, void *stream) {
    return ss_critic_grad_frames(critic_params, 1, obs, act, target, dropout_keep, dropout_rate, seed, counter, n, n_global,
                                 row_offset, grad_out, sse_out, workspace, workspace_bytes, stream);
}

int ss_actor_grad(const float *actor_params, const float *critic_params, const float *obs, int64_t n,
                  float *grad_out, float *q_sum_out, void *workspace, int64_t workspace_bytes, void *stream) {
    return ss_actor_grad_frames(actor_params, critic_params, 1, obs, n, grad_out, q_sum_out, workspace, workspace_bytes, stream);
}

int ss_adam_tf(float *params, const float *grads, float *m, float *v, float *target_params, int64_t n,
               int64_t step, float lr, float beta1, float beta2, float eps, float tau, float grad_scale,
               void *stream) {
    if (!params || !grads || !m || !v || n <= 0 || step < 1) return SS_ERR_INVALID_ARG;
    // lr_t = lr * sqrt(1 - beta2^t) / (1 - beta1^t), evaluated in double on the host like Keras does in Python
    const double lr_t = (double)lr * sqrt(1.0 - pow((double)beta2, (double)step)) / (1.0 - pow((double)beta1, (double)step));
    adam_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(params, grads, m, v, target_params, n,
                                                                               (float)lr_t, beta1, beta2, eps, tau,
                                                                               grad_scale);
    return check_launch();
}

int ss_reduce_adam_tf(const void *workspace, int parts, int n_params, float *aux_out, float *grad_out, float *params, float *m,
                      float *v, float *target_params, int64_t step, float lr, float beta1, float beta2, float eps, float tau,
                      float grad_scale, void *stream) {
    if (!workspace || parts < 1 || n_params < 1 || !params || !m || !v || step < 1) return SS_ERR_INVALID_ARG;
    const double lr_t = (double)lr * sqrt(1.0 - pow((double)beta2, (double)step)) / (1.0 - pow((double)beta1, (double)step));
    if (sslaunch::launch(reduce_adam_kernel, dim3((n_params + 1 + 63) / 64), dim3(64, 4), 0, (cudaStream_t)stream,
                         (const float *)workspace, parts, n_params, aux_out, grad_out, params, m, v, target_params, (float)lr_t,
                         beta1, beta2, eps, tau, grad_scale) != cudaSuccess)
        return SS_ERR_CUDA;
    return check_launch();
}

int ss_replay_push_frames(float *ring_obs, float *ring_act, float *ring_reward, float *ring_next_obs, uint8_t *ring_done,
                          int64_t capacity, int64_t write_pos, int frames, const float *obs, const float *act,
                          const float *reward, const float *next_obs, const uint8_t *done, int done_div, int64_t n,
                          void *stream) {
    if (!ring_obs || !ring_act || !ring_reward || !ring_next_obs || !ring_done || !obs || !act || !reward || !next_obs)
        return SS_ERR_INVALID_ARG;
    if (capacity <= 0 || n <= 0 || n > capacity || write_pos < 0 || write_pos >= capacity || done_div < 1 || frames < 1 ||
        frames > SS_MAX_FRAMES)
        return SS_ERR_INVALID_ARG;
    if (((uintptr_t)ring_obs | (uintptr_t)ring_next_obs | (uintptr_t)obs | (uintptr_t)next_obs) & 15)
        return SS_ERR_INVALID_ARG;
    Ring R{ring_obs, ring_act, ring_reward, ring_next_obs, ring_done, capacity};
    const int w4 = 3 * frames;
    replay_push_kernel<<<(unsigned)((w4 * n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(R, write_pos, obs, act, reward,
                                                                                          next_obs, done, done_div, n, w4);
    return check_launch();
}

int ss_replay_sample_frames(const float *ring_obs, const float *ring_act, const float *ring_reward,
                            const float *ring_next_obs, const uint8_t *ring_done, int64_t capacity, int64_t size, int frames,
                            const int64_t *indices, uint64_t seed, uint64_t counter, int64_t batch,
                            float *obs, float *act, float *reward, float *next_obs, uint8_t *done, int64_t *indices_out,
                            void *stream) {
    if (!ring_obs || !ring_act || !ring_reward || !ring_next_obs || !ring_done || !obs || !act || !reward ||
        !next_obs || !done)
        return SS_ERR_INVALID_ARG;
    if (capacity <= 0 || size <= 0 || size > capacity || batch <= 0 || frames < 1 || frames > SS_MAX_FRAMES)
        return SS_ERR_INVALID_ARG;
    Ring R{(float *)ring_obs, (float *)ring_act, (float *)ring_reward, (float *)ring_next_obs, (uint8_t *)ring_done,
           capacity};
    const int w4 = 3 * frames;
    const int early = (sslaunch::pdl_mode() & sslaunch::kPdlOn) && (sslaunch::pdl_mode() & sslaunch::kPdlSampleEarly) ? 1 : 0;
    if (sslaunch::launch(replay_sample_kernel, dim3((unsigned)((w4 * batch + 255) / 256)), dim3(256), 0, (cudaStream_t)stream, R,
                         size, indices, seed, counter, batch, obs, act, reward, next_obs, done, indices_out, w4, early) != cudaSuccess)
        return SS_ERR_CUDA;
    return check_launch();
}

int ss_replay_sample_nstep(const float *ring_obs, const float *ring_act, const float *ring_reward, const float *ring_next_obs,
                           const uint8_t *ring_done, int64_t capacity, int frames, int64_t tick_rows, int n_step, float gamma,
                           const int64_t *runs_host, int n_runs, uint64_t seed, uint64_t counter, int64_t batch, float *obs,
                           float *act, float *reward, float *next_obs, uint8_t *done, int64_t *indices_out, uint8_t *steps_out,
                           void *stream) {
    if (!ring_obs || !ring_act || !ring_reward || !ring_next_obs || !ring_done || !obs || !act || !reward || !next_obs ||
        !done || !runs_host)
        return SS_ERR_INVALID_ARG;
    if (capacity <= 0 || batch <= 0 || frames < 1 || frames > SS_MAX_FRAMES || tick_rows < 1 || n_step < 1 ||
        n_step > SS_REPLAY_MAX_NSTEP || tick_rows > capacity / n_step || n_runs < 1 || n_runs > SS_REPLAY_MAX_RUNS ||
        !std::isfinite(gamma))
        return SS_ERR_INVALID_ARG;
    if (((uintptr_t)ring_obs | (uintptr_t)ring_next_obs | (uintptr_t)obs | (uintptr_t)next_obs) & 15) return SS_ERR_INVALID_ARG;
    NstepRuns runs{};
    int64_t total = 0;
    for (int i = 0; i < n_runs; ++i) {
        const int64_t st = runs_host[2 * i], len = runs_host[2 * i + 1];
        if (st < 0 || len < 1 || st >= capacity || len > capacity - st) return SS_ERR_INVALID_ARG;
        runs.start[i] = st;
        runs.length[i] = len;
        total += len;
    }
    runs.n = n_runs;
    if (total >= ((int64_t)1 << 32)) return SS_ERR_INVALID_ARG;
    Ring R{(float *)ring_obs, (float *)ring_act, (float *)ring_reward, (float *)ring_next_obs, (uint8_t *)ring_done, capacity};
    const int w4 = 3 * frames;
    const int early = (sslaunch::pdl_mode() & sslaunch::kPdlOn) && (sslaunch::pdl_mode() & sslaunch::kPdlSampleEarly) ? 1 : 0;
    if (sslaunch::launch(replay_sample_nstep_kernel, dim3((unsigned)((w4 * batch + 255) / 256)), dim3(256), 0, (cudaStream_t)stream,
                         R, runs, total, tick_rows, n_step, gamma, seed, counter, batch, obs, act, reward, next_obs, done,
                         indices_out, steps_out, w4, early) != cudaSuccess)
        return SS_ERR_CUDA;
    return check_launch();
}

int64_t ss_replay_priority_scratch_bytes(int64_t capacity) { return capacity < 1 ? -1 : pri_scratch_bytes(capacity); }

int ss_replay_sample_prioritized(const float *ring_obs, const float *ring_act, const float *ring_reward, const float *ring_next_obs,
                                 const uint8_t *ring_done, int64_t capacity, int frames, int64_t tick_rows, int n_step, float gamma,
                                 const int64_t *runs_host, int n_runs, uint64_t seed, uint64_t counter, int64_t batch, float *obs,
                                 float *act, float *reward, float *next_obs, uint8_t *done, int64_t *indices_out, uint8_t *steps_out,
                                 const float *priority, void *scratch, int64_t scratch_bytes, float beta, float *weights_out,
                                 void *stream) {
    if (!ring_obs || !ring_act || !ring_reward || !ring_next_obs || !ring_done || !obs || !act || !reward || !next_obs ||
        !done || !runs_host || !priority || !scratch || !weights_out)
        return SS_ERR_INVALID_ARG;
    if (capacity <= 0 || batch <= 0 || frames < 1 || frames > SS_MAX_FRAMES || tick_rows < 1 || n_step < 1 ||
        n_step > SS_REPLAY_MAX_NSTEP || tick_rows > capacity / n_step || n_runs < 1 || n_runs > SS_REPLAY_MAX_RUNS ||
        !std::isfinite(gamma) || !std::isfinite(beta) || beta < 0.f || beta > 1.f)
        return SS_ERR_INVALID_ARG;
    if (((uintptr_t)ring_obs | (uintptr_t)ring_next_obs | (uintptr_t)obs | (uintptr_t)next_obs) & 15) return SS_ERR_INVALID_ARG;
    if (((uintptr_t)scratch & 7) || ((uintptr_t)priority & 3) || ((uintptr_t)weights_out & 3) || ((uintptr_t)indices_out & 7) ||
        ((uintptr_t)act & 7))
        return SS_ERR_INVALID_ARG;
    if (scratch_bytes < pri_scratch_bytes(capacity)) return SS_ERR_INVALID_ARG;
    NstepRuns runs{};
    int64_t total = 0;
    for (int i = 0; i < n_runs; ++i) {
        const int64_t st = runs_host[2 * i], len = runs_host[2 * i + 1];
        if (st < 0 || len < 1 || st >= capacity || len > capacity - st) return SS_ERR_INVALID_ARG;
        runs.start[i] = st;
        runs.length[i] = len;
        total += len;
    }
    runs.n = n_runs;
    if (total > capacity) return SS_ERR_INVALID_ARG;          // (runs that overlap)
    Ring R{(float *)ring_obs, (float *)ring_act, (float *)ring_reward, (float *)ring_next_obs, (uint8_t *)ring_done, capacity};
    const PriScratch S = pri_scratch(scratch, capacity);
    const int64_t nb = (total + kPriChunk - 1) / kPriChunk;
    cudaStream_t st = (cudaStream_t)stream;
    if (sslaunch::launch(priority_scan_kernel, dim3((unsigned)nb), dim3(kPriThreads), 0, st, priority, runs, total, S) != cudaSuccess)
        return SS_ERR_CUDA;
    if (sslaunch::launch(priority_blocks_kernel, dim3(1), dim3(kPriBlocksThreads), 0, st, nb, S) != cudaSuccess)
        return SS_ERR_CUDA;
    if (sslaunch::launch(replay_sample_prioritized_kernel, dim3((unsigned)((batch + kPriRows - 1) / kPriRows)), dim3(256), 0, st, R,
                         runs, total, nb, S, priority, tick_rows, n_step, gamma, seed, counter, batch, beta, obs, act, reward,
                         next_obs, done, indices_out, steps_out, weights_out, 3 * frames) != cudaSuccess)
        return SS_ERR_CUDA;
    return check_launch();
}

int ss_replay_priority_update(float *priority, float *priority_max, int64_t capacity, const int64_t *indices, const float *td_abs,
                              int64_t batch, float alpha, float eps, int32_t *scratch, void *stream) {
    if (!priority || !priority_max || !indices || !td_abs || !scratch || capacity < 1 || batch < 1 || batch > INT32_MAX)
        return SS_ERR_INVALID_ARG;
    if (!std::isfinite(alpha) || alpha < 0.f || !std::isfinite(eps) || !(eps > 0.f)) return SS_ERR_INVALID_ARG;
    if (((uintptr_t)priority | (uintptr_t)priority_max | (uintptr_t)td_abs | (uintptr_t)scratch) & 3 || ((uintptr_t)indices & 7))
        return SS_ERR_INVALID_ARG;
    const dim3 grid((unsigned)((batch + 255) / 256));
    cudaStream_t st = (cudaStream_t)stream;
    if (sslaunch::launch(priority_mark_kernel, grid, dim3(256), 0, st, indices, batch, capacity, (int *)scratch) != cudaSuccess ||
        sslaunch::launch(priority_claim_kernel, grid, dim3(256), 0, st, indices, batch, capacity, (int *)scratch) != cudaSuccess ||
        sslaunch::launch(priority_write_kernel, grid, dim3(256), 0, st, indices, td_abs, batch, capacity, (const int *)scratch, alpha,
                         eps, priority, priority_max) != cudaSuccess)
        return SS_ERR_CUDA;
    return check_launch();
}

int ss_replay_priority_fill(float *priority, const float *priority_max, int64_t capacity, int64_t pos, int64_t n, void *stream) {
    if (!priority || !priority_max || capacity < 1 || pos < 0 || pos >= capacity || n < 1 || n > capacity) return SS_ERR_INVALID_ARG;
    if (((uintptr_t)priority | (uintptr_t)priority_max) & 3) return SS_ERR_INVALID_ARG;
    if (sslaunch::launch(priority_fill_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, (cudaStream_t)stream, priority,
                         priority_max, capacity, pos, n) != cudaSuccess)
        return SS_ERR_CUDA;
    return check_launch();
}

int ss_replay_push(float *ring_obs, float *ring_act, float *ring_reward, float *ring_next_obs, uint8_t *ring_done,
                   int64_t capacity, int64_t write_pos, const float *obs, const float *act, const float *reward,
                   const float *next_obs, const uint8_t *done, int done_div, int64_t n, void *stream) {
    return ss_replay_push_frames(ring_obs, ring_act, ring_reward, ring_next_obs, ring_done, capacity, write_pos, 1, obs, act,
                                 reward, next_obs, done, done_div, n, stream);
}

int ss_replay_sample(const float *ring_obs, const float *ring_act, const float *ring_reward,
                     const float *ring_next_obs, const uint8_t *ring_done, int64_t capacity, int64_t size,
                     const int64_t *indices, uint64_t seed, uint64_t counter, int64_t batch,
                     float *obs, float *act, float *reward, float *next_obs, uint8_t *done, int64_t *indices_out,
                     void *stream) {
    return ss_replay_sample_frames(ring_obs, ring_act, ring_reward, ring_next_obs, ring_done, capacity, size, 1, indices, seed,
                                   counter, batch, obs, act, reward, next_obs, done, indices_out, stream);
}

// The in-place ring form with the env step running BESIDE the forward kernel (see ss_env_step_tiles).  The forward kernels go
// to `st_hi`, a stream of HIGHER priority than the caller's: both kernels of a tick become eligible at the same moment (when
// the previous tick's env step ends), and the forward kernel's CTAs, which need a whole SM's shared memory and three quarters
// of its registers, must be placed first -- the one-warp env CTAs then fill what is left beside them; placed the other way
// round they occupy every SM and the forward kernel starves while they wait for it (measured: every tile timed out).
// env step(t) runs on the caller's stream; forward(t + 1) waits for it by an event, and reads its second observation copy.
static int rollout_overlapped(void *env_state, int64_t n_envs, const float *actor_params, float *obs_a, float *actions, float *reward,
                              uint8_t *done, uint8_t *winner, float *ring_obs, float *ring_act, float *ring_reward,
                              float *ring_next_obs, uint8_t *ring_done, int64_t capacity, int64_t write_pos, int n_ticks,
                              float param_noise_sd, int64_t noise_group, float action_noise_sd, int reward_mode, int64_t tick_limit,
                              int reset_mode, uint64_t env_seed, uint64_t env_counter, uint64_t noise_seed, uint64_t noise_counter,
                              uint32_t *status, int step_flags, int *tile_ready, cudaStream_t st, cudaStream_t st_hi) {
    const int64_t rows = 2 * n_envs, segs = capacity / rows;
    int64_t seg = write_pos / rows;
    cudaEvent_t ev;                                            // one event, re-recorded: each wait is enqueued before the next record
    if (cudaEventCreateWithFlags(&ev, cudaEventDisableTiming) != cudaSuccess) return SS_ERR_CUDA;
    int rc = SS_OK;
    auto fail = [&](int code) { cudaEventDestroy(ev); return code; };
    if (cudaMemcpyAsync(ring_obs + seg * rows * 12, obs_a, (size_t)rows * 48, cudaMemcpyDeviceToDevice, st) != cudaSuccess)
        return fail(SS_ERR_CUDA);
    for (int t = 0; t < n_ticks; ++t, seg = (seg + 1) % segs) {
        float *o = ring_obs + seg * rows * 12, *a = ring_act + seg * rows * 2;
        float *o_next = (t + 1 < n_ticks) ? ring_obs + ((seg + 1) % segs) * rows * 12 : obs_a;
        // the forward reads what the caller's stream has produced so far: the previous tick's env step (or, first, the copy above)
        if (cudaEventRecord(ev, st) != cudaSuccess || cudaStreamWaitEvent(st_hi, ev, 0) != cudaSuccess) return fail(SS_ERR_CUDA);
        int grid_fwd = 0;
        int64_t units = 0;
        rc = ss_actor_forward_tc_signal(actor_params, o, a, rows, param_noise_sd, noise_group, action_noise_sd, noise_seed,
                                        noise_counter + (uint64_t)t, tile_ready, &grid_fwd, &units, st_hi);
        if (rc != SS_OK) return fail(rc);
        rc = ss_env_step_tiles(env_state, n_envs, a, ring_next_obs + seg * rows * 12, o_next, ring_reward + seg * rows, done,
                               ring_done + seg * rows, winner, reward_mode, tick_limit, reset_mode, env_seed,
                               env_counter + (uint64_t)t, status, step_flags, tile_ready, units, grid_fwd, st);
        if (rc != SS_OK) return fail(rc);
    }
    // the caller's stream also waits for the last forward kernel itself (it has consumed all of its tiles, so this is immediate)
    if (cudaEventRecord(ev, st_hi) != cudaSuccess || cudaStreamWaitEvent(st, ev, 0) != cudaSuccess) return fail(SS_ERR_CUDA);
    seg = (seg + segs - 1) % segs;
    if (cudaMemcpyAsync(actions, ring_act + seg * rows * 2, (size_t)rows * 8, cudaMemcpyDeviceToDevice, st) != cudaSuccess ||
        cudaMemcpyAsync(reward, ring_reward + seg * rows, (size_t)rows * 4, cudaMemcpyDeviceToDevice, st) != cudaSuccess)
        return fail(SS_ERR_CUDA);
    cudaEventDestroy(ev);
    return SS_OK;
}

int ss_selfplay_rollout2(void *env_state, int64_t n_envs, const float *actor_params, float *obs_a, float *obs_b,
                         float *actions, float *reward, uint8_t *done, uint8_t *winner,
                         float *ring_obs, float *ring_act, float *ring_reward, float *ring_next_obs, uint8_t *ring_done,
                         int64_t capacity, int64_t write_pos, int n_ticks, float param_noise_sd, int64_t noise_group,
                         float action_noise_sd, int tensor_cores, int reward_mode, int64_t tick_limit, int reset_mode,
                         uint64_t env_seed, uint64_t env_counter, uint64_t noise_seed, uint64_t noise_counter,
                         const void *speeds, uint32_t *status, int step_flags, int *tile_ready, void *stream2, void *stream) {
    const int64_t rows = 2 * n_envs;
    const bool in_place = ring_obs && winner && n_envs > 0 && capacity % rows == 0 && write_pos % rows == 0 && write_pos >= 0 &&
                          write_pos < capacity && (capacity / rows >= 2 || n_ticks == 1);
    if (in_place && tile_ready && stream2 && stream2 != stream && tensor_cores && !speeds && reward_mode != SS_REWARD_SIMPLE &&
        env_state && actor_params && obs_a && actions && reward && done && n_ticks > 0)
        return rollout_overlapped(env_state, n_envs, actor_params, obs_a, actions, reward, done, winner, ring_obs, ring_act,
                                  ring_reward, ring_next_obs, ring_done, capacity, write_pos, n_ticks, param_noise_sd, noise_group,
                                  action_noise_sd, reward_mode, tick_limit, reset_mode, env_seed, env_counter, noise_seed,
                                  noise_counter, status, step_flags, tile_ready, (cudaStream_t)stream, (cudaStream_t)stream2);
    return ss_selfplay_rollout(env_state, n_envs, actor_params, obs_a, obs_b, actions, reward, done, winner, ring_obs, ring_act,
                               ring_reward, ring_next_obs, ring_done, capacity, write_pos, n_ticks, param_noise_sd, noise_group,
                               action_noise_sd, tensor_cores, reward_mode, tick_limit, reset_mode, env_seed, env_counter, noise_seed,
                               noise_counter, speeds, status, step_flags, stream);
}

int ss_selfplay_rollout(void *env_state, int64_t n_envs, const float *actor_params, float *obs_a, float *obs_b,
                        float *actions, float *reward, uint8_t *done, uint8_t *winner,
                        float *ring_obs, float *ring_act, float *ring_reward, float *ring_next_obs, uint8_t *ring_done,
                        int64_t capacity, int64_t write_pos, int n_ticks, float param_noise_sd, int64_t noise_group,
                        float action_noise_sd, int tensor_cores, int reward_mode, int64_t tick_limit, int reset_mode,
                        uint64_t env_seed, uint64_t env_counter, uint64_t noise_seed, uint64_t noise_counter,
                        const void *speeds, uint32_t *status, int step_flags, void *stream) {
    if (!env_state || !actor_params || !obs_a || !obs_b || !actions || !reward || !done || n_envs <= 0 || n_ticks <= 0)
        return SS_ERR_INVALID_ARG;
    const bool store = ring_obs != nullptr;
    if (store && (2 * n_envs > capacity || write_pos < 0 || write_pos >= capacity)) return SS_ERR_INVALID_ARG;
    const int64_t rows = 2 * n_envs;
    if (store && !winner) return SS_ERR_INVALID_ARG;      // the ring's done flag is the hit flag (winner != 0)
    // (with a single segment the step kernel's second observation copy would land in the very rows the actor has just read
    //  and overwrite the stored transition's obs with its next_obs: the in-place form needs two segments or a single tick)
    if (store && capacity % rows == 0 && write_pos % rows == 0 && (capacity / rows >= 2 || n_ticks == 1)) {
        // transitions produced in place: tick t owns ring rows [seg_t * rows, (seg_t + 1) * rows)
        const int64_t segs = capacity / rows;
        cudaStream_t st = (cudaStream_t)stream;
        int64_t seg = write_pos / rows;
        if (cudaMemcpyAsync(ring_obs + seg * rows * 12, obs_a, (size_t)rows * 48, cudaMemcpyDeviceToDevice, st) != cudaSuccess)
            return SS_ERR_CUDA;
        // The two kernels of a tick form a dependent-launch chain (ss_launch.cuh): each grid is placed while its predecessor
        // drains and holds at griddepcontrol.wait.  From the second tick on the forward kernel also stages (and perturbs) the
        // actor's parameters ahead of that wait -- its predecessor, the env step, does not write them; the first tick's
        // forward may follow an update's Adam kernel and waits first.  ss_set_dependent_launch(0): ordinary launches.
        // A tick stays two kernels: the whole tick as ONE kernel (ss_actor_forward_step_tc, the env step in the forward
        // kernel's output stage) is bit-identical and slower, 119 us per tick at 262,144 envs against 71 us -- the env tick
        // is ~450 dependent instructions, three float64 sin / cos among them, and the four output warps that would run it
        // are one warp per scheduler: nothing hides its latency there, while the stand-alone kernel runs 32 warps per SM
        // (profiles/r2_rollout_fused_vs_two_kernels.txt).
        const int kOn = (tensor_cores && sslaunch::chain_enabled()) ? sslaunch::kPdlOn : sslaunch::kPdlOff;
        sslaunch::PdlScope scope(kOn);
        for (int t = 0; t < n_ticks; ++t, seg = (seg + 1) % segs) {
            float *o = ring_obs + seg * rows * 12, *a = ring_act + seg * rows * 2;
            // the last tick's observation goes to the caller's buffer, the others to the next segment's rows
            float *o_next = (t + 1 < n_ticks) ? ring_obs + ((seg + 1) % segs) * rows * 12 : obs_a;
            sslaunch::pdl_mode() = (kOn && t > 0) ? (sslaunch::kPdlOn | sslaunch::kPdlEarlyWeights) : kOn;
            int rc = tensor_cores
                         ? ss_actor_forward_tc(actor_params, o, a, rows, param_noise_sd, noise_group, action_noise_sd, noise_seed,
                                               noise_counter + (uint64_t)t, stream)
                         : ss_actor_forward(actor_params, o, a, rows, param_noise_sd, noise_group, action_noise_sd, noise_seed,
                                            noise_counter + (uint64_t)t, stream);
            if (rc != SS_OK) return rc;
            sslaunch::pdl_mode() = kOn;
            rc = ss_env_step_ring(env_state, n_envs, a, ring_next_obs + seg * rows * 12, o_next, ring_reward + seg * rows, done,
                                  ring_done + seg * rows, winner, 1, reward_mode, tick_limit, 1, reset_mode, env_seed,
                                  env_counter + (uint64_t)t, speeds, status, step_flags, stream);
            if (rc != SS_OK) return rc;
        }
        // the last tick's actions and rewards for the caller's scratch tensors
        seg = (seg + segs - 1) % segs;
        if (cudaMemcpyAsync(actions, ring_act + seg * rows * 2, (size_t)rows * 8, cudaMemcpyDeviceToDevice, st) != cudaSuccess ||
            cudaMemcpyAsync(reward, ring_reward + seg * rows, (size_t)rows * 4, cudaMemcpyDeviceToDevice, st) != cudaSuccess)
            return SS_ERR_CUDA;
        return SS_OK;
    }
    for (int t = 0; t < n_ticks; ++t) {
        float *cur = (t & 1) ? obs_b : obs_a, *next = (t & 1) ? obs_a : obs_b;
        // both players of every env act from the same pre-tick observation (SkillshotLearner.py:304-310)
        int rc = tensor_cores
                     ? ss_actor_forward_tc(actor_params, cur, actions, 2 * n_envs, param_noise_sd, noise_group, action_noise_sd,
                                           noise_seed, noise_counter + (uint64_t)t, stream)
                     : ss_actor_forward(actor_params, cur, actions, 2 * n_envs, param_noise_sd, noise_group, action_noise_sd,
                                        noise_seed, noise_counter + (uint64_t)t, stream);
        if (rc != SS_OK) return rc;
        // game_tick, reward of the post-tick state, next observation; finished games restart (SkillshotLearner.py:312-315)
        rc = ss_env_step(env_state, n_envs, actions, next, reward, done, winner, 1, reward_mode, tick_limit, 1, reset_mode,
                         env_seed, env_counter + (uint64_t)t, speeds, status, step_flags, stream);
        if (rc != SS_OK) return rc;
        if (store) {
            rc = ss_replay_push(ring_obs, ring_act, ring_reward, ring_next_obs, ring_done, capacity,
                                (write_pos + (int64_t)t * 2 * n_envs) % capacity, cur, actions, reward, next, winner, 2,
                                2 * n_envs, stream);     // terminal = a hit (winner != 0); a tick-limit restart keeps its bootstrap
            if (rc != SS_OK) return rc;
        }
    }
    return SS_OK;
}

int64_t ss_actor_frames_params(int frames) { return frames < 1 ? -1 : (int64_t)DS * frames * H1 + H1 + H1 * H2 + H2 + H2 * DA + DA; }

int ss_param_noise_groups(const float *params, float *out, int64_t n_params, int64_t n_groups, int64_t stride, float sd,
                          uint64_t seed, uint64_t counter, void *stream) {
    if (!params || !out || n_params <= 0 || n_groups <= 0 || n_groups > 65535 || stride < n_params) return SS_ERR_INVALID_ARG;
    if ((((uintptr_t)params | (uintptr_t)out) & 15) || (stride & 3)) return SS_ERR_INVALID_ARG;
    const int64_t quads = (n_params + 3) / 4;
    param_noise_groups_kernel<<<dim3((unsigned)((quads + 127) / 128), (unsigned)n_groups), 128, 0, (cudaStream_t)stream>>>(
        params, out, n_params, stride, sd, seed, counter);
    return check_launch();
}

int ss_obs_stack_push(float *stack, int64_t n_rows, int frames, int64_t head, const float *obs, const uint8_t *done,
                      int done_div, void *stream) {
    if (!stack || !obs || n_rows <= 0 || frames < 1 || head < 0 || done_div < 1) return SS_ERR_INVALID_ARG;
    if (((uintptr_t)stack | (uintptr_t)obs) & 15) return SS_ERR_INVALID_ARG;
    obs_stack_push_kernel<<<(unsigned)((3 * n_rows + 255) / 256), 256, 0, (cudaStream_t)stream>>>(stack, n_rows, frames, head, obs,
                                                                                                 done, done_div);
    return check_launch();
}

int ss_obs_stack_ordered(const float *stack, int64_t n_rows, int frames, int64_t head, float *out, void *stream) {
    if (!stack || !out || n_rows <= 0 || frames < 1 || frames > SS_MAX_FRAMES || head < 0) return SS_ERR_INVALID_ARG;
    if (((uintptr_t)stack | (uintptr_t)out) & 15) return SS_ERR_INVALID_ARG;
    obs_stack_ordered_kernel<<<(unsigned)((3 * frames * n_rows + 255) / 256), 256, 0, (cudaStream_t)stream>>>(stack, n_rows, frames,
                                                                                                          head, out);
    return check_launch();
}

int ss_actor_forward_frames(const float *params, int64_t param_stride, int64_t noise_group, const float *stack, int frames,
                            int64_t head, float *act_out, int64_t n, void *stream) {
    if (!params || !stack || !act_out || n <= 0 || frames < 1 || frames > SS_MAX_FRAMES || head < 0 || param_stride < 0)
        return SS_ERR_INVALID_ARG;
    if (param_stride > 0 && noise_group <= 0) return SS_ERR_INVALID_ARG;
    if (((uintptr_t)params & 15) || (param_stride & 3) || ((uintptr_t)act_out & 7)) return SS_ERR_INVALID_ARG;
    FramesFwdArgs A{params, stack, act_out, n, param_stride > 0 ? noise_group : n, param_stride, head, frames};
    const size_t smem = (size_t)(DS * frames + H1 + H2 + DA) * PITCH * 4;
    const int64_t units = ((n + A.group - 1) / A.group) * ((A.group + TB - 1) / TB);
    const int grid = grid_for(actor_frames_fwd_kernel, smem, units, 0);
    if (grid < 0) return SS_ERR_CUDA;
    actor_frames_fwd_kernel<<<grid, NT, smem, (cudaStream_t)stream>>>(A);
    return check_launch();
}

}  // extern "C"
