// ss_mlp_tc.cu -- actor and critic forward passes on the 5th-generation tensor cores
// (tcgen05.mma, accumulators in tensor memory), sm_100a only.
//
// model_act* of the reference (SkillshotLearner.py:215-281) evaluates
// 12 -> 256 relu -> 128 relu -> 2 tanh for ONE observation per Keras predict().
// The batched rollout evaluates it for 2 x envs observations per tick
// (BASELINE.json configs 3-4: 524,288 .. 2,097,152 rows), which is two GEMMs per
// 128-row tile:
//
//   layer 1   D1[128 x 256] = X0[128 x 16]  . W1'[16 x 256]     fp16 operands, K = 12 + bias rows
//   layer 2   D2[128 x 128] = A1[128 x 272] . W2'[272 x 128]    bf16 operands, K = 256 + bias (+ action) rows
//   layer 3   128 -> 2 (actor, tanh) or 128 -> 1 (critic) on the CUDA cores in the epilogue, fp32
//
// The critic (SkillshotLearner.py:98-121, Dropout off) is the same pipeline: its action enters
// layer 2 through the tail chunk of A1, and its epilogue also produces -dQ/da (the upstream
// gradient of model_actor_fit_step) and the TD target r + gamma (1 - done) Q.
//
// One persistent CTA per SM keeps the weights resident in shared memory in the UMMA canonical
// K-major no-swizzle layout (ss_tc_common.cuh) and streams tiles through the role pipeline
// described above the kernel.  Synchronisation is mbarrier-only (tcgen05.commit arrives when
// the MMAs retire).
//
// Precision: fp32 master weights stay in HBM; accumulation is fp32.  Layer 1 runs in fp16: the
// observation's positions are multiples of 1/250 and fp16's 11-bit significand resolves them
// 8x finer than a pixel (a single bf16 would merge neighbouring pixels), the weights keep 11
// bits too, and K = 16 is a single MMA step.  Layer 2 runs in bf16 (the hidden activations are
// rounded to bf16 when they become its A operand).  All biases ride through the tensor core as
// extra K rows against a constant 1 in the A operand (bias as a high + low pair, accurate to
// 2^-17 or better), so epilogue 1 is tcgen05.ld -> cvt.rn.relu.bf16x2 -> st.shared only.
//
// Parameter noise (SkillshotLearner.py:260-265): the CTA perturbs the weights while staging
// them, w + w * (sd * eps), eps from the same Philox stream as the float32 path (ss_rng.cuh),
// one draw per noise group; groups are multiples of the 128-row tile so a tile never mixes two
// draws.
#include <stdlib.h>

#include "ss_tc_common.cuh"

#include "ss_env_pp.cuh"

namespace {

using namespace sstc;

struct FwdArgs {
    const float *params, *obs;
    int64_t n, group;
    // actor: actions out, exploration noise
    float *act_out;
    float param_sd, action_sd;
    uint64_t seed, counter;
    // critic: actions in; any of q_out / up_out / y_out
    const float *act_in;
    float *q_out;            // [n]     Q(s, a)
    float *up_out;           // [n][2]  -dQ/da, the upstream gradient of the actor's policy-gradient step
    float *y_out;            // [n]     reward + gamma * (1 - done) * Q   (TD target when params are the target critic)
    const float *reward;
    const uint8_t *done;
    float gamma;
    // fused env step (ss_actor_forward_step_tc): rows are players in env order (row = 2 env + player); the output-warp lane
    // that has just computed a player's action plays that player's tick (ss_env_pp.cuh) and writes the transition
    void *env_state;         // packed env state of n / 2 envs
    ss::TickParams TP;
    float4 *obs_next, *obs_next2;     // the next observation, [n][12] floats each (second copy may be NULL)
    float *reward_out;       // [n]
    uint8_t *done_out, *winner_out, *done_rows_out;     // [n / 2], [n / 2], [n]
    uint32_t *env_status;
    unsigned long long *env_stats;
    // overlapped rollout (ss_selfplay_rollout): tile_ready[row / 128] is incremented once by each of the four output warps
    // when its 32 actions of that tile are in global memory; the env step kernel running beside this one consumes them
    int *tile_ready;
    int early_weights;       // ss_launch.cuh: the parameters may be staged ahead of griddepcontrol.wait (set by launch_fwd)
    // actor -> critic pair in ONE launch (mlp_fwd_pair_kernel): the actor role's output lane of a row also writes the row's
    // two actions into pair_mail[row]; the critic role's producer lane of that row polls those 8 bytes until neither word is
    // the empty mark, takes them and puts the mark back.  The data is its own flag: no fence, no separate flag traffic
    // (a release store per tile cost the output warps ~700 cycles each, measured).
    int2 *pair_mail;
    // grouped forward (ss_actor_forward_groups_tc): row i uses the parameter vector params + (i / group) * param_stride
    int64_t param_stride;
};

// 32 accumulator columns (hidden-2 units) -> ReLU -> layer 3, four split accumulators per output.
// actor: the two 128 -> 2 dot products (W3 as stored, two units per 16-byte load).
// critic: q, and dq/da_m = sum_k [z_k > 0] W3[k] W2[256+m][k].
template <int NET>
__device__ __forceinline__ void layer3(const uint32_t (&v)[32], const float4 *w3x, float (&acc)[3][4]) {
    if (NET == NET_ACTOR) {
#pragma unroll
        for (int c = 0; c < 16; ++c) {
            const float4 w = w3x[c];                                           // W3[2c][0..1], W3[2c+1][0..1]
            const float ha = fmaxf(__uint_as_float(v[c * 2 + 0]), 0.f), hb = fmaxf(__uint_as_float(v[c * 2 + 1]), 0.f);
            acc[0][(c & 1) * 2 + 0] = fmaf(ha, w.x, acc[0][(c & 1) * 2 + 0]);
            acc[1][(c & 1) * 2 + 0] = fmaf(ha, w.y, acc[1][(c & 1) * 2 + 0]);
            acc[0][(c & 1) * 2 + 1] = fmaf(hb, w.z, acc[0][(c & 1) * 2 + 1]);
            acc[1][(c & 1) * 2 + 1] = fmaf(hb, w.w, acc[1][(c & 1) * 2 + 1]);
        }
    } else {
#pragma unroll
        for (int c = 0; c < 32; ++c) {
            const float4 w = w3x[c];
            const float z = __uint_as_float(v[c]);
            const float gate = z > 0.f ? 1.f : 0.f;
            acc[0][c & 3] = fmaf(fmaxf(z, 0.f), w.x, acc[0][c & 3]);
            acc[1][c & 3] = fmaf(gate, w.y, acc[1][c & 3]);
            acc[2][c & 3] = fmaf(gate, w.z, acc[2][c & 3]);
        }
    }
}

// ---- the kernel ------------------------------------------------------------------------
// Three roles run as a software pipeline over the CTA's 128-row tiles:
//
//   P warps (4)   stage X0(t+2);  wait MMA1(t);  D1 -> ReLU -> bf16 -> A1[t % 2]       (layer-1 epilogue)
//   Q warps (4)   wait MMA2(t);  D2[t % 2] -> ReLU -> layer 3 -> output
//   MMA warp      MMA1(t+1): D1 = X0[(t+1) % 2] . W1'    then    MMA2(t): D2[t % 2] = A1[t % 2] . W2'
//
// A1, X0 and D2 are double-buffered, D1 is single (256 + 2 x 128 tensor-memory columns, 220 KB of shared
// memory).  Per tile the MMA warp waits twice and commits twice.  History (profiles/README.md): a first
// version gave each of two whole-tile "slots" its own four warps for the entire chain stage -> MMA1 ->
// epilogue 1 -> MMA2 -> epilogue 2 (tensor pipe 43-47 % busy: the chain is ~4x a tile's MMA time and there
// is no shared memory for a third 68 KB tile); a 64-column block pipeline between the layers ran 2x SLOWER
// (issue-bound: 25 MMAs, 10 waits, 10 commits per tile on the one issuing thread).  An event trace of this
// version (profiles/r1_actor_fwd_tc_event_trace.txt) showed the MMA warp as the pacing role.
namespace pipe {

// the "empty" word of the pair mailbox: a NaN payload no arithmetic produces (tanhf of a NaN gives the canonical 0x7fffffff)
constexpr int kMailEmpty = SS_PAIR_MAIL_EMPTY;

constexpr int P_WARPS = 4, Q_WARPS = 4, MMA_W = 8, NTH = 32 * 9;

constexpr uint32_t SMP_B1 = 0;                              // [K1F/8][256][8] fp16
constexpr uint32_t SMP_B2 = SMP_B1 + (K1F / 8) * CHUNK_B1;  // [K2/8][128][8] bf16
constexpr uint32_t SMP_A1 = SMP_B2 + B2_BYTES;              // 2 x [K2/8][128][8] bf16: hidden layer 1 (+ tail) of tile t in A1[t & 1]
constexpr uint32_t SMP_X0 = SMP_A1 + 2 * X2_BYTES;          // 2 x [K1F/8][128][8] fp16: observations of tile t in X0[t & 1]
constexpr uint32_t X0_BYTES = (K1F / 8) * CHUNK_A;
constexpr uint32_t SMP_W3 = SMP_X0 + 2 * X0_BYTES;
constexpr uint32_t SMP_B3 = SMP_W3 + H2 * 16;
constexpr uint32_t SMP_BAR = SMP_B3 + 16;
// barriers: X (producers -> MMA warp, one arrival round per hand-off), Z (MMA1 retired), Y[2] (MMA2 retired),
// D2E[2] (output warps have read D2[s])
constexpr int B_X = 0, B_Z = 1, B_Y = 2, B_D2E = 4, B_COUNT = 6;
constexpr uint32_t SMP_TMEM = SMP_BAR + B_COUNT * 8;
constexpr uint32_t SMP_TOTAL = SMP_TMEM + 16;
static_assert(SMP_TOTAL <= 227 * 1024, "shared memory budget");

// GROUPS: this CTA's tiles [u0, u1) when the CTAs are split over the groups in proportion to the groups' tiles (the last
// group may be shorter), every range inside one group, so that a CTA stages one parameter vector once.  With fewer CTAs
// than groups the tiles are split evenly and a range may cross groups (the segment loop restages at each boundary).
__device__ __forceinline__ void group_units(int64_t n, int64_t group, int64_t upg, int cta, int ncta, int64_t &u0, int64_t &u1) {
    const int64_t G = (n + group - 1) / group;
    const int64_t last = (n - (G - 1) * group + TM - 1) / TM;          // tiles of the last group
    if (ncta < G) {
        u0 = G * upg * cta / ncta; u1 = G * upg * (cta + 1) / ncta;
        return;
    }
    const int64_t T = (G - 1) * upg + last;
    // group g owns CTAs [floor(g upg ncta / T), floor((g + 1) upg ncta / T)), the last group up to ncta; each owns >= 1
    const int64_t g = min(G - 1, ((int64_t)(cta + 1) * T - 1) / (upg * ncta));
    const int64_t c0 = g * upg * ncta / T, c1 = g + 1 == G ? ncta : (g + 1) * upg * ncta / T;
    const int64_t tiles = g + 1 == G ? last : upg, j = cta - c0, k = c1 - c0;
    u0 = g * upg + tiles * j / k; u1 = g * upg + tiles * (j + 1) / k;
}

// SEGMENTS: the unit -> (segment, first row) table of ss_actor_forward_segments_tc, passed by value beside FwdArgs.  Segment s
// = tiles [unit0[s], unit0[s + 1]) = rows [row0[s], row0[s + 1]), worked by CTAs [cta0[s], cta0[s + 1]) (at least one).
struct SegTable {
    int n;
    int64_t unit0[SS_LEAGUE_MAX_POLICIES + 1], row0[SS_LEAGUE_MAX_POLICIES + 1];
    int cta0[SS_LEAGUE_MAX_POLICIES + 1];
};

// the segment that holds tile u (the segments are few: a linear walk)
__device__ __forceinline__ int segment_of(const SegTable &T, int64_t u) {
    int s = 0;
    while (s + 1 < T.n && u >= T.unit0[s + 1]) ++s;
    return s;
}

// cta / ncta: this CTA's index among the CTAs that share the work of A (the whole grid, or one role's part of a pair launch)
// GROUPS (actor only): one parameter vector per group of A.group rows instead of one perturbed vector per noise group
// SEGS (actor only): one parameter vector per segment of *T instead; no tile mixes two segments
template <int NET, bool FUSED, bool GROUPS = false, bool SEGS = false>
__device__ __forceinline__ void fwd_body(const FwdArgs &A, const int cta, const int ncta, const SegTable *T = nullptr) {
    extern __shared__ __align__(128) uint8_t smem[];
    const uint32_t sbase = smem_u32(smem);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    auto bar = [&](int idx) -> uint32_t { return sbase + SMP_BAR + (uint32_t)idx * 8; };
    if (threadIdx.x == 0) {
        mbar_init(bar(B_X), 128);
        mbar_init(bar(B_Z), 1);
        for (int i = 0; i < 2; ++i) { mbar_init(bar(B_Y + i), 1); mbar_init(bar(B_D2E + i), 128); }
        mbar_fence_init();
    }
    if (warp == MMA_W) tmem_alloc(sbase + SMP_TMEM, 512);
    // (stage_weights writes every byte of both weight images except the layer-2 image's padding chunk)
    for (uint32_t o = threadIdx.x * 16; o < CHUNK_B2; o += NTH * 16)
        *reinterpret_cast<uint4 *>(smem + SMP_B2 + (K2 / 8 - 1) * CHUNK_B2 + o) = make_uint4(0, 0, 0, 0);
    if (warp < P_WARPS) {                                    // tail chunks of both activation tiles: actor {1 1 0 ..} | 0
        for (int t = 0; t < 2; ++t) {
            uint8_t *arow = smem + SMP_A1 + t * X2_BYTES + threadIdx.x * 16;
            *reinterpret_cast<uint4 *>(arow + (H1 / 8) * CHUNK_A) = tail_chunk_actor();
            *reinterpret_cast<uint4 *>(arow + (H1 / 8 + 1) * CHUNK_A) = make_uint4(0, 0, 0, 0);
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *reinterpret_cast<const volatile uint32_t *>(smem + SMP_TMEM);

    const bool noisy = NET == NET_ACTOR && !GROUPS && !SEGS && A.param_sd > 0.f;
    const int64_t group = (noisy || GROUPS) ? A.group : A.n;
    const int64_t upg = (group + TM - 1) / TM;
    const int64_t n_groups = (A.n + group - 1) / group;
    const int64_t units = n_groups * upg;
    int64_t u0 = units * cta / ncta, u1 = units * (cta + 1) / ncta;
    if (GROUPS) group_units(A.n, group, upg, cta, ncta, u0, u1);
    if (SEGS) {                                              // this CTA's share of its segment's tiles
        int s = 0;
        while (s + 1 < T->n && cta >= T->cta0[s + 1]) ++s;
        const int64_t tiles = T->unit0[s + 1] - T->unit0[s], j = cta - T->cta0[s], k = T->cta0[s + 1] - T->cta0[s];
        u0 = T->unit0[s] + tiles * j / k; u1 = T->unit0[s] + tiles * (j + 1) / k;
    }

    uint32_t tcount = 0;                                     // tiles done by this CTA: buffers = tcount & 1, parities from tcount
    uint32_t xph = 0;                                        // MMA warp: parity of the next X hand-off
    uint32_t env_status = 0;                                 // FUSED: SS_STATUS_* bits of this thread's env ticks
    bool waited = false;                                     // griddepcontrol.wait executed (ss_launch.cuh)

    for (int64_t u = u0; u < u1;) {
        const int64_t g = SEGS ? segment_of(*T, u) : u / upg;
        const int64_t seg_end = SEGS ? min(u1, T->unit0[g + 1]) : min(u1, (g + 1) * upg);
        const int64_t ntiles = seg_end - u;
        const int64_t end = SEGS ? T->row0[g + 1] : min(A.n, (g + 1) * group);
        // first row of the segment's first tile
        const int64_t row0 = SEGS ? T->row0[g] + (u - T->unit0[g]) * TM : g * group + (u - g * upg) * TM;
        const int r = (warp & 3) * 32 + lane;                     // row of the tile = tensor-memory lane

        float4 xin[3];
        // first segment of a dependent launch (ss_launch.cuh): everything above ran beside the previous grid's tail; the
        // weights are staged ahead of the wait too when the caller knows that grid does not write them
        if (!waited && !A.early_weights) { sslaunch::griddep_wait(); sslaunch::griddep_launch(); waited = true; }
        if (waited && warp < P_WARPS) load_obs(A.obs, row0 + r, end, xin);
        stage_weights<NET, NTH, true>(Stager{(GROUPS || SEGS) ? A.params + g * A.param_stride : A.params, smem + SMP_B1, smem + SMP_B2,
                                             reinterpret_cast<float4 *>(smem + SMP_W3), reinterpret_cast<float *>(smem + SMP_B3),
                                             noisy, A.param_sd, A.seed, A.counter, (uint32_t)g});
        if (!waited) {
            sslaunch::griddep_wait();
            sslaunch::griddep_launch();
            waited = true;
            if (warp < P_WARPS) load_obs(A.obs, row0 + r, end, xin);
        }
        fence_proxy_async();
        __syncthreads();

        if (warp < P_WARPS) {
            // ============ producer warps: observation staging and the layer-1 epilogue ============
            const uint32_t tl = tmem + ((uint32_t)((warp & 3) * 32) << 16);
            auto stage_x0 = [&](int64_t i) {                      // observations of tile i -> X0[(tcount + i) & 1]
                store_obs_row_f16(xin, smem + SMP_X0 + ((tcount + (uint32_t)i) & 1) * X0_BYTES + r * 16);
                load_obs(A.obs, row0 + (i + 1) * TM + r, (i + 1 < ntiles) ? end : 0, xin);   // prefetch the next tile's row
            };
            int2 pair_v = make_int2(0, 0);                        // pair launch, critic role: this lane's row of the mailbox ...
            bool pair_have = false;                               // ... holds the coming tile's actions already
            stage_x0(0);
            fence_proxy_async();
            mbar_arrive(bar(B_X));                                // -> MMA1(tile 0)
            if (ntiles > 1) stage_x0(1);
            for (int64_t i = 0; i < ntiles; ++i) {
                const uint32_t tc = tcount + (uint32_t)i;
                uint8_t *arow = smem + SMP_A1 + (tc & 1) * X2_BYTES + r * 16;
                float2 act = make_float2(0.f, 0.f);
                if (NET == NET_CRITIC && A.pair_mail) {
                    // pair launch: this row's action comes from the actor role.  Usually it was taken during the previous
                    // tile (below); otherwise poll for it here.
                    const int64_t prow = row0 + i * TM + r;
                    if (!pair_have) {
                        uint32_t spins = 0;
                        for (;;) {
                            if (prow < end)
                                asm volatile("ld.volatile.global.v2.s32 {%0, %1}, [%2];" : "=r"(pair_v.x), "=r"(pair_v.y) : "l"(A.pair_mail + prow));
                            if (__all_sync(0xffffffffu, prow >= end || (pair_v.x != kMailEmpty && pair_v.y != kMailEmpty))) break;
                            if (++spins > (1u << 24)) __trap();       // the actor role never ran: a protocol bug, not a hang
                            __nanosleep(20);
                        }
                        if (prow < end) A.pair_mail[prow] = make_int2(kMailEmpty, kMailEmpty);      // left empty for the next launch
                    }
                    if (prow < end) act = make_float2(__int_as_float(pair_v.x), __int_as_float(pair_v.y));
                    pair_have = false;
                    // one look at the next tile's row, issued now and examined at the end of this iteration
                    if (i + 1 < ntiles && prow + TM < end)
                        asm volatile("ld.volatile.global.v2.s32 {%0, %1}, [%2];" : "=r"(pair_v.x), "=r"(pair_v.y) : "l"(A.pair_mail + prow + TM));
                } else if (NET == NET_CRITIC && row0 + i * TM + r < end) {
                    act = __ldg(reinterpret_cast<const float2 *>(A.act_in) + row0 + i * TM + r);
                }
                // MMA1(tile) retired: D1 holds layer 1 and X0[tc & 1] is dead.  The tensor pipe retires one thread's MMAs
                // in issue order and MMA2(tile - 2) was issued before MMA1(tile), so A1[tc & 1] is free as well.
                mbar_wait(bar(B_Z), tc & 1);
                tc_fence_after();
                if (NET == NET_CRITIC) *reinterpret_cast<uint4 *>(arow + (H1 / 8) * CHUNK_A) = tail_chunk_critic(act.x, act.y);
                {
                    uint32_t va[32], vb[32];
                    tmem_ld32(tl, va);
#pragma unroll
                    for (int j = 0; j < H1 / 32; j += 2) {
                        tmem_wait_ld();
                        tmem_ld32(tl + (j + 1) * 32, vb);
                        relu_pack_store(va, arow + (uint32_t)(j * 4) * CHUNK_A);
                        tmem_wait_ld();
                        if (j + 2 < H1 / 32) tmem_ld32(tl + (j + 2) * 32, va);
                        relu_pack_store(vb, arow + (uint32_t)((j + 1) * 4) * CHUNK_A);
                    }
                }
                fence_proxy_async();
                tc_fence_before();
                mbar_arrive(bar(B_X));                            // A1[tile] full, D1 free, X0(tile + 1) staged
                if (i + 2 < ntiles) stage_x0(i + 2);              // into X0[tc & 1]
                if (NET == NET_CRITIC && A.pair_mail && i + 1 < ntiles) {
                    // the next tile's actions, if the actor role has delivered all 32 by now
                    const int64_t nrow = row0 + (i + 1) * TM + r;
                    pair_have = __all_sync(0xffffffffu, nrow >= end || (pair_v.x != kMailEmpty && pair_v.y != kMailEmpty));
                    if (pair_have && nrow < end) A.pair_mail[nrow] = make_int2(kMailEmpty, kMailEmpty);
                }
            }
        } else if (warp < P_WARPS + Q_WARPS) {
            // ============ output warps: layer 3 on D2 ============
            const uint32_t tl = tmem + ((uint32_t)((warp & 3) * 32) << 16) + 256;
            const float4 *w3x = reinterpret_cast<const float4 *>(smem + SMP_W3);
            const float *b3 = reinterpret_cast<const float *>(smem + SMP_B3);
            for (int64_t i = 0; i < ntiles; ++i) {
                const uint32_t tc = tcount + (uint32_t)i, slot = tc & 1;
                const int64_t row = row0 + i * TM + r;
                // FUSED: this row's player.  Its state and the sin / cos of its two rotations do not depend on the action:
                // they are fetched and evaluated here, in the time this warp would otherwise spend waiting for MMA2.
                sspp::LaneState L;
                sspp::LaneTrig T;
                const int64_t gl = FUSED ? min(row, A.n - 2 + (int64_t)(lane & 1)) : 0;      // rows past the end replay the last env
                if (FUSED) {
                    sspp::lane_load((const char *)A.env_state, A.n >> 1, gl, L);
                    sspp::lane_trig(L, T);
                }
                mbar_wait(bar(B_Y + slot), (tc >> 1) & 1);
                tc_fence_after();
                float acc[3][4] = {{b3[0], 0.f, 0.f, 0.f}, {NET == NET_ACTOR ? b3[1] : 0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
                {
                    constexpr int kW3Step = NET == NET_ACTOR ? 16 : 32;
                    uint32_t va[32], vb[32];
                    tmem_ld32(tl + slot * 128, va);
#pragma unroll
                    for (int j = 0; j < H2 / 32; j += 2) {
                        tmem_wait_ld();
                        tmem_ld32(tl + slot * 128 + (j + 1) * 32, vb);
                        layer3<NET>(va, w3x + j * kW3Step, acc);
                        tmem_wait_ld();
                        if (j + 2 < H2 / 32) tmem_ld32(tl + slot * 128 + (j + 2) * 32, va);
                        else { tc_fence_before(); mbar_arrive(bar(B_D2E + slot)); }     // D2[slot] fully read
                        layer3<NET>(vb, w3x + (j + 1) * kW3Step, acc);
                    }
                }
                const float out0 = (acc[0][0] + acc[0][1]) + (acc[0][2] + acc[0][3]);
                const float out1 = (acc[1][0] + acc[1][1]) + (acc[1][2] + acc[1][3]);
                const float out2 = (acc[2][0] + acc[2][1]) + (acc[2][2] + acc[2][3]);
                float fa0 = 0.f, fa1 = 0.f;                   // FUSED: the action this lane hands to its player's tick
                if (row < end) {
                    if (NET == NET_ACTOR) {
                        float a0 = tanhf(out0), a1 = tanhf(out1);
                        if (A.action_sd > 0.f) {
                            float zn[4];
                            normal4(A.seed, kTagActionNoise, (uint32_t)row, (uint32_t)(row >> 32), A.counter, zn);
                            a0 += A.action_sd * zn[0];
                            a1 += A.action_sd * zn[1];
                        }
                        reinterpret_cast<float2 *>(A.act_out)[row] = make_float2(a0, a1);
                        if (A.pair_mail) A.pair_mail[row] = make_int2(__float_as_int(a0), __float_as_int(a1));
                        if (FUSED) { fa0 = a0; fa1 = a1; }
                    } else {
                        if (A.q_out) A.q_out[row] = out0;
                        if (A.up_out) reinterpret_cast<float2 *>(A.up_out)[row] = make_float2(-out1, -out2);
                        if (A.y_out) A.y_out[row] = A.reward[row] + A.gamma * ((A.done && A.done[row]) ? 0.f : 1.f) * out0;
                    }
                }
                if (NET == NET_ACTOR && A.tile_ready) {
                    __threadfence();                                      // this lane's action store, device-wide
                    __syncwarp();
                    if (lane == 0) atomicAdd(A.tile_ready + (row0 + i * TM) / TM, 1);
                }
                if (FUSED) {
                    // do_actions + game_tick + reward + auto-reset + next observation of this player, on the spot: all 32
                    // lanes take part (the hit test is a shuffle and a ballot between the two lanes of an env)
                    const int P = lane & 1;
                    sspp::LaneTickOut o;
                    sspp::lane_obs_tick(L, T, fa0, fa1, A.TP, (uint64_t)(gl >> 1), A.TP.counter, lane, P, env_status, o);
                    const int v_other = __shfl_xor_sync(0xffffffffu, L.valid, 1);
                    if (row < end) {
                        sspp::lane_store((char *)A.env_state, A.n >> 1, row, L, v_other);
                        if (A.reward_out) A.reward_out[row] = o.reward;
                        uint8_t *flag = P ? A.winner_out : A.done_out;
                        if (flag) flag[row >> 1] = (uint8_t)(P ? o.winner : o.done);
                        if (A.done_rows_out) A.done_rows_out[row] = o.winner ? 1 : 0;
                        if (A.env_stats && !P && o.episode_len >= 0)
                            sspp::count_episode_pp(A.env_stats, o.episode_len, o.winner, (int)A.TP.tick_limit);
#pragma unroll
                        for (int j = 0; j < 3; ++j) {
                            A.obs_next[row * 3 + j] = o.obs[j];
                            if (A.obs_next2) A.obs_next2[row * 3 + j] = o.obs[j];
                        }
                    }
                }
            }
        } else {
            // ============ the MMA-issuing warp ============
            // Measured on B200 (tools/umma_probe.cu): ~54 cycles to issue one tcgen05.mma, ~50 per commit and ~170 for a
            // wait even on a completed barrier, against 68 cycles of execution for a 128 x 128 x 16 MMA: per tile this
            // warp can afford two waits and two commits, not more.  Tried and measured, none of them a gain:
            //  * slotting the next tile's hand-off into the middle of the layer-2 chain -- no change (the pipe queues
            //    only a couple of MMAs: the issue stream is never far ahead of it; tools/umma_probe3.cu shows that
            //    tcgen05.ld, shared-memory and bulk-copy traffic beside an MMA stream do not slow it);
            //  * two issuing warps alternating tiles -- the tensor pipe is one in-order queue, so MMA1(t+1), which the
            //    producers wait for, lands behind the other warp's 17-step MMA2 chain; and two issuing warps split by
            //    LAYER (one issues every MMA1 the moment a tile is handed over, the other the MMA2 chains back to back,
            //    producers waiting explicitly for MMA2(t-2)) -- correct, 5 % slower: the output warps' ~1.8 k cycles per
            //    tile and the producers' ~1.2 k are then the pace, not the issuing thread;
            //  * both waits first, then MMA1(t+1) and the MMA2(t) chain back to back with one fence -- no change;
            //  * ablations (a development build, 524,288 rows): 44.5 us whole, 37.4 with the output warps' layer 3 switched
            //    off, 40.2 with the producers' conversion off, 35.3 with both off -- the issuing loop alone (two waits,
            //    MMA1, 17 x MMA2, two commits per tile) already takes ~1.9 k cycles per tile against 1.29 k of MMA execution;
            //  * fetching the output warps' layer-3 weights eight loads ahead of their FMAs -- their pass over D2 drops
            //    from ~1.6 k to ~1.2 k cycles per tile (event trace) and the KERNEL gets 6 % slower;
            //  * eight producer warps (two per tensor-memory lane quadrant) -- 12 % SLOWER;
            //  * cta_group::2 (a cluster of two CTAs, one thread issuing M = 256 pair MMAs for both, each CTA holding
            //    half of the weight images, hand-offs through the cluster address window, multicast commits) --
            //    correct on the first run and 13 % SLOWER: halving the issue overhead does not help because the
            //    producers' loop (wait MMA1 -> epilogue 1 -> hand-off -> issuer wake-up -> MMA1) is the pacing chain
            //    and its MMA1 round trip then crosses SMs.  With D1 single-buffered (tensor memory is full: 256 + 2 x
            //    128 columns) that round trip cannot be overlapped; a packed fp16 layer-1 accumulator (128 columns)
            //    would make room for a second D1 and is the remaining idea.
            constexpr uint32_t kI1 = umma_idesc_f16(TM, H1), kI2 = umma_idesc(TM, H2);
            const uint64_t a1d = desc_kmajor(sbase + SMP_A1, CHUNK_A), x0d = desc_kmajor(sbase + SMP_X0, CHUNK_A);
            const uint64_t b1d = desc_kmajor(sbase + SMP_B1, CHUNK_B1), b2d = desc_kmajor(sbase + SMP_B2, CHUNK_B2);
            const uint32_t tc0 = __shfl_sync(0xffffffffu, tcount, 0);     // warp-uniform for the descriptor arithmetic
            auto mma1 = [&](uint32_t tc) {                        // D1 = X0(tile tc) . W1'   (fp16, one K step)
                if (lane == 0) {
                    umma_bf16(tmem, desc_advance(x0d, (tc & 1) * X0_BYTES), b1d, kI1, 0);
                    umma_commit(bar(B_Z));
                }
            };
            mbar_wait_likely_done(bar(B_X), xph); xph ^= 1;
            tc_fence_after();
            mma1(tc0);
            for (int64_t i = 0; i < ntiles; ++i) {
                const uint32_t tc = __shfl_sync(0xffffffffu, tc0 + (uint32_t)i, 0), slot = tc & 1;
                mbar_wait_likely_done(bar(B_X), xph); xph ^= 1;   // A1[tile] full, D1 free, X0(tile + 1) staged
                tc_fence_after();
                if (i + 1 < ntiles) mma1(tc + 1);
                mbar_wait_likely_done(bar(B_D2E + slot), ((tc >> 1) & 1) ^ 1);    // the output warps have drained D2[slot]
                tc_fence_after();
                if (lane == 0) {
                    const uint64_t ad = desc_advance(a1d, slot * X2_BYTES);
#pragma unroll
                    for (int ks = 0; ks < K2 / 16; ++ks)
                        umma_bf16(tmem + 256 + slot * 128, desc_advance(ad, 2 * CHUNK_A * ks), desc_advance(b2d, 2 * CHUNK_B2 * ks),
                                  kI2, ks > 0);
                    umma_commit(bar(B_Y + slot));
                }
            }
        }
        tcount += (uint32_t)ntiles;
        u = seg_end;
        tc_fence_before();
        __syncthreads();                   // pipeline drained: the output warps have read the last D2
        tc_fence_after();
    }

    if (!waited) { sslaunch::griddep_wait(); sslaunch::griddep_launch(); }      // a CTA without a tile still waits
    tc_fence_before();
    __syncthreads();
    if (warp == MMA_W) {
        tc_fence_after();
        tmem_dealloc(tmem, 512);
    }
    if (FUSED && env_status && A.env_status) atomicOr(A.env_status, env_status);
}

template <int NET, bool FUSED = false>
__global__ void __launch_bounds__(NTH, 1) mlp_fwd_pipe_kernel(const FwdArgs A) {
    fwd_body<NET, FUSED>(A, (int)blockIdx.x, (int)gridDim.x);
}

// a = actor(s) and critic(s, a) in ONE launch: the first `ga` CTAs play the actor role, the others the critic role, each
// over all the tiles; a critic CTA walks the same tiles in the same order as the actor CTA of the same index and takes
// each row's actions as soon as they are out (pair_mail).  At a 65,536-row minibatch a forward launch is mostly set-up
// and pipeline fill (3.5 tiles per CTA); two launches back to back pay that twice, the pair once, on half the SMs each.
// All CTAs are resident together (grid <= SMs, one CTA per SM), and a producer never waits for a consumer.
__global__ void __launch_bounds__(NTH, 1) mlp_fwd_pair_kernel(const FwdArgs Aa, const FwdArgs Ac, const int ga) {
    if ((int)blockIdx.x < ga) fwd_body<NET_ACTOR, false>(Aa, (int)blockIdx.x, ga);
    else fwd_body<NET_CRITIC, false>(Ac, (int)blockIdx.x - ga, (int)gridDim.x - ga);
}

// ss_actor_forward_groups_tc: the actor pipeline with one parameter vector per group of rows
__global__ void __launch_bounds__(NTH, 1) mlp_fwd_groups_kernel(const FwdArgs A) {
    fwd_body<NET_ACTOR, false, true>(A, (int)blockIdx.x, (int)gridDim.x);
}

// ss_actor_forward_segments_tc: the actor pipeline with one parameter vector per segment of rows (the table by value: it is
// read in place from the parameter space)
__global__ void __launch_bounds__(NTH, 1) mlp_fwd_segments_kernel(const FwdArgs A, const __grid_constant__ SegTable T) {
    fwd_body<NET_ACTOR, false, false, true>(A, (int)blockIdx.x, (int)gridDim.x, &T);
}

}  // namespace pipe

template <int NET, bool FUSED = false>
int launch_fwd(const FwdArgs &A, void *stream) {
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return SS_ERR_CUDA;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return SS_ERR_CUDA;
    const int64_t n_groups = (A.n + A.group - 1) / A.group;
    const int64_t units = n_groups * ((A.group + TM - 1) / TM);
    // no more CTAs than the rounds need (512 tiles on 148 SMs: 128 CTAs of four tiles each; fewer CTAs stage the weights)
    const int64_t rounds = (units + sms - 1) / sms;
    int grid = (int)((units + rounds - 1) / rounds);
    // perturbed weights are staged once per noise group a CTA touches: when the groups fit the SMs, give every CTA
    // exactly one group (the kernel's even split of units is then group-aligned) instead of letting ranges straddle two
    if (A.group < A.n && n_groups <= sms) grid = (int)n_groups;
    if (cudaFuncSetAttribute(pipe::mlp_fwd_pipe_kernel<NET, FUSED>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)pipe::SMP_TOTAL) != cudaSuccess)
        return SS_ERR_CUDA;
    FwdArgs B = A;
    B.early_weights = sslaunch::take_early_weights();
    if (sslaunch::launch(pipe::mlp_fwd_pipe_kernel<NET, FUSED>, dim3(grid), dim3(pipe::NTH), pipe::SMP_TOTAL, (cudaStream_t)stream, B) !=
        cudaSuccess)
        return SS_ERR_CUDA;
    return cudaGetLastError() == cudaSuccess ? SS_OK : SS_ERR_CUDA;
}

}  // namespace

// tile_ready (may be NULL): int32 [ceil(n / 128)], see FwdArgs; *grid_out / *units_out (may be NULL) receive the launch's
// CTA count and tile count, which a consumer kernel needs to walk the tiles in the order this one completes them
extern "C" int ss_actor_forward_tc_signal(const float *actor_params, const float *obs, float *act_out, int64_t n,
                                          float param_noise_sd, int64_t noise_group, float action_noise_sd,
                                          uint64_t seed, uint64_t counter, int *tile_ready, int *grid_out, int64_t *units_out,
                                          void *stream) {
    if (!actor_params || !obs || !act_out || n <= 0 || param_noise_sd < 0.f || action_noise_sd < 0.f)
        return SS_ERR_INVALID_ARG;
    if (((uintptr_t)actor_params | (uintptr_t)obs) & 15 || ((uintptr_t)act_out & 7)) return SS_ERR_INVALID_ARG;
    const bool noisy = param_noise_sd > 0.f;
    if (noisy && (noise_group <= 0 || noise_group % TM != 0)) return SS_ERR_INVALID_ARG;
    FwdArgs A{};
    A.params = actor_params; A.obs = obs; A.n = n; A.group = noisy ? noise_group : n;
    A.act_out = act_out; A.param_sd = param_noise_sd; A.action_sd = action_noise_sd; A.seed = seed; A.counter = counter;
    A.tile_ready = tile_ready;
    if (grid_out || units_out) {                              // the launch geometry of launch_fwd, for the consumer
        int dev = 0, sms = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
            return SS_ERR_CUDA;
        const int64_t n_groups = (A.n + A.group - 1) / A.group, units = n_groups * ((A.group + TM - 1) / TM);
        const int64_t rounds = (units + sms - 1) / sms;
        int grid = (int)((units + rounds - 1) / rounds);
        if (A.group < A.n && n_groups <= sms) grid = (int)n_groups;
        if (grid_out) *grid_out = grid;
        if (units_out) *units_out = units;
    }
    return launch_fwd<NET_ACTOR>(A, stream);
}

// One parameter vector per group of group_rows rows.  Launch geometry: as many CTAs as launch_fwd would give the real
// tiles, but at least one per group while the groups fit the SMs -- and the CTAs are split over the groups in proportion
// to their tiles (group_units), not one CTA per group: a match's two groups of 131,072 rows would otherwise run on 2 SMs.
extern "C" int ss_actor_forward_groups_tc(const float *params, int64_t param_stride, int64_t group_rows, const float *obs,
                                          float *act_out, int64_t n, void *stream) {
    if (!params || !obs || !act_out || n <= 0 || group_rows <= 0 || param_stride < 0) return SS_ERR_INVALID_ARG;
    if ((param_stride & 3) || (param_stride > 0 && param_stride < SS_ACTOR_PARAMS)) return SS_ERR_INVALID_ARG;
    if ((((uintptr_t)params | (uintptr_t)obs) & 15) || ((uintptr_t)act_out & 7)) return SS_ERR_INVALID_ARG;
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return SS_ERR_CUDA;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return SS_ERR_CUDA;
    const int64_t group = group_rows < n ? group_rows : n;
    const int64_t n_groups = (n + group - 1) / group;
    const int64_t tiles = (n_groups - 1) * ((group + TM - 1) / TM) + (n - (n_groups - 1) * group + TM - 1) / TM;
    const int64_t rounds = (tiles + sms - 1) / sms;
    int grid = (int)((tiles + rounds - 1) / rounds);
    if (n_groups <= sms && grid < n_groups) grid = (int)n_groups;
    FwdArgs A{};
    A.params = params; A.obs = obs; A.n = n; A.group = group; A.act_out = act_out; A.param_stride = param_stride;
    if (cudaFuncSetAttribute(pipe::mlp_fwd_groups_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pipe::SMP_TOTAL) !=
        cudaSuccess)
        return SS_ERR_CUDA;
    A.early_weights = sslaunch::take_early_weights();
    if (sslaunch::launch(pipe::mlp_fwd_groups_kernel, dim3(grid), dim3(pipe::NTH), pipe::SMP_TOTAL, (cudaStream_t)stream, A) !=
        cudaSuccess)
        return SS_ERR_CUDA;
    return cudaGetLastError() == cudaSuccess ? SS_OK : SS_ERR_CUDA;
}

// One parameter vector per segment.  Launch geometry: as many CTAs as launch_fwd would give the segments' tiles, but at
// least one per segment; each segment gets one CTA, then the rest go one at a time to the segment with the most tiles per
// CTA (never more CTAs than tiles), so the CTAs are split in proportion to the tiles and no CTA mixes two segments.
extern "C" int ss_actor_forward_segments_tc(const float *params, int64_t param_stride, const int64_t *seg_rows_host, int n_segs,
                                            const float *obs, float *act_out, void *stream) {
    if (!params || !obs || !act_out || !seg_rows_host || n_segs < 1 || n_segs > SS_LEAGUE_MAX_POLICIES || param_stride < 0)
        return SS_ERR_INVALID_ARG;
    if ((param_stride & 3) || (param_stride > 0 && param_stride < SS_ACTOR_PARAMS)) return SS_ERR_INVALID_ARG;
    if ((((uintptr_t)params | (uintptr_t)obs) & 15) || ((uintptr_t)act_out & 7)) return SS_ERR_INVALID_ARG;
    pipe::SegTable T{};
    T.n = n_segs;
    int64_t tiles[SS_LEAGUE_MAX_POLICIES];
    for (int s = 0; s < n_segs; ++s) {
        if (seg_rows_host[s] <= 0) return SS_ERR_INVALID_ARG;
        tiles[s] = (seg_rows_host[s] + TM - 1) / TM;
        T.row0[s + 1] = T.row0[s] + seg_rows_host[s];
        T.unit0[s + 1] = T.unit0[s] + tiles[s];
    }
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return SS_ERR_CUDA;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return SS_ERR_CUDA;
    const int64_t units = T.unit0[n_segs], rounds = (units + sms - 1) / sms;
    int grid = (int)((units + rounds - 1) / rounds);
    int ctas[SS_LEAGUE_MAX_POLICIES], given = n_segs;
    for (int s = 0; s < n_segs; ++s) ctas[s] = 1;
    while (given < grid) {
        int best = -1;                                        // the segment with the most tiles per CTA that can take one more
        for (int s = 0; s < n_segs; ++s)
            if (ctas[s] < tiles[s] && (best < 0 || tiles[s] * ctas[best] > tiles[best] * ctas[s])) best = s;
        if (best < 0) break;
        ++ctas[best];
        ++given;
    }
    for (int s = 0; s < n_segs; ++s) T.cta0[s + 1] = T.cta0[s] + ctas[s];
    FwdArgs A{};
    A.params = params; A.obs = obs; A.n = T.row0[n_segs]; A.group = A.n; A.act_out = act_out; A.param_stride = param_stride;
    if (cudaFuncSetAttribute(pipe::mlp_fwd_segments_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pipe::SMP_TOTAL) !=
        cudaSuccess)
        return SS_ERR_CUDA;
    A.early_weights = sslaunch::take_early_weights();
    if (sslaunch::launch(pipe::mlp_fwd_segments_kernel, dim3(given), dim3(pipe::NTH), pipe::SMP_TOTAL, (cudaStream_t)stream, A, T) !=
        cudaSuccess)
        return SS_ERR_CUDA;
    return cudaGetLastError() == cudaSuccess ? SS_OK : SS_ERR_CUDA;
}

extern "C" int ss_actor_forward_tc(const float *actor_params, const float *obs, float *act_out, int64_t n,
                                   float param_noise_sd, int64_t noise_group, float action_noise_sd,
                                   uint64_t seed, uint64_t counter, void *stream) {
    return ss_actor_forward_tc_signal(actor_params, obs, act_out, n, param_noise_sd, noise_group, action_noise_sd, seed, counter,
                                      nullptr, nullptr, nullptr, stream);
}

// The rollout tick as ONE kernel: actor forward on the players' observations, and in its output stage the env step of
// those very players (ss_env_pp.cuh) -- do_actions, game_tick, reward, auto-reset, next observation -- written straight
// into the replay ring's rows.  Same results, bit for bit, as ss_actor_forward_tc followed by ss_env_step_ring.
extern "C" int ss_actor_forward_step_tc(const float *actor_params, const float *obs, float *act_out, int64_t n_rows,
                                        float param_noise_sd, int64_t noise_group, float action_noise_sd, uint64_t seed,
                                        uint64_t counter, void *env_state, float *obs_next, float *obs_next2, float *reward_out,
                                        uint8_t *done_out, uint8_t *done_rows_out, uint8_t *winner_out, int reward_mode,
                                        int64_t tick_limit, int reset_mode, uint64_t env_seed, uint64_t env_counter,
                                        uint32_t *status, int flags, void *stream) {
    if (!actor_params || !obs || !act_out || n_rows <= 0 || (n_rows & 1) || param_noise_sd < 0.f || action_noise_sd < 0.f ||
        !env_state || !obs_next)
        return SS_ERR_INVALID_ARG;
    if (((uintptr_t)actor_params | (uintptr_t)obs | (uintptr_t)env_state | (uintptr_t)obs_next | (uintptr_t)obs_next2) & 15 ||
        ((uintptr_t)act_out & 7) || ((uintptr_t)reward_out & 3))
        return SS_ERR_INVALID_ARG;
    if (reward_mode != SS_REWARD_NONE && reward_mode != SS_REWARD_LOOKING && reward_mode != SS_REWARD_TERMINAL) return SS_ERR_INVALID_ARG;
    if (reset_mode != SS_RESET_FIXED && reset_mode != SS_RESET_RANDOM) return SS_ERR_INVALID_ARG;
    const bool noisy = param_noise_sd > 0.f;
    if (noisy && (noise_group <= 0 || noise_group % TM != 0)) return SS_ERR_INVALID_ARG;
    FwdArgs A{};
    A.params = actor_params; A.obs = obs; A.n = n_rows; A.group = noisy ? noise_group : n_rows;
    A.act_out = act_out; A.param_sd = param_noise_sd; A.action_sd = action_noise_sd; A.seed = seed; A.counter = counter;
    A.env_state = env_state; A.obs_next = (float4 *)obs_next; A.obs_next2 = (float4 *)obs_next2;
    A.reward_out = reward_mode != SS_REWARD_NONE ? reward_out : nullptr;
    A.done_out = done_out; A.winner_out = winner_out; A.done_rows_out = done_rows_out; A.env_status = status;
    A.env_stats = (status && (flags & SS_STEP_EPISODE_STATS)) ? reinterpret_cast<unsigned long long *>(status) + 1 : nullptr;
    if (A.env_stats && ((uintptr_t)status & 7)) return SS_ERR_INVALID_ARG;
    A.TP.seed = env_seed; A.TP.counter = env_counter; A.TP.tick_limit = tick_limit; A.TP.reward_mode = reward_mode;
    A.TP.auto_reset = 1; A.TP.reset_mode = reset_mode;
    return launch_fwd<NET_ACTOR, true>(A, stream);
}

extern "C" int ss_critic_forward_tc(const float *critic_params, const float *obs, const float *act, int64_t n,
                                    float *q_out, float *neg_dq_da_out, const float *reward, const uint8_t *done,
                                    float gamma, float *y_out, void *stream) {
    if (!critic_params || !obs || !act || n <= 0 || (!q_out && !neg_dq_da_out && !y_out)) return SS_ERR_INVALID_ARG;
    if (y_out && !reward) return SS_ERR_INVALID_ARG;
    if (((uintptr_t)critic_params | (uintptr_t)obs) & 15 || (((uintptr_t)act | (uintptr_t)neg_dq_da_out) & 7))
        return SS_ERR_INVALID_ARG;
    FwdArgs A{};
    A.params = critic_params; A.obs = obs; A.n = n; A.group = n;
    A.act_in = act; A.q_out = q_out; A.up_out = neg_dq_da_out; A.y_out = y_out; A.reward = reward; A.done = done;
    A.gamma = gamma;
    return launch_fwd<NET_CRITIC>(A, stream);
}

// a = actor(s) -> act_out, then critic(s, a) -> any of q_out / neg_dq_da_out / y_out, as ONE launch (mlp_fwd_pair_kernel).
// Same results, bit for bit, as ss_actor_forward_tc (no noise) followed by ss_critic_forward_tc.
extern "C" int ss_actor_critic_forward_tc(const float *actor_params, const float *critic_params, const float *obs, float *act_out,
                                          int64_t n, float *q_out, float *neg_dq_da_out, const float *reward, const uint8_t *done,
                                          float gamma, float *y_out, void *pair_mail, void *stream) {
    if (!actor_params || !critic_params || !obs || !act_out || !pair_mail || n <= 0 || (!q_out && !neg_dq_da_out && !y_out))
        return SS_ERR_INVALID_ARG;
    if (y_out && !reward) return SS_ERR_INVALID_ARG;
    if (((uintptr_t)actor_params | (uintptr_t)critic_params | (uintptr_t)obs) & 15 ||
        (((uintptr_t)act_out | (uintptr_t)neg_dq_da_out | (uintptr_t)pair_mail) & 7))
        return SS_ERR_INVALID_ARG;
    FwdArgs Aa{}, Ac{};
    Aa.params = actor_params; Aa.obs = obs; Aa.n = n; Aa.group = n; Aa.act_out = act_out; Aa.pair_mail = (int2 *)pair_mail;
    Ac.params = critic_params; Ac.obs = obs; Ac.n = n; Ac.group = n; Ac.act_in = act_out; Ac.pair_mail = (int2 *)pair_mail;
    Ac.q_out = q_out; Ac.up_out = neg_dq_da_out; Ac.y_out = y_out; Ac.reward = reward; Ac.done = done; Ac.gamma = gamma;
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return SS_ERR_CUDA;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return SS_ERR_CUDA;
    const int64_t units = (n + TM - 1) / TM;
    const int half = sms / 2;
    if (half < 1) return SS_ERR_CUDA;
    const int64_t prounds = (units + half - 1) / half;
    const int ga = (int)((units + prounds - 1) / prounds);      // the two roles split the tiles identically: same count
    if (cudaFuncSetAttribute(pipe::mlp_fwd_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pipe::SMP_TOTAL) !=
        cudaSuccess)
        return SS_ERR_CUDA;
    // (the critic role stages behind the wait when the launch directly follows the kernel that writes the critic)
    const int critic_late = sslaunch::pdl_mode() & sslaunch::kPdlPairCriticLate;
    Aa.early_weights = sslaunch::take_early_weights();
    Ac.early_weights = critic_late ? 0 : Aa.early_weights;
    if (sslaunch::launch(pipe::mlp_fwd_pair_kernel, dim3(2 * ga), dim3(pipe::NTH), pipe::SMP_TOTAL, (cudaStream_t)stream, Aa, Ac, ga) !=
        cudaSuccess)
        return SS_ERR_CUDA;
    return cudaGetLastError() == cudaSuccess ? SS_OK : SS_ERR_CUDA;
}
