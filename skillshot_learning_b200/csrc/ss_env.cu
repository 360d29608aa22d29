// ss_env.cu -- sm_100a kernels for the SkillshotGame hot path and their C ABI
// (include/skillshot_b200.h).  Compiled with -fmad=false (see ss_env_core.cuh).
//
// Data layout: four 16-byte SoA planes per env (header).  One thread owns one
// env: four coalesced 16-byte loads bring the whole game into registers, K ticks
// are played there, four 16-byte stores put it back.  Per tick a thread reads one
// float4 of actions and writes a float2 reward, two status bytes and (optionally)
// the 2x12 float observation, which is staged through shared memory so that each
// warp writes its 3 KB of observations as six fully coalesced 512-byte requests.
// The step is HBM-bound by design (SURVEY.md 8(d)): no tensor-core work here.
#include <cuda_runtime.h>
#include <stdint.h>
#include <atomic>
#include <stdlib.h>

#include "../../include/skillshot_b200.h"
#include "ss_env_core.cuh"
#include "ss_env_pp.cuh"
#include "ss_launch.cuh"
#include "ss_pool_blocks.cuh"

namespace {

using namespace ss;

constexpr int kBlock = 64;             // 2 warps: fine-grained CTAs balance small grids over 148 SMs
constexpr int kRowF4 = 7;              // 6 float4 of observation + 1 pad: conflict-free float4 smem rows

struct StatePlanes {
    double2 *rot;    // plane 0
    double2 *qrot;   // plane 1
    int4 *ia;        // plane 2
    int4 *ib;        // plane 3
};
__host__ __device__ inline StatePlanes planes_of(void *state, int64_t n) {
    char *b = (char *)state;
    return StatePlanes{(double2 *)b, (double2 *)(b + 16 * n), (int4 *)(b + 32 * n), (int4 *)(b + 48 * n)};
}

__device__ __forceinline__ void load_env(const StatePlanes &s, int64_t i, Env &e) {
    double2 r = s.rot[i], q = s.qrot[i];
    int4 a = s.ia[i], b = s.ib[i];
    unpack(e, r.x, r.y, q.x, q.y, Int4{a.x, a.y, a.z, a.w}, Int4{b.x, b.y, b.z, b.w});
}
__device__ __forceinline__ void store_env(const StatePlanes &s, int64_t i, const Env &e) {
    Int4 a, b;
    pack(e, a, b);
    s.rot[i] = make_double2(e.prot[0], e.prot[1]);
    s.qrot[i] = make_double2(e.qrot[0], e.qrot[1]);
    s.ia[i] = make_int4(a.x, a.y, a.z, a.w);
    s.ib[i] = make_int4(b.x, b.y, b.z, b.w);
}
__device__ __forceinline__ Speeds load_speeds(const void *speeds, int64_t n, int64_t i) {
    const char *b = (const char *)speeds;
    double2 a = ((const double2 *)b)[i];
    const double *p1 = (const double *)(b + 16 * n) + 2 * i;
    long long cm = ((const long long *)(b + 16 * n))[2 * i + 1];
    return Speeds{a.x, a.y, p1[0], (int)cm, 1.0f / (float)cm};
}

// fast_obs sink: the thread's row of the warp's shared-memory staging tile
struct SmemSink {
    float4 *row;
    __device__ __forceinline__ void put(int j, float a, float b, float c, float d) { row[j] = make_float4(a, b, c, d); }
};

// One finished game into the episode statistics (SS_STEP_EPISODE_STATS).  Kept out of line: it runs once per game,
// and inlined it cost the step kernels 30-40 registers.
__device__ __noinline__ void count_episode(unsigned long long *stats, int len, int winner, int tick_limit) {
    const int width = tick_limit > 0 ? (tick_limit + 63) / 64 : 32;
    atomicAdd(stats + 0, 1ull);
    atomicAdd(stats + (winner == 1 ? 1 : winner == 2 ? 2 : 3), 1ull);
    atomicAdd(stats + 4, (unsigned long long)len);
    atomicAdd(stats + 8 + min(63, len / width), 1ull);
}

struct StepArgs {
    void *state;
    int64_t n;
    const float4 *actions;
    float4 *obs_out;
    float2 *reward_out;
    uint8_t *done_out;
    uint8_t *winner_out;
    float4 *obs_out2;          // second copy of the observation (the replay ring's next segment), or NULL
    uint16_t *done_rows_out;   // terminal (hit) flag once per player row ([n][2] bytes, the replay ring's layout), or NULL
    const void *speeds;
    uint32_t *status;
    unsigned long long *stats;  // episode statistics (SS_STEP_EPISODE_STATS) or NULL
    uint8_t *packed_out;        // ss_env_step_packed: one byte per env and tick instead of reward / done / winner
    TickParams P;
    int n_ticks, obs_every_tick;
};

// OBS: write observations.  CARRY: keep sin/cos of the rotations in registers across
// ticks (fused ticks, observations, shaped rewards); !CARRY is the lean one-tick
// physics-only kernel.
template <bool OBS, bool CARRY, bool SPEEDS, int MINB = 1, bool STATS = false, bool PDL = false, int BLK = kBlock>
__global__ void __launch_bounds__(BLK, MINB) step_kernel(const StepArgs A) {
    __shared__ float4 tile[OBS ? BLK / 32 : 1][OBS ? 32 * kRowF4 : 1];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t i = (int64_t)blockIdx.x * BLK + threadIdx.x;
    const int64_t warp_base = i - lane;
    const bool active = i < A.n;
    const StatePlanes S = planes_of(A.state, A.n);

    // Programmatic dependent launch (one-tick physics launches, ss_env_step_ring): this grid may have been scheduled while
    // the previous kernel of the stream was still running; nothing of global memory is touched before that kernel has
    // completed.  A launch without the attribute passes straight through.
    if (PDL) asm volatile("griddepcontrol.wait;" ::: "memory");
    Env e;
    Speeds k = default_speeds();
    if (active) {
        load_env(S, i, e);
        if (SPEEDS) k = load_speeds(A.speeds, A.n, i);
    } else {
        reset_env(e, 50, 50, 200, 200);
    }
    if (PDL) asm volatile("griddepcontrol.launch_dependents;");     // the next launch may start its own prologue
    uint32_t status = 0;
    const bool write_reward = A.reward_out && A.P.reward_mode != SS_REWARD_NONE;
    Trig tr;
    if (CARRY) trig_of(e, tr);

    float4 a_next = make_float4(0.f, 0.f, 0.f, 0.f);
    if (active) a_next = __ldg(A.actions + i);
    for (int t = 0; t < A.n_ticks; ++t) {
        const int64_t row = (int64_t)t * A.n + i;
        const float4 a = a_next;
        if (active && t + 1 < A.n_ticks) a_next = __ldg(A.actions + row + A.n);   // prefetch: hide the load behind this tick
        const bool want_obs = OBS && (A.obs_every_tick || t == A.n_ticks - 1);
        float r[2];
        int done, winner;
        SmemSink sink{&tile[OBS ? warp : 0][OBS ? lane * kRowF4 : 0]};
        // a game that is over before the tick (no auto-reset) stays "done" and is not an episode end again
        const int ticks_before = !STATS ? 0 : (!e.live || (A.P.tick_limit > 0 && e.ticks >= A.P.tick_limit)) ? -1 : e.ticks;
        tick_env<OBS, CARRY>(e, a.x, a.y, a.z, a.w, k, A.P, (uint64_t)i, t, want_obs, status, tr, r, done, winner, sink);
        if (STATS && active && done && ticks_before >= 0)          // rare: a few atomics per finished game
            count_episode(A.stats, ticks_before + 1, winner, (int)A.P.tick_limit);
        if (active) {
            if (write_reward) A.reward_out[row] = make_float2(r[0], r[1]);
            if (A.done_out) A.done_out[row] = (uint8_t)done;
            // the replay ring's flag masks the TD bootstrap: a hit is a true termination, a tick-limit restart is not
            if (A.done_rows_out) A.done_rows_out[row] = (uint16_t)(winner ? 0x0101 : 0);
            if (A.winner_out) A.winner_out[row] = (uint8_t)winner;
        }
        if (OBS && want_obs) {
            // the warp's 32 x 24 floats are staged in shared memory (SmemSink); write them as
            // 6 coalesced 512-byte requests
            __syncwarp();
            const int64_t tick_off = A.obs_every_tick ? (int64_t)t * A.n * 6 : 0;
            float4 *dst = A.obs_out + tick_off + warp_base * 6;
#pragma unroll
            for (int j = 0; j < 6; ++j) {
                int idx = j * 32 + lane, rw = idx / 6, cl = idx - rw * 6;
                if (warp_base + rw < A.n) {
                    const float4 v = tile[warp][rw * kRowF4 + cl];
                    dst[idx] = v;
                    if (A.obs_out2) A.obs_out2[warp_base * 6 + idx] = v;
                }
            }
            __syncwarp();
        }
    }
    if (active) store_env(S, i, e);
    if (status && A.status) atomicOr(A.status, status);
}

// ---------------------------------------------------------------------------------------------------------------------
// step_pp_kernel -- the fused physics-only step with ONE THREAD PER PLAYER.
//
// Lanes 2i and 2i+1 of a warp are players 1 and 2 of env i: each lane owns its player (position, rotation) and that
// player's projectile, the env's three scalars (ticks, live, winner) are replicated in both lanes.  Everything a tick
// does is per player except the hit test, which needs the OTHER player's projectile: one __shfl_xor of the packed
// (x, y, valid) word, and one warp ballot that gives both lanes the pair's two hit bits (SkillshotGame.check_collision's
// "player 1 first, first hit wins" is then a bit test).  Compared with one thread per env (step_kernel) a 65,536-env
// launch has twice the warps (6.9 instead of 3.5 per scheduler, which was latency-bound: ncu round 1, 36 % of cycles
// without an eligible warp) and each thread half the dependent chain.
//
// The arithmetic is the core's (ss_env_core.cuh), restated without the conversion instructions, which ncu and
// tools/op_probe.cu showed to be the scarce pipe (I2F.F64 / F2I.F64 issue once per 8-9 cycles and take 18-19, a DADD once
// per 2 and 8):
//   int -> double   (2^52 + x) - 2^52 with x placed in the low word of 2^52's bit pattern: exact for 0 <= x < 2^32
//   double -> int   low word of v + 1.5 * 2^52: the add rounds v to an integer, half-to-even, exactly Python's
//                   int(round(v)) and cvt.rni (|v| < 2^31)
// so positions stay integers in registers and both conversions are one DADD.  The float32 -> float64 conversion of the
// two actions stays (2 per lane and tick).  The clip keeps the reference's NaN behaviour (a NaN falls through both
// compares, Player.py:36-37, 60-61): min.NaN / max.NaN.  Where the reference raises (int(round(nan)), Player.py:63,
// Projectile.py:40) SS_STATUS_NAN is set from ONE unordered compare of the two candidate x coordinates per tick.
//
// Physics-only: reward modes none / terminal, reference speed constants, no observations, no episode statistics; the
// other combinations stay on step_kernel.  Same HBM layout, same outputs, bit-identical results (tests: every fused
// physics test of tests/test_gpu_env_parity.py runs through it, bench shape included).
constexpr int kBlockPP = 64;        // the per-player observation kernel's CTA, and the smallest of step_pp_kernel's (pp_block_for)
constexpr double kRound = 6755399441055744.0;      // 1.5 * 2^52

// A position coordinate x (0 ... 250) is carried as the double kRound + x: its low word IS the integer (hit test, bounds,
// packing read it for free), kRound + x - kRound is the exact double (one DADD), and rounding a candidate v to the nearest
// integer, half to even, is v + kRound, already in this form.  A commit replaces the low word only (the high word is
// 0x43380000 for every committed value).
__device__ __forceinline__ double coord(int x) { return __hiloint2double(0x43380000, x); }
__device__ __forceinline__ int icoord(double w) { return __double2loint(w); }
__device__ __forceinline__ double with_low(double w, int lo) { return __hiloint2double(__double2hiint(w), lo); }

struct Lane {
    double rot;                     // Player.rotation (Projectile.rotation is parked in shared memory: only a spawn writes it)
    double s3, c3;                  // sin / cos of rot times Player.speed_move (3)
    double qs5, qc5;                // sin / cos of the projectile's rotation times Projectile.speed_move (5)
    double wx, wy, ux, uy;          // player and projectile position in coord() form
    int cd, age, valid, live, winner, ticks;
};

__device__ __forceinline__ float clip_unit_nan(float v) {        // Player.py:36-37, 60-61; NaN falls through
    float r;
    asm("max.NaN.f32 %0, %1, 0fBF800000;" : "=f"(r) : "f"(v));
    asm("min.NaN.f32 %0, %1, 0f3F800000;" : "=f"(r) : "f"(r));
    return r;
}
__device__ __forceinline__ bool either_nan(double a, double b) {
    int p;
    asm("{ .reg .pred q; setp.nan.f64 q, %1, %2; selp.s32 %0, 1, 0, q; }" : "=r"(p) : "d"(a), "d"(b));
    return p != 0;
}

__device__ __forceinline__ void lane_reset(Lane &L, double *qrot, int x, int y) {      // SkillshotGame.__init__, this player's half
    L.wx = coord(x); L.wy = coord(y); L.rot = 0.0;
    L.ux = coord(0); L.uy = coord(0); *qrot = 0.0; L.cd = 0; L.age = 0; L.valid = 0;
    L.ticks = 0; L.live = 1; L.winner = 0;
    L.s3 = 0.0; L.c3 = 3.0; L.qs5 = 0.0; L.qc5 = 5.0;                                   // sin 0 = 0, cos 0 = 1
}

struct LaneIo {                     // per-lane cursor into the per-tick tensors: ONE 32-bit element index, advanced once per tick
    uint32_t idx;                   // tick * 2n + global lane: this lane's float2 action, its float reward; idx >> 1 = its env's flag byte
    uint32_t n2;                    // 2n: lanes per tick
    const float2 *actions;
    float *reward;
    uint8_t *flags;                 // done_out (player-1 lanes) or winner_out (player-2 lanes)
};

// sin / cos of the player's rotation, computed one tick AHEAD of its use.  rot(t) = rot(t-1) + clip(look(t)) * 0.25
// depends on the actions alone (Player.py:33-39), not on anything the tick computes, so the longest dependent chain of a
// tick -- argument reduction and the two polynomial evaluations, ~150 cycles -- is taken off the tick's critical path: tick
// t runs beside the sin / cos of tick t + 1, two independent instruction streams the scheduler interleaves.  Only a game
// reset (rotation back to 0) invalidates the speculation; the reset path redoes it.
struct Turn {
    double rot, s, c;               // post-turn rotation of a tick and its sin / cos
};

template <bool CHECKED>
__device__ __forceinline__ void turn_from(Turn &out, double rot_before, float look) {
    out.rot = fma((double)clip_unit_nan(look), 0.25, rot_before);    // rot + angle * 0.25: the product is exact (Player.py:39)
    if (CHECKED) sincos_d(out.rot, &out.s, &out.c);
    else sincos_d_unchecked(out.rot, &out.s, &out.c);
}

// What a tick writes: OUT_FLAGS = done / winner bytes (+ zero rewards when asked), OUT_TERMINAL = those + the +1 / -1 / 0
// reward (readme.md:10), OUT_PACKED = one byte per env {bit 0 done, bits 1-2 winner_id, bit 3 "the hit happened on this
// tick"} from which the other three follow (ss_env_step_packed: the host-buffer path moves 1 byte per env-step, not 10).
enum { OUT_FLAGS = 0, OUT_TERMINAL = 1, OUT_PACKED = 2 };

// One tick of one player.  `now` = this tick's post-turn rotation with its sin / cos (computed during the previous tick),
// `next` = the next tick's, computed here from `look_next`.  CHECKED: sin / cos with the |rot| < 1e5 range check.
template <int TERMINAL, bool CHECKED>
__device__ __forceinline__ void lane_tick(Lane &L, double *qrot, const float move, const float look_next, const Turn &now, Turn &next,
                                          const StepArgs &A, LaneIo &io, int lane, int P, int64_t env, int tick, int limit,
                                          bool write_zero, bool &nan_seen) {
    turn_from<CHECKED>(next, now.rot, look_next);
    // ---- do_actions (SkillshotLearner.py:206-213): move with the rotation BEFORE the turn, turn, shoot ----
    const double speed = (double)clip_unit_nan(move);
    const double vx = sub(sub(L.wx, kRound), mul(L.s3, speed));       // Player.py:63
    const double vy = sub(sub(L.wy, kRound), mul(L.c3, speed));       // Player.py:64
    const double cx = add(vx, kRound), cy = add(vy, kRound);          // int(round(.)), in coord() form
    const bool ok = (unsigned)icoord(cx) <= (unsigned)(kBoard - kPlayerSize) &&
                    (unsigned)icoord(cy) <= (unsigned)(kBoard - kPlayerSize);
    L.wx = with_low(L.wx, ok ? icoord(cx) : icoord(L.wx));            // Player.py:66-68: both or neither
    L.wy = with_low(L.wy, ok ? icoord(cy) : icoord(L.wy));
    L.rot = now.rot;
    L.s3 = mul(now.s, 3.0); L.c3 = mul(now.c, 3.0);
    if (L.cd <= 0) {                                                  // Player.move_shoot_projectile, Player.py:78-89
        L.ux = with_low(L.ux, icoord(L.wx)); L.uy = with_low(L.uy, icoord(L.wy));
        *qrot = now.rot;
        L.qs5 = mul(now.s, 5.0); L.qc5 = mul(now.c, 5.0);
        L.valid = 1; L.cd = 15; L.age = 0;
    }
    // ---- game_tick (SkillshotGame.py:115-122), gated on game_live ----
    const int lv = L.live;
    const double zx = sub(sub(L.ux, kRound), L.qs5);                  // Projectile.py:40
    const double zy = sub(sub(L.uy, kRound), L.qc5);                  // Projectile.py:41
    if (either_nan(vx, zx)) nan_seen = true;                          // int(round(nan)) raises
    const double dx = add(zx, kRound), dy = add(zy, kRound);
    const bool inb = (unsigned)icoord(dx) <= (unsigned)(kBoard - kProjSize) &&
                     (unsigned)icoord(dy) <= (unsigned)(kBoard - kProjSize);
    const bool fly = lv && L.valid && inb;                            // Projectile.py:43-47
    L.ux = with_low(L.ux, fly ? icoord(dx) : icoord(L.ux));
    L.uy = with_low(L.uy, fly ? icoord(dy) : icoord(L.uy));
    L.valid = lv ? (int)fly : L.valid;
    L.ticks += lv; L.cd -= lv; L.age += lv;                           // SkillshotGame.py:118, Projectile.py:52-53
    // check_collision (SkillshotGame.py:58-94): my player against the OTHER player's projectile
    const uint32_t mine = (uint32_t)icoord(L.ux) | ((uint32_t)icoord(L.uy) << 8) | ((uint32_t)L.valid << 16);
    const uint32_t theirs = __shfl_xor_sync(0xffffffffu, mine, 1);
    const int jx = theirs & 255, jy = (theirs >> 8) & 255, px = icoord(L.wx), py = icoord(L.wy);
    const bool in_x = (unsigned)(jx + kProjSize - px) <= (unsigned)kPlayerSize || (unsigned)(jx - px) <= (unsigned)kPlayerSize;
    const bool in_y = (unsigned)(jy - py) <= (unsigned)kPlayerSize || (unsigned)(jy - kProjSize - py) <= (unsigned)kPlayerSize;  // :72 minus
    const bool hit = lv && (theirs >> 16) && in_x && in_y;
    const uint32_t pair = (__ballot_sync(0xffffffffu, hit) >> (lane & 30)) & 3u;     // bit 0: player 1 hit, bit 1: player 2 hit
    float r = 0.f;
    if (pair) {                                                       // the pair with player 1 first; the first hit breaks
        L.winner = (pair & 1u) ? 1 : 2;                               // winner_id = the player that was HIT (:77)
        L.live = 0;
        r = (L.winner - 1 == P) ? -1.f : 1.f;                         // readme.md:10: -1 for the hit player, +1 for the shooter
    }
    const bool done = !L.live || L.ticks >= limit;
    if (TERMINAL == OUT_PACKED) {
        if (!P) io.flags[io.idx >> 1] = (uint8_t)((int)done | (L.winner << 1) | (pair ? 8 : 0));
    } else {
        if (TERMINAL == OUT_TERMINAL) io.reward[io.idx] = r;
        else if (write_zero) io.reward[io.idx] = 0.f;
        io.flags[io.idx >> 1] = (uint8_t)(P ? L.winner : (int)done);
    }
    io.idx += io.n2;
    if (A.P.auto_reset && done) {                                     // game_reset (SkillshotGame.py:168-169)
        int x = P ? 200 : 50, y = x;
        if (A.P.reset_mode == SS_RESET_RANDOM) {
            const uint64_t ctr = A.P.counter + (uint64_t)tick;
            const U4 u = philox4x32_10(U4{(uint32_t)env, (uint32_t)((uint64_t)env >> 32), (uint32_t)ctr, (uint32_t)(ctr >> 32)},
                                       (uint32_t)A.P.seed, (uint32_t)(A.P.seed >> 32));
            x = rand_coord(P ? u.z : u.x); y = rand_coord(P ? u.w : u.y);
        }
        lane_reset(L, qrot, x, y);
        turn_from<CHECKED>(next, 0.0, look_next);                     // the next tick turns from rotation 0
    }
}

// The action stream of step_pp_kernel goes through a ring of kRingD slots per lane in shared memory: slot s of a lane is
// ring[s * BLK + threadIdx.x], so a warp's 32 float2 of one slot are 256 contiguous bytes (no bank conflicts).  Each lane
// copies the 8 bytes it will read itself with cp.async and waits only on its own copies (cp.async.wait_group): no barrier,
// no other thread involved.  The copy of tick k is issued during tick k - kRingD + 1 and first read during tick k - 1,
// kRingD - 2 ticks (~250 cycles of a warp's own time each) ahead of its use.  8 slots measured as fast as 16 at 256 and
// 1,024 ticks per launch and faster at 32 (the prologue waits for its first copies once per launch), in half the shared
// memory (profiles/r13_step_ring_step0.txt).
constexpr int kRingD = 8;
static_assert((kRingD & (kRingD - 1)) == 0 && kRingD >= 4, "kRingD is a power of two >= 4");

__device__ __forceinline__ void ring_copy(float2 *dst, const float2 *src, bool valid) {   // 8 bytes; zero-filled when !valid
    const uint32_t d = (uint32_t)__cvta_generic_to_shared(dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;\n" ::"r"(d), "l"(src), "r"(valid ? 8 : 0) : "memory");
    asm volatile("cp.async.commit_group;\n" ::: "memory");
}
__device__ __forceinline__ float2 ring_read(const float2 *slot) {       // after this lane's copies up to `slot` have landed
    asm volatile("cp.async.wait_group %0;\n" ::"n"(kRingD - 2) : "memory");
    return *slot;
}

template <int TERMINAL, bool CHECKED, int BLK>
__device__ __forceinline__ void lane_loop(Lane &L, double *qrot, const StepArgs &A, LaneIo &io, float2 *ring, int lane, int P,
                                          int64_t env, bool &nan_seen) {
    const int limit = A.P.tick_limit > 0 ? (int)min((int64_t)0x7fffffff, A.P.tick_limit) : 0x7fffffff;
    const bool write_zero = TERMINAL == OUT_FLAGS && A.reward_out && A.P.reward_mode != SS_REWARD_NONE;
    const int T = A.n_ticks;
    // tick t needs move(t) and look(t + 1): the action of tick t + 1 is consumed during tick t (its look half now, its
    // move half one tick later).  The ring holds ticks t ... t + kRingD - 1 during tick t.  Ticks >= T are zero-filled
    // copies from index 0 (a valid address), so every lane commits one group per tick and no tick branches on the end.
    // src is the element index of the next tick to copy; it is only dereferenced while that tick is < T, where it is below
    // 2n * T (the launch checks that 2n * (n_ticks + 2) fits 32 bits).
    uint32_t src = io.idx;
#pragma unroll
    for (int k = 0; k < kRingD - 1; ++k, src += io.n2) ring_copy(ring + k * BLK, io.actions + (k < T ? src : 0u), k < T);
    float2 a0 = ring_read(ring);
    Turn ta, tb;
    turn_from<CHECKED>(ta, L.rot, a0.y);
    float move = a0.x;
    // Tick t refills the slot of tick t - 1 with tick t + kRingD - 1.  That slot was last read by the shared-memory load
    // of tick t - 2, whose two values were consumed by arithmetic before tick t began, so the load has completed and the
    // asynchronous write cannot overtake it.  Its own slot t + 1 is then read after waiting for all but the kRingD - 2
    // newest groups, which leaves the copies of ticks 0 ... t + 1 landed.
    for (int t = 0; t < T; t += 2) {
        ring_copy(ring + ((t - 1) & (kRingD - 1)) * BLK, io.actions + (t + kRingD - 1 < T ? src : 0u), t + kRingD - 1 < T);
        src += io.n2;
        float2 q = ring_read(ring + ((t + 1) & (kRingD - 1)) * BLK);
        lane_tick<TERMINAL, CHECKED>(L, qrot, move, q.y, ta, tb, A, io, lane, P, env, t, limit, write_zero, nan_seen);
        move = q.x;
        if (t + 1 < T) {
            ring_copy(ring + (t & (kRingD - 1)) * BLK, io.actions + (t + kRingD < T ? src : 0u), t + kRingD < T);
            src += io.n2;
            q = ring_read(ring + ((t + 2) & (kRingD - 1)) * BLK);
            lane_tick<TERMINAL, CHECKED>(L, qrot, move, q.y, tb, ta, A, io, lane, P, env, t + 1, limit, write_zero, nan_seen);
            move = q.x;
        }
    }
    asm volatile("cp.async.wait_all;\n" ::: "memory");              // the zero-fill copies past the end
}

// TERMINAL: one of OUT_FLAGS / OUT_TERMINAL / OUT_PACKED.
// BLK: threads per CTA, 896 / BLK CTAs per SM (always 28 warps of 72 registers: the whole register file).  The work is the
// same whatever BLK; what changes is how the SM's 28 warps are made up.  As ONE CTA (BLK = 896) they are dealt to the four
// schedulers seven each; as 14 CTAs of two warps the launch measured 7.6 % slower at 65,536 envs (200.4 vs 215.7 us for 256
// ticks, profiles/r2_step_blk_sweep.txt; CTAs of 32 / 128 / 224 threads were like 64, 448 in between), with ncu showing
// 22.8 active warps per SM on average out of 28 -- warps finishing at different times.  (Neither start-up phase offsets
// between the warps nor a CTA barrier every 16 / 64 ticks helped: profiles/r2_step_stagger_experiment.txt.)
// pp_block_for() picks BLK from the env count.
template <int TERMINAL, int BLK = kBlockPP>
__global__ void __launch_bounds__(BLK, 896 / BLK) step_pp_kernel(const StepArgs A) {
    constexpr int kBlockPP = BLK;
    __shared__ double qrot_sh[kBlockPP];
    const int lane = threadIdx.x & 31, P = lane & 1;
    // global lane = 2 * env + player.  Lanes past the end replay the last env (same inputs, same values stored twice):
    // no lane of the warp is ever inactive, so the shuffle and the ballot need no guards and the loop no predicates.
    int64_t gl = (int64_t)blockIdx.x * kBlockPP + threadIdx.x;
    gl = min(gl, 2 * A.n - 2 + P);
    const int64_t env = gl >> 1;
    char *const base = (char *)A.state;
    double *const qrot = &qrot_sh[threadIdx.x];
    Lane L;
    {
        L.rot = ((const double *)base)[gl];                               // plane 0 is double2 per env: this lane's half
        *qrot = ((const double *)(base + 16 * A.n))[gl];
        const int4 a = ((const int4 *)(base + 32 * A.n))[env], b = ((const int4 *)(base + 48 * A.n))[env];
        const uint32_t pp = (uint32_t)a.x >> (16 * P), qq = (uint32_t)a.y >> (16 * P), f = (uint32_t)b.w;
        L.wx = coord(pp & 255); L.wy = coord((pp >> 8) & 255); L.ux = coord(qq & 255); L.uy = coord((qq >> 8) & 255);
        L.cd = P ? a.w : a.z; L.age = P ? b.y : b.x; L.ticks = b.z;
        L.valid = (f >> P) & 1; L.live = (f >> 2) & 1; L.winner = (f >> 4) & 3;
        double s, c;
        sincos_d(L.rot, &s, &c);
        L.s3 = mul(s, 3.0); L.c3 = mul(c, 3.0);
        sincos_d(*qrot, &s, &c);
        L.qs5 = mul(s, 5.0); L.qc5 = mul(c, 5.0);
    }
    bool nan_seen = false;
    LaneIo io;
    io.idx = (uint32_t)gl; io.n2 = (uint32_t)(2 * A.n);               // (the launch checks that 2n * (n_ticks + 2) fits 32 bits)
    io.actions = (const float2 *)A.actions;
    io.reward = (float *)A.reward_out;
    io.flags = TERMINAL == OUT_PACKED ? A.packed_out : (P ? A.winner_out : A.done_out);
    // A rotation moves by at most 0.25 per tick and a reset zeroes it, so |rot| + 0.25 * n_ticks < 1e5 at the start keeps
    // every rotation of this launch inside the range of the fast sin / cos: the per-tick range check (and the basic-block
    // boundary it puts in the middle of the tick) then goes.  Otherwise (400,000 ticks of one-sided turning without a
    // reset, or a NaN) the warp runs the checked loop.
    const bool in_range = fabs(L.rot) + 0.25 * (double)A.n_ticks + 1.0 < 1.0e5;
    extern __shared__ float2 ring_sh[];                                 // kRingD * BLK float2: the action ring (lane_loop)
    float2 *const ring = ring_sh + threadIdx.x;
    if (__all_sync(0xffffffffu, in_range)) lane_loop<TERMINAL, false, BLK>(L, qrot, A, io, ring, lane, P, env, nan_seen);
    else lane_loop<TERMINAL, true, BLK>(L, qrot, A, io, ring, lane, P, env, nan_seen);
    // the partner's valid bit for the env's flag word
    const int v_other = __shfl_xor_sync(0xffffffffu, L.valid, 1);
    ((double *)base)[gl] = L.rot;
    ((double *)(base + 16 * A.n))[gl] = *qrot;
    char *ia = base + 32 * A.n + env * 16, *ib = base + 48 * A.n + env * 16;
    ((uint16_t *)ia)[P] = (uint16_t)(icoord(L.wx) | (icoord(L.wy) << 8));
    ((uint16_t *)ia)[2 + P] = (uint16_t)(icoord(L.ux) | (icoord(L.uy) << 8));
    ((int *)ia)[2 + P] = L.cd;
    ((int *)ib)[P] = L.age;
    if (!P) ((int2 *)ib)[1] = make_int2(L.ticks, L.valid | (v_other << 1) | (L.live << 2) | (L.winner << 4));
    if (nan_seen && A.status) atomicOr(A.status, kStatusNaN);
}

// ---------------------------------------------------------------------------------------------------------------------
// step_pp_obs_kernel -- ONE tick with observations, one thread per player (ss_env_pp.cuh): the rollout's env step.
// Each lane loads its player's half of the state, plays the tick, and writes its reward, its 12-float observation (three
// float4, staged through shared memory so that a warp's 1,536 bytes leave as three fully coalesced 512-byte requests,
// to both copies when the replay ring wants two), its terminal byte; the env's done / winner bytes come from the two
// lanes of the pair.  Bit-identical to step_kernel<OBS = true> (the golden lockstep tests run through this kernel).
//
// The body is templated on a ROW RULE: which row of which buffer a lane reads its action from and writes its outputs to.
//   SelfPlayRows (ss_env_step_ring): row = global lane, every output in the caller's [n][2] rows.
//   PoolRows (ss_env_step_pool): the training-against-a-pool layout of the header.  Env i < S is
//     self-play (rows 2i + p of the learner rows); in pool env j >= S the learner's player is learner row 2S + (j - S) and
//     the frozen opponent's player is row j - S of the opponent rows.  Opponent k owns the b consecutive pool envs from
//     S + k b, the learner being player 1 in the first b / 2 of them.  An opponent lane writes only its observation (to the
//     opponent rows); reward and terminal flag are the learner's alone.  A warp's learner rows and its opponent rows are
//     each one contiguous run, so the observations still leave through the shared-memory tile as coalesced stores.
//   BlockPoolRows (ss_env_step_pool_blocks): PoolRows with one block size per opponent.  Opponent k owns the pool envs
//     from S + start[k] to S + start[k + 1], the learner being player 1 in the first half of them; the rows are PoolRows'.
//     The lane finds its block by a 6-step search of the table, a kernel parameter that the search reads in place from
//     the parameter bank (LDC with a register offset; no copy to the stack, profiles/r7_pool_blocks_ptxas.txt).  Marking
//     the parameter __grid_constant__ would change the code of the PoolRows instantiations, so it is not marked.
struct SelfPlayRows {
    static constexpr bool kPool = false;
};
struct PoolRows {
    static constexpr bool kPool = true, kBlocks = false;
    int64_t S, b;                       // self-play envs; pool envs per opponent (even, >= 2)
    const float2 *opp_actions;          // [M] opponent rows
    float4 *opp_obs;                    // [M][3]
    unsigned long long *pool_stats;     // [K][8] or NULL
};
struct BlockPoolRows {
    static constexpr bool kPool = true, kBlocks = true;
    int64_t S;
    const float2 *opp_actions;
    float4 *opp_obs;
    unsigned long long *pool_stats;
    int start[SS_LEAGUE_MAX_POLICIES + 1];   // B_0 = 0 .. B_K = M, then M up to entry 64 (M < 2^31)
};

// R.S and R.start from the table opp_envs [K] (NULL: M / K each); false: the table is invalid (ss_pool_blocks.cuh) or
// M >= 2^31.  M = 0 takes no table (every env is self-play).
bool pool_block_table(int64_t n, int64_t M, int K, const int64_t *opp_envs, BlockPoolRows &R) {
    int64_t start[SS_LEAGUE_MAX_POLICIES + 1];
    R.S = n - M;
    if (M == 0) return !opp_envs;
    if (M > 0x7fffffff || !sspool::block_starts(M, K, opp_envs, start)) return false;
    for (int k = 0; k <= SS_LEAGUE_MAX_POLICIES; ++k) R.start[k] = (int)(k <= K ? start[k] : M);
    return true;
}

// the block of pool env S + j (0 <= j < M) and the learner's player in it
__device__ __forceinline__ int pool_block_of(const BlockPoolRows &R, int j, int &learner_player) {
    int k = 0;
#pragma unroll
    for (int s = SS_LEAGUE_MAX_POLICIES / 2; s >= 1; s >>= 1)
        if (R.start[k + s] <= j) k += s;
    const int b0 = R.start[k];
    learner_player = j - b0 >= ((R.start[k + 1] - b0) >> 1) ? 1 : 0;
    return k;
}

// One finished pool game into its opponent's counters {episodes, learner wins, learner losses, tick-limit endings, ticks}.
// winner_id is the player that was HIT.  Out of line for the reason count_episode is.
__device__ __noinline__ void count_pool_game(unsigned long long *c, int len, int winner, int learner_player) {
    atomicAdd(c + 0, 1ull);
    atomicAdd(c + (winner == 0 ? 3 : winner == learner_player + 1 ? 2 : 1), 1ull);
    atomicAdd(c + 4, (unsigned long long)len);
}

template <bool STATS, class Rows>
__global__ void __launch_bounds__(kBlockPP) step_pp_obs_kernel(const StepArgs A, const Rows R) {
    __shared__ float4 tile[kBlockPP / 32][96];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, P = lane & 1;
    const int64_t g0 = (int64_t)blockIdx.x * kBlockPP + threadIdx.x;
    const int64_t last = 2 * A.n - 2 + P;
    const bool active = g0 <= last;
    const int64_t gl = active ? g0 : last;            // lanes past the end replay the last env and store nothing
    const int64_t env = gl >> 1;
    // ss_launch.cuh: in the rollout loop this grid is placed while the forward kernel's last CTAs finish, and waits here
    sslaunch::griddep_wait();
    sslaunch::griddep_launch();
    bool learner = true;                              // this lane's row is a learner row (else an opponent row)
    int64_t row = gl, block = 0;
    int learner_player = 0;
    if constexpr (Rows::kPool) {
        if (env >= R.S) {
            const int64_t j = env - R.S;
            if constexpr (Rows::kBlocks) {
                block = pool_block_of(R, (int)j, learner_player);
            } else {
                block = j / R.b;
                learner_player = j - block * R.b >= (R.b >> 1) ? 1 : 0;
            }
            learner = P == learner_player;
            row = learner ? 2 * R.S + j : j;
        }
    }
    sspp::LaneState L;
    sspp::lane_load((const char *)A.state, A.n, gl, L);
    const float2 *act = (const float2 *)A.actions;
    if constexpr (Rows::kPool) {
        if (!learner) act = R.opp_actions;
    }
    const float2 a = __ldg(act + row);
    uint32_t status = 0;
    sspp::LaneTrig T;
    sspp::lane_trig(L, T);
    sspp::LaneTickOut out;
    sspp::lane_obs_tick(L, T, a.x, a.y, A.P, (uint64_t)env, A.P.counter, lane, P, status, out);
    const int v_other = __shfl_xor_sync(0xffffffffu, L.valid, 1);
    if (active) {
        sspp::lane_store((char *)A.state, A.n, gl, L, v_other);
        if (learner && A.reward_out && A.P.reward_mode != SS_REWARD_NONE) ((float *)A.reward_out)[row] = out.reward;
        uint8_t *flag = P ? A.winner_out : A.done_out;
        if (flag) flag[env] = (uint8_t)(P ? out.winner : out.done);
        if (learner && A.done_rows_out) ((uint8_t *)A.done_rows_out)[row] = out.winner ? 1 : 0;
        if (STATS && !P && out.episode_len >= 0) count_episode(A.stats, out.episode_len, out.winner, (int)A.P.tick_limit);
        if constexpr (Rows::kPool) {
            if (!P && R.pool_stats && env >= R.S && out.episode_len >= 0)
                count_pool_game(R.pool_stats + block * 8, out.episode_len, out.winner, learner_player);
        }
    }
    if constexpr (Rows::kPool) {
        // the warp's learner lanes (rows l0 ...) take tile slots [0, nl), its opponent lanes (rows o0 ...) the next no slots
        const unsigned lmask = __ballot_sync(0xffffffffu, active && learner), omask = __ballot_sync(0xffffffffu, active && !learner);
        const unsigned below = (1u << lane) - 1u;
        const int nl = __popc(lmask), no = __popc(omask);
        const int64_t l0 = __shfl_sync(0xffffffffu, row, lmask ? __ffs(lmask) - 1 : 0);
        const int64_t o0 = __shfl_sync(0xffffffffu, row, omask ? __ffs(omask) - 1 : 0);
        const int slot = learner ? __popc(lmask & below) : nl + __popc(omask & below);
        if (active) {
#pragma unroll
            for (int j = 0; j < 3; ++j) tile[warp][slot * 3 + j] = out.obs[j];
        }
        __syncwarp();
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            const int idx = j * 32 + lane;
            if (idx < 3 * nl) {
                const float4 v = tile[warp][idx];
                A.obs_out[l0 * 3 + idx] = v;
                if (A.obs_out2) A.obs_out2[l0 * 3 + idx] = v;
            } else if (idx < 3 * (nl + no)) {
                R.opp_obs[o0 * 3 + (idx - 3 * nl)] = tile[warp][idx];
            }
        }
    } else {
        // observations: lane's three float4 -> tile -> three coalesced stores per warp and copy
#pragma unroll
        for (int j = 0; j < 3; ++j) tile[warp][lane * 3 + j] = out.obs[j];
        __syncwarp();
        const int64_t warp_base = (g0 - lane) * 3;                        // in float4
        const int64_t total = 2 * A.n * 3;
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            const int64_t idx = warp_base + j * 32 + lane;
            if (idx < total) {
                const float4 v = tile[warp][j * 32 + lane];
                A.obs_out[idx] = v;
                if (A.obs_out2) A.obs_out2[idx] = v;
            }
        }
    }
    if (status && A.status) atomicOr(A.status, status);
}

// pool_restart_kernel -- ss_pool_restart: every pool env starts a new game, one thread per player of the pool envs.  The
// start state is the auto-reset of lane_obs_tick under Philox counter (env, counter); the observation is the one an
// auto-reset tick writes for it (the post-reset view, sin 0 and cos 1), to the learner's or the opponent's row of the
// block layout in R.  No game ended, so nothing is counted.
__global__ void __launch_bounds__(kBlockPP) pool_restart_kernel(void *state, int64_t n, float4 *obs, int reset_mode, uint64_t seed,
                                                                uint64_t counter, const __grid_constant__ BlockPoolRows R) {
    const int64_t g = (int64_t)blockIdx.x * kBlockPP + threadIdx.x;
    if (g >= 2 * (n - R.S)) return;
    const int P = (int)(g & 1), j = (int)(g >> 1);
    const int64_t env = R.S + j;
    int learner_player;
    pool_block_of(R, j, learner_player);
    sspp::LaneState L;
    int ox, oy;
    sspp::lane_reset(L, P, (uint64_t)env, counter, reset_mode, seed, ox, oy);
    sspp::lane_store((char *)state, n, 2 * env + P, L, 0);
    const sspp::LaneView v = sspp::lane_view(L, ox, oy, 0.0, 1.0, 0.0, 1.0);
    float4 o[3];
    sspp::lane_obs(L, v, o);
    float4 *dst = P == learner_player ? obs + (2 * R.S + j) * 3 : R.opp_obs + (int64_t)j * 3;
#pragma unroll
    for (int q = 0; q < 3; ++q) dst[q] = o[q];
}


// ---------------------------------------------------------------------------------------------------------------------
// step_pp_tiles_kernel -- the rollout's env step running BESIDE the actor forward kernel that produces its actions.
// The forward kernel (ss_mlp_tc.cu) bumps tile_ready[tile] once per output warp when a 128-row tile's actions are in
// memory; this kernel, launched on a second stream, walks the tiles in the order the forward kernel's CTAs complete them
// (same even split of tiles over the same number of CTAs), waits for a tile's four arrivals and plays the tick of its 128
// players -- so the env step costs no time of its own: it ends a few microseconds after the forward kernel does.
// One WARP per CTA, at most 64 registers and NO shared memory, so that it fits beside the forward kernel's CTA on every SM.
// That CTA owns 222 KB of shared memory and 9 warps of 168 registers, and registers are per SM SUB-PARTITION (4 x 16 K): the
// partition that holds three of its warps has 256 registers left, the others 5.6 K each -- room for two 64-register warps
// per partition, six per SM, but not for a multi-warp CTA that needs a slot in every partition (first attempt: 8-warp CTAs
// never became resident beside the forward kernel and every tile timed out).
// The wait is bounded: if a tile never arrives (the forward kernel failed) SS_STATUS_ROLLOUT_TIMEOUT is raised.
struct TilesArgs {
    StepArgs S;
    int *tile_ready;
    int64_t units;          // tiles of the forward launch
    int grid_fwd;           // its CTA count
};

template <bool STATS>
__global__ void __launch_bounds__(32, 16) step_pp_tiles_kernel(const TilesArgs T) {
    const StepArgs &A = T.S;
    const int lane = threadIdx.x, P = lane & 1;
    // One warp per CTA, one quarter tile (32 rows) per CTA.  CTAs are numbered in the order the forward kernel completes its
    // tiles: its CTA c walks tiles u0(c), u0(c) + 1, ..., so step j of every forward CTA comes before step j + 1 of any.
    const int per_step = 4 * T.grid_fwd;
    const int64_t j = blockIdx.x / per_step;
    const int c = (int)(blockIdx.x % per_step) >> 2, quarter = blockIdx.x & 3;
    const int64_t u0 = T.units * c / T.grid_fwd, u1 = T.units * (c + 1) / T.grid_fwd;
    const int64_t tile = u0 + j;
    if (tile >= u1) return;
    const int64_t rows = 2 * A.n;
    uint32_t status = 0;
    // wait for the four output warps of the forward kernel
    if (lane == 0) {
        int seen = 0;
        uint32_t spins = 0;
        for (;;) {
            asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(seen) : "l"(T.tile_ready + tile) : "memory");
            if (seen >= 4) break;
            if (++spins > (1u << 20)) { status |= SS_STATUS_ROLLOUT_TIMEOUT; break; }
            __nanosleep(200);
        }
    }
    __syncwarp();
    const int64_t g0 = tile * 128 + quarter * 32 + lane;
    const int64_t last = rows - 2 + P;
    const bool active = g0 <= last;
    const int64_t gl = active ? g0 : last;
    const int64_t env = gl >> 1;
    sspp::LaneState L;
    sspp::lane_load((const char *)A.state, A.n, gl, L);
    const float2 a = __ldcg((const float2 *)A.actions + gl);
    sspp::LaneTrig Tr;
    sspp::lane_trig(L, Tr);
    sspp::LaneTickOut out;
    sspp::lane_obs_tick(L, Tr, a.x, a.y, A.P, (uint64_t)env, A.P.counter, lane, P, status, out);
    const int v_other = __shfl_xor_sync(0xffffffffu, L.valid, 1);
    if (active) {
        sspp::lane_store((char *)A.state, A.n, gl, L, v_other);
        if (A.reward_out && A.P.reward_mode != SS_REWARD_NONE) ((float *)A.reward_out)[gl] = out.reward;
        uint8_t *flag = P ? A.winner_out : A.done_out;
        if (flag) flag[env] = (uint8_t)(P ? out.winner : out.done);
        if (A.done_rows_out) ((uint8_t *)A.done_rows_out)[gl] = out.winner ? 1 : 0;
        if (STATS && !P && out.episode_len >= 0) sspp::count_episode_pp(A.stats, out.episode_len, out.winner, (int)A.P.tick_limit);
#pragma unroll
        for (int q = 0; q < 3; ++q) {
            A.obs_out[gl * 3 + q] = out.obs[q];
            if (A.obs_out2) A.obs_out2[gl * 3 + q] = out.obs[q];
        }
    }
    // hand the counter back for the next tick (the four quarter-tile CTAs each take one arrival away)
    __syncwarp();
    if (lane == 0) atomicSub(T.tile_ready + tile, 1);
    if (status && A.status) atomicOr(A.status, status);
}

__global__ void reset_kernel(void *state, int64_t n, const uint8_t *mask, int reset_mode,
                             const int32_t *positions, uint64_t seed, uint64_t counter) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (mask && !mask[i]) return;
    Env e;
    if (reset_mode == SS_RESET_GIVEN) {
        const int4 p = ((const int4 *)positions)[i];
        reset_env(e, p.x, p.y, p.z, p.w);
    } else if (reset_mode == SS_RESET_RANDOM) {
        reset_random(e, seed, (uint64_t)i, counter);
    } else {
        reset_env(e, 50, 50, 200, 200);
    }
    store_env(planes_of(state, n), i, e);
}

template <bool SPEEDS>
__global__ void features_kernel(const void *state, int64_t n, double *feat_out, double *obs_out,
                                int32_t *general_out, const void *speeds) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Env e;
    load_env(planes_of((void *)state, n), i, e);
    Speeds k = default_speeds();
    if (SPEEDS) k = load_speeds(speeds, n, i);
    if (general_out) {
        general_out[i * 3 + 0] = e.live; general_out[i * 3 + 1] = e.ticks; general_out[i * 3 + 2] = e.winner;
    }
    if (feat_out) {
        double f[kNumFeat];
        features_of<0>(e, f);
        for (int j = 0; j < kNumFeat; ++j) feat_out[(i * 2 + 0) * kNumFeat + j] = f[j];
        features_of<1>(e, f);
        for (int j = 0; j < kNumFeat; ++j) feat_out[(i * 2 + 1) * kNumFeat + j] = f[j];
    }
    if (obs_out) {
        double o[kNumObs];
        View v0 = view_of<0, false>(e), v1 = view_of<1, false>(e);
        obs_of<0>(e, v0, k, o);
        for (int j = 0; j < kNumObs; ++j) obs_out[(i * 2 + 0) * kNumObs + j] = o[j];
        obs_of<1>(e, v1, k, o);
        for (int j = 0; j < kNumObs; ++j) obs_out[(i * 2 + 1) * kNumObs + j] = o[j];
    }
}

__global__ void export_kernel(const void *state, int64_t n, int64_t first, int64_t count,
                              int32_t *ints, double *rots) {
    int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= count) return;
    Env e;
    load_env(planes_of((void *)state, n), first + j, e);
    int32_t *o = ints + j * SS_EXPORT_INTS;
    o[0] = e.px[0]; o[1] = e.px[1]; o[2] = e.py[0]; o[3] = e.py[1];
    o[4] = e.qx[0]; o[5] = e.qx[1]; o[6] = e.qy[0]; o[7] = e.qy[1];
    o[8] = e.cd[0]; o[9] = e.cd[1]; o[10] = e.age[0]; o[11] = e.age[1];
    o[12] = e.valid[0]; o[13] = e.valid[1]; o[14] = e.ticks; o[15] = e.live; o[16] = e.winner;
    double *r = rots + j * 4;
    r[0] = e.prot[0]; r[1] = e.prot[1]; r[2] = e.qrot[0]; r[3] = e.qrot[1];
}

__global__ void import_kernel(void *state, int64_t n, int64_t first, int64_t count,
                              const int32_t *ints, const double *rots) {
    int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= count) return;
    Env e;
    const int32_t *o = ints + j * SS_EXPORT_INTS;
    e.px[0] = o[0] & 255; e.px[1] = o[1] & 255; e.py[0] = o[2] & 255; e.py[1] = o[3] & 255;
    e.qx[0] = o[4] & 255; e.qx[1] = o[5] & 255; e.qy[0] = o[6] & 255; e.qy[1] = o[7] & 255;
    e.cd[0] = o[8]; e.cd[1] = o[9]; e.age[0] = o[10]; e.age[1] = o[11];
    e.valid[0] = o[12] != 0; e.valid[1] = o[13] != 0; e.ticks = o[14]; e.live = o[15] != 0; e.winner = o[16] & 3;
    const double *r = rots + j * 4;
    e.prot[0] = r[0]; e.prot[1] = r[1]; e.qrot[0] = r[2]; e.qrot[1] = r[3];
    store_env(planes_of(state, n), first + j, e);
}

template <int P>
__device__ void apply_player_op(Env &e, int op, double value, const Speeds &k, uint32_t &status) {
    double s, c;
    switch (op) {
        case SS_OP_MOVE_DIRECTION_FLOAT:
            sincos_d(e.prot[P], &s, &c);
            move_direction_float<P>(e, value, s, c, k, status);
            break;
        case SS_OP_MOVE_LOOK_FLOAT: move_look_float<P>(e, value, k); break;
        case SS_OP_SHOOT: move_shoot<P>(e, k); break;
        // Player.move_forwards / move_backwards (Player.py:41-55) are
        // pos -/+ sin(rot)*speed_move: the same IEEE values as
        // move_direction_float(+1 / -1).
        case SS_OP_MOVE_FORWARDS:
            sincos_d(e.prot[P], &s, &c);
            move_direction_float<P>(e, 1.0, s, c, k, status);
            break;
        case SS_OP_MOVE_BACKWARDS:
            sincos_d(e.prot[P], &s, &c);
            move_direction_float<P>(e, -1.0, s, c, k, status);
            break;
        case SS_OP_LOOK_LEFT: e.prot[P] = add(e.prot[P], k.speed_look); break;     // Player.py:28
        case SS_OP_LOOK_RIGHT: e.prot[P] = sub(e.prot[P], k.speed_look); break;    // Player.py:31
        default: break;
    }
}

__global__ void apply_kernel(void *state, int64_t n, int64_t env, int player, int op, double value,
                             const void *speeds, uint32_t *status_out) {
    Env e;
    const StatePlanes S = planes_of(state, n);
    load_env(S, env, e);
    Speeds k = speeds ? load_speeds(speeds, n, env) : default_speeds();
    uint32_t status = 0;
    if (op == SS_OP_GAME_TICK) {
        if (e.live) {                                   // SkillshotGame.py:115-122
            double s, c;
            e.ticks += 1;
            sincos_d(e.qrot[0], &s, &c); proj_tick<0>(e, s, c, k, status);
            sincos_d(e.qrot[1], &s, &c); proj_tick<1>(e, s, c, k, status);
            check_collision(e);
        }
    } else if (player == 0) {
        apply_player_op<0>(e, op, value, k, status);
    } else {
        apply_player_op<1>(e, op, value, k, status);
    }
    store_env(S, env, e);
    if (status && status_out) atomicOr(status_out, status);
}

// ---------------------------------------------------------------------------------------------------------------------
// Matches (ss_env_step_match, ss_match_summary): two policies, one game per env, the seat map of the header -- in env
// i < split policy A is player 1.  Actions and observations are policy-major ([2][n] rows, env i at row i of each half).
struct MatchStepArgs {
    void *state;
    int64_t n, split, tick_limit;
    const float2 *actions;      // [2][n]
    float4 *obs_out;            // [2][n][3]
    const void *speeds;
    uint32_t *status;
};

// fast_obs sink: player P's three float4 go to the row of the policy that sits in seat P
struct SeatSink {
    float4 *p1, *p2;
    __device__ __forceinline__ void put(int j, float a, float b, float c, float d) {
        (j < 3 ? p1 : p2)[j < 3 ? j : j - 3] = make_float4(a, b, c, d);
    }
};

// Leagues (ss_env_step_seated, ss_league_summary): any number of policies, each env's two rows given by a seat table.
struct SeatedStepArgs {
    void *state;
    int64_t n, n_rows, tick_limit;
    const int2 *seat_rows;      // [n]
    const float2 *actions;      // [n_rows]
    float4 *obs_out;            // [n_rows][3]
    const void *speeds;
    uint32_t *status;
};

// How match_step_kernel finds an env's two rows (static functions of the kernel's arguments).  ok() is false when the env
// is not to be stepped at all; act_a / act_b and obs_a / obs_b are the two rows' actions and observations, and player 1's
// row is the "a" row when a_first().
// SplitSeats (ss_env_step_match): env i < split seats policy A (rows [0, n)) first, the others policy B (rows [n, 2 n)).
struct SplitSeats {
    using Args = MatchStepArgs;
    __device__ __forceinline__ static bool ok(const Args &, int64_t) { return true; }
    __device__ __forceinline__ static bool a_first(const Args &A, int64_t i) { return i < A.split; }
    __device__ __forceinline__ static const float2 *act_a(const Args &A, int64_t i) { return A.actions + i; }
    __device__ __forceinline__ static const float2 *act_b(const Args &A, int64_t i) { return A.actions + A.n + i; }
    __device__ __forceinline__ static float4 *obs_a(const Args &A, int64_t i) { return A.obs_out + i * 3; }
    __device__ __forceinline__ static float4 *obs_b(const Args &A, int64_t i) { return A.obs_out + (A.n + i) * 3; }
};

// TableSeats (ss_env_step_seated): seat_rows[i] = {row of player 1, row of player 2}.  An env with a row outside
// [0, n_rows) is not stepped, reads and writes no row and raises SS_STATUS_SEAT_RANGE.
struct TableSeats {
    using Args = SeatedStepArgs;
    __device__ __forceinline__ static bool ok(const Args &A, int64_t i) {
        const int2 r = __ldg(A.seat_rows + i);
        return r.x >= 0 && r.y >= 0 && r.x < A.n_rows && r.y < A.n_rows;
    }
    __device__ __forceinline__ static bool a_first(const Args &, int64_t) { return true; }
    __device__ __forceinline__ static const float2 *act_a(const Args &A, int64_t i) { return A.actions + __ldg(A.seat_rows + i).x; }
    __device__ __forceinline__ static const float2 *act_b(const Args &A, int64_t i) { return A.actions + __ldg(A.seat_rows + i).y; }
    __device__ __forceinline__ static float4 *obs_a(const Args &A, int64_t i) { return A.obs_out + (int64_t)__ldg(A.seat_rows + i).x * 3; }
    __device__ __forceinline__ static float4 *obs_b(const Args &A, int64_t i) { return A.obs_out + (int64_t)__ldg(A.seat_rows + i).y * 3; }
};

// One tick of one env per thread: the arithmetic of step_kernel<OBS, CARRY> with reward mode none and no auto-reset
// (act_and_tick_carry, then fast_view / fast_obs of the post-tick state), hence the same bits.  A live game at the tick
// limit is left as it is; its observation is written again.
template <bool SPEEDS, class Seats>
__global__ void __launch_bounds__(kBlock, 8) match_step_kernel(const typename Seats::Args A) {
    const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (i >= A.n) return;
    if (!Seats::ok(A, i)) {
        if (A.status) atomicOr(A.status, (uint32_t)SS_STATUS_SEAT_RANGE);
        return;
    }
    const StatePlanes S = planes_of(A.state, A.n);
    Env e;
    load_env(S, i, e);
    const Speeds k = SPEEDS ? load_speeds(A.speeds, A.n, i) : default_speeds();
    const bool a_first = Seats::a_first(A, i);
    const float2 aa = __ldg(Seats::act_a(A, i)), ab = __ldg(Seats::act_b(A, i));
    const float2 p1 = a_first ? aa : ab, p2 = a_first ? ab : aa;
    Trig tr;
    trig_of(e, tr);
    uint32_t status = 0;
    const bool frozen = e.live && e.ticks >= A.tick_limit;
    if (!frozen) act_and_tick_carry(e, p1.x, p1.y, p2.x, p2.y, k, status, tr);
    const FastView v0 = fast_view<0>(e, tr, false), v1 = fast_view<1>(e, tr, false);
    float4 *row_a = Seats::obs_a(A, i), *row_b = Seats::obs_b(A, i);
    SeatSink sink{a_first ? row_a : row_b, a_first ? row_b : row_a};
    fast_obs<0>(e, v0, k, sink);
    fast_obs<1>(e, v1, k, sink);
    if (!frozen) store_env(S, i, e);
    if (status && A.status) atomicOr(A.status, status);
}

// The [P][P][8] counters of ss_league_summary.  The envs are pair-major, so the lanes of a warp nearly always share one
// or two cells: the lanes of one cell (__match_any_sync) count their outcomes with ballots and sum their ticks with one
// reduction, and the cell's lowest lane adds the totals -- one atomic per non-zero counter, cell and warp.  An env whose
// policy index is >= P is not counted.
__global__ void league_summary_kernel(const void *state, int64_t n, const uint8_t *seat_policy, int P, int64_t tick_limit,
                                      unsigned long long *out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    int cell = -1, ticks = 0, k = -1;                 // k: the counter this env adds one to (1..4)
    if (i < n) {
        const uchar2 sp = __ldg(reinterpret_cast<const uchar2 *>(seat_policy) + i);
        if (sp.x < P && sp.y < P) {
            const int4 b = planes_of((void *)state, n).ib[i];
            const int live = (b.w >> 2) & 1, winner = (b.w >> 4) & 3;
            cell = sp.x * P + sp.y;
            // winner_id = the player that was hit: seat 1 wins when player 2 was hit
            k = !live ? (winner == 2 ? 1 : 2) : (b.z >= tick_limit ? 3 : 4);
            ticks = live ? 0 : b.z;
        }
    }
    const unsigned peers = __match_any_sync(0xffffffffu, cell);
    const unsigned mine[5] = {peers & __ballot_sync(0xffffffffu, cell >= 0), peers & __ballot_sync(0xffffffffu, k == 1),
                              peers & __ballot_sync(0xffffffffu, k == 2), peers & __ballot_sync(0xffffffffu, k == 3),
                              peers & __ballot_sync(0xffffffffu, k == 4)};
    // ticks < 2^31: the two 16-bit halves summed over at most 32 lanes cannot overflow 32 bits
    const unsigned lo = __reduce_add_sync(peers, (unsigned)ticks & 0xffffu), hi = __reduce_add_sync(peers, (unsigned)ticks >> 16);
    if (cell < 0 || lane != __ffs(peers) - 1) return;
    unsigned long long *c = out + (int64_t)cell * 8;
#pragma unroll
    for (int j = 0; j < 5; ++j)
        if (mine[j]) atomicAdd(c + j, (unsigned long long)__popc(mine[j]));
    const unsigned long long t = (unsigned long long)lo + ((unsigned long long)hi << 16);
    if (t) atomicAdd(c + 5, t);
}

// The [2][8] outcome counters of ss_match_summary: per-CTA sums in shared memory, then one atomic per counter and CTA.
__global__ void match_summary_kernel(const void *state, int64_t n, int64_t split, int64_t tick_limit, unsigned long long *out) {
    __shared__ unsigned long long acc[SS_MATCH_STATS];
    if (threadIdx.x < SS_MATCH_STATS) acc[threadIdx.x] = 0;
    __syncthreads();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        const int4 b = planes_of((void *)state, n).ib[i];
        const int ticks = b.z, live = (b.w >> 2) & 1, winner = (b.w >> 4) & 3;
        const int seat = i < split ? 0 : 1;              // block 0: A is player 1
        unsigned long long *c = acc + 8 * seat;
        atomicAdd(c + 0, 1ull);
        if (!live) {
            // winner_id = the player that was hit: A was hit when it is A's seat (player 1 in block 0, player 2 in block 1)
            atomicAdd(c + (winner == seat + 1 ? 2 : 1), 1ull);
            atomicAdd(c + 5, (unsigned long long)ticks);
        } else {
            atomicAdd(c + (ticks >= tick_limit ? 3 : 4), 1ull);
        }
    }
    __syncthreads();
    if (threadIdx.x < SS_MATCH_STATS && acc[threadIdx.x]) atomicAdd(out + threadIdx.x, acc[threadIdx.x]);
}

// ---------------------------------------------------------------------------------------------------------------------
// pool_step_speeds_kernel -- ss_env_step_pool_speeds: one tick of the pool with per-env speeds, ONE THREAD PER ENV.  The
// per-player kernels fold the reference constants into their arithmetic (ss_env_pp.cuh); per-env speeds run on the core's
// tick_env, called as step_kernel<OBS, CARRY, SPEEDS> calls it, so the bytes of every env are ss_env_step_ring's.  The
// rows are BlockPoolRows': self-play env i < S reads its float2 actions from learner rows 2i, 2i + 1; in pool env S + j
// the learner's float2 is learner row 2S + j and the opponent's opponent row j, seated by the block's learner player.
// The learner rows of the warp's envs are one contiguous run (env S - 1 ends at row 2S - 1, the pool's start at 2S), and
// so are its opponent rows: learner row r takes tile slot r - l0 and opponent row o slot nl + o - o0.  Slot s is staged
// at float4 3s + (s >> 1) of the warp's tile -- for a self-play warp that is step_kernel's conflict-free 7-float4 row per
// env -- and the warp writes each run with coalesced stores, as step_pp_obs_kernel does.
__device__ __forceinline__ int slot_at(int s) { return 3 * s + (s >> 1); }

template <bool STATS>
__global__ void __launch_bounds__(kBlock, 8) pool_step_speeds_kernel(const StepArgs A, const BlockPoolRows R) {
    __shared__ float4 tile[kBlock / 32][32 * kRowF4];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    const int64_t e0 = i - lane, e1 = min(e0 + 32, A.n);           // the warp's envs
    const bool active = i < A.n;
    const StatePlanes S = planes_of(A.state, A.n);
    // first learner row of env e (e = n gives L); an env past the self-play envs has one learner row
    auto lrow = [&](int64_t e) { return e < R.S ? 2 * e : R.S + e; };
    const int64_t l0 = lrow(e0), o0 = max(e0, R.S) - R.S;
    const int nl = (int)(lrow(e1) - l0);
    const bool pool = i >= R.S;
    int learner_player = 0, block = 0;
    if (active && pool) block = pool_block_of(R, (int)(i - R.S), learner_player);
    // tile slots of player 1's and player 2's rows
    const int ls = (int)(lrow(i) - l0), os = nl + (int)(i - R.S - o0);
    const int s1 = !pool ? ls : learner_player == 0 ? ls : os;
    const int s2 = !pool ? ls + 1 : learner_player == 1 ? ls : os;
    // ss_launch.cuh: in the rollout loop this grid is placed while the forward kernels' last CTAs finish, and waits here
    sslaunch::griddep_wait();
    sslaunch::griddep_launch();
    uint32_t status = 0;
    if (active) {
        Env e;
        load_env(S, i, e);
        const Speeds k = load_speeds(A.speeds, A.n, i);
        const float2 *act = (const float2 *)A.actions;
        float2 p1, p2;
        if (!pool) {
            p1 = __ldg(act + 2 * i); p2 = __ldg(act + 2 * i + 1);
        } else {
            const float2 la = __ldg(act + R.S + i), oa = __ldg(R.opp_actions + (i - R.S));
            p1 = learner_player == 0 ? la : oa; p2 = learner_player == 0 ? oa : la;
        }
        // a game that is over before the tick stays "done" and is not an episode end again (step_kernel's STATS rule)
        const int ticks_before = (!e.live || (A.P.tick_limit > 0 && e.ticks >= A.P.tick_limit)) ? -1 : e.ticks;
        Trig tr;
        trig_of(e, tr);
        float r[2];
        int done, winner;
        SeatSink sink{&tile[warp][slot_at(s1)], &tile[warp][slot_at(s2)]};
        tick_env<true, true>(e, p1.x, p1.y, p2.x, p2.y, k, A.P, (uint64_t)i, 0, true, status, tr, r, done, winner, sink);
        store_env(S, i, e);
        const bool write_reward = A.reward_out && A.P.reward_mode != SS_REWARD_NONE;
        float *reward = (float *)A.reward_out;
        uint8_t *done_rows = (uint8_t *)A.done_rows_out;
        if (!pool) {
            if (write_reward) { reward[2 * i] = r[0]; reward[2 * i + 1] = r[1]; }
            if (done_rows) { done_rows[2 * i] = winner ? 1 : 0; done_rows[2 * i + 1] = winner ? 1 : 0; }
        } else {
            if (write_reward) reward[R.S + i] = r[learner_player];
            if (done_rows) done_rows[R.S + i] = winner ? 1 : 0;
        }
        if (A.done_out) A.done_out[i] = (uint8_t)done;
        if (A.winner_out) A.winner_out[i] = (uint8_t)winner;
        if (done && ticks_before >= 0) {                                // rare: a few atomics per finished game
            if (STATS) count_episode(A.stats, ticks_before + 1, winner, (int)A.P.tick_limit);
            if (pool && R.pool_stats) count_pool_game(R.pool_stats + block * 8, ticks_before + 1, winner, learner_player);
        }
    }
    __syncwarp();
    const int n_out = 3 * (nl + (int)(max(e1, R.S) - R.S - o0));
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        const int idx = j * 32 + lane;
        if (idx < 3 * nl) {
            const float4 v = tile[warp][idx + (idx / 3 >> 1)];
            A.obs_out[l0 * 3 + idx] = v;
            if (A.obs_out2) A.obs_out2[l0 * 3 + idx] = v;
        } else if (idx < n_out) {
            R.opp_obs[o0 * 3 + (idx - 3 * nl)] = tile[warp][idx + (idx / 3 >> 1)];
        }
    }
    if (status && A.status) atomicOr(A.status, status);
}

inline int check_launch() { return cudaGetLastError() == cudaSuccess ? SS_OK : SS_ERR_CUDA; }
inline unsigned blocks_for(int64_t n, int block) { return (unsigned)((n + block - 1) / block); }
// CTA size of step_pp_kernel for n_envs (see the kernel): 896 when that still makes at least ~one CTA per SM (65,536 envs
// are 147 CTAs on 148 SMs), else 448, else 64.  SS_STEP_BLK = 64 / 448 / 896 forces one (A/B measurements, the equality test).
// SM count of the current device (asked once: the GPUs of a box are alike)
inline int sm_count() {
    static int sms = 0;
    if (sms == 0) {
        int dev = 0, v = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v < 1) v = 148;
        sms = v;
    }
    return sms;
}
inline int pp_block_for(int64_t n_envs) {
    if (const char *e = getenv("SS_STEP_BLK")) {
        const int v = atoi(e);
        if (v == 64 || v == 448 || v == 896) return v;
    }
    const int sms = sm_count();
    // Measured on one box (profiles/r2_step_blk_sweep.txt, 256 ticks per launch, 896 against 64 threads): 65,536 envs
    // +7.6 %, 131,072 +6.7 %, 262,144 +1.8 % (-1.2 % at 32 ticks), 1,048,576 -1.6 % (-5.3 % at 32 ticks): with many waves
    // the small CTAs refill an SM two warps at a time and win.  Hence: one big CTA per SM up to three waves.
    const int64_t lanes = 2 * n_envs, c896 = (lanes + 895) / 896, c448 = (lanes + 447) / 448;
    if (c896 * 20 >= (int64_t)sms * 19) return c896 <= 3 * (int64_t)sms ? 896 : 64;
    if (c448 * 20 >= (int64_t)sms * 19) return 448;
    return 64;
}
template <int OUT, int BLK>
inline int launch_step_pp_blk(const StepArgs &A, int64_t n_envs, cudaStream_t st) {
    constexpr int ring_bytes = kRingD * BLK * (int)sizeof(float2);      // 56 KB at 896 threads: above the 48 KB default
    // The launch needs the function's dynamic shared-memory limit raised, and that limit belongs to the function on one
    // device: it is set the first time this process launches the kernel on each device (devices past 63 on every call).
    static std::atomic<uint64_t> configured{0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return SS_ERR_CUDA;
    const uint64_t bit = dev < 64 ? 1ull << dev : 0;
    if (!(configured.load(std::memory_order_acquire) & bit)) {
        if (cudaFuncSetAttribute(step_pp_kernel<OUT, BLK>, cudaFuncAttributeMaxDynamicSharedMemorySize, ring_bytes) != cudaSuccess)
            return SS_ERR_CUDA;
        configured.fetch_or(bit, std::memory_order_acq_rel);
    }
    step_pp_kernel<OUT, BLK><<<blocks_for(2 * n_envs, BLK), BLK, ring_bytes, st>>>(A);
    return check_launch();
}
template <int OUT>
inline int launch_step_pp(const StepArgs &A, int64_t n_envs, cudaStream_t st) {
    switch (pp_block_for(n_envs)) {
        case 896: return launch_step_pp_blk<OUT, 896>(A, n_envs, st);
        case 448: return launch_step_pp_blk<OUT, 448>(A, n_envs, st);
        default: return launch_step_pp_blk<OUT, 64>(A, n_envs, st);
    }
}

}  // namespace

extern "C" {

int ss_version(void) { return 100; }

int64_t ss_state_bytes(int64_t n_envs) { return n_envs * SS_STATE_BYTES_PER_ENV; }

int ss_env_reset(void *state, int64_t n_envs, const uint8_t *mask, int reset_mode,
                 const int32_t *positions, uint64_t seed, uint64_t counter, void *stream) {
    if (!state || n_envs <= 0 || reset_mode < 0 || reset_mode > 2) return SS_ERR_INVALID_ARG;
    if (reset_mode == SS_RESET_GIVEN && !positions) return SS_ERR_INVALID_ARG;
    reset_kernel<<<blocks_for(n_envs, 256), 256, 0, (cudaStream_t)stream>>>(state, n_envs, mask, reset_mode,
                                                                            positions, seed, counter);
    return check_launch();
}

int ss_env_step_ring(void *state, int64_t n_envs, const float *actions, float *obs_out, float *obs_out2,
                     float *reward_out, uint8_t *done_out, uint8_t *done_rows_out, uint8_t *winner_out,
                     int n_ticks, int reward_mode, int64_t tick_limit, int auto_reset,
                     int reset_mode, uint64_t seed, uint64_t counter, const void *speeds,
                     uint32_t *status, int flags, void *stream) {
    if (!state || !actions || n_envs <= 0 || n_ticks <= 0) return SS_ERR_INVALID_ARG;
    if ((obs_out2 && (!obs_out || n_ticks != 1)) || ((uintptr_t)obs_out2 & 15) || ((uintptr_t)done_rows_out & 1))
        return SS_ERR_INVALID_ARG;
    if (reward_mode < 0 || reward_mode > 3) return SS_ERR_INVALID_ARG;
    if (auto_reset && reset_mode != SS_RESET_FIXED && reset_mode != SS_RESET_RANDOM) return SS_ERR_INVALID_ARG;
    if (((uintptr_t)state | (uintptr_t)actions | (uintptr_t)obs_out) & 15) return SS_ERR_INVALID_ARG;
    if ((uintptr_t)reward_out & 7) return SS_ERR_INVALID_ARG;
    StepArgs A;
    A.state = state; A.n = n_envs; A.actions = (const float4 *)actions; A.obs_out = (float4 *)obs_out;
    A.reward_out = (float2 *)reward_out; A.done_out = done_out; A.winner_out = winner_out;
    A.obs_out2 = (float4 *)obs_out2; A.done_rows_out = (uint16_t *)done_rows_out;
    A.speeds = speeds; A.status = status; A.packed_out = nullptr;
    A.stats = (status && (flags & SS_STEP_EPISODE_STATS)) ? reinterpret_cast<unsigned long long *>(status) + 1 : nullptr;
    if (A.stats && ((uintptr_t)status & 7)) return SS_ERR_INVALID_ARG;
    A.P.seed = seed; A.P.counter = counter; A.P.tick_limit = tick_limit;
    A.P.reward_mode = reward_mode; A.P.auto_reset = auto_reset ? 1 : 0; A.P.reset_mode = reset_mode;
    A.n_ticks = n_ticks; A.obs_every_tick = (flags & SS_STEP_OBS_EVERY_TICK) ? 1 : 0;
    const dim3 grid(blocks_for(n_envs, kBlock)), block(kBlock);
    cudaStream_t st = (cudaStream_t)stream;
    const bool shaped = (reward_mode == SS_REWARD_LOOKING || reward_mode == SS_REWARD_SIMPLE) && reward_out;
    const bool carry = obs_out || n_ticks > 1 || shaped;
    // The staging tile is 7 KB + 1 KB driver reserve per CTA; ask for a carve-out that fits 8+ CTAs.
    static bool configured = false;
    if (!configured) {
        cudaFuncSetAttribute(step_kernel<true, true, false, 8>, cudaFuncAttributePreferredSharedMemoryCarveout, 50);
        cudaFuncSetAttribute(step_kernel<true, true, true, 8>, cudaFuncAttributePreferredSharedMemoryCarveout, 50);
        cudaFuncSetAttribute(step_kernel<true, true, false, 8, true>, cudaFuncAttributePreferredSharedMemoryCarveout, 50);
        cudaFuncSetAttribute(step_kernel<true, true, true, 8, true>, cudaFuncAttributePreferredSharedMemoryCarveout, 50);
        configured = true;
    }
    // (the statistics variants are separate instantiations: the bookkeeping costs the physics-only kernels a few
    //  registers and ~5 % when compiled in)
    if (obs_out && n_ticks == 1 && !speeds && reward_mode != SS_REWARD_SIMPLE) {
        // the rollout's env step: one tick with observations, one thread per player
        const dim3 grid_pp(blocks_for(2 * n_envs, kBlockPP));
        if ((A.stats ? sslaunch::launch(step_pp_obs_kernel<true, SelfPlayRows>, grid_pp, dim3(kBlockPP), 0, st, A, SelfPlayRows{})
                     : sslaunch::launch(step_pp_obs_kernel<false, SelfPlayRows>, grid_pp, dim3(kBlockPP), 0, st, A, SelfPlayRows{})) != cudaSuccess)
            return SS_ERR_CUDA;
    } else if (obs_out) {
        // 8 CTAs (16 warps) per SM: capping the observation kernel at 128 registers measured
        // 83 us vs 100 us uncapped at 1M envs (profiles/README.md)
        if (A.stats) {
            if (speeds) step_kernel<true, true, true, 8, true><<<grid, block, 0, st>>>(A);
            else step_kernel<true, true, false, 8, true><<<grid, block, 0, st>>>(A);
        } else {
            if (speeds) step_kernel<true, true, true, 8><<<grid, block, 0, st>>>(A);
            else step_kernel<true, true, false, 8><<<grid, block, 0, st>>>(A);
        }
    } else if (n_ticks > 1 && !A.stats && !speeds && !shaped && !done_rows_out && done_out && winner_out &&
               2 * n_envs * ((int64_t)n_ticks + 2) < (int64_t)0x7fffffff) {     // (32-bit running index)
        // physics-only fused ticks (bench.py's timed shape): one thread per player.  (A single tick per launch stays on
        // the one-thread-per-env kernel: a launch then pays 3 sincos per lane to set up what it carries, measured 4.1 vs 3.9 us.)
        if ((reward_out && reward_mode == SS_REWARD_TERMINAL ? launch_step_pp<OUT_TERMINAL>(A, n_envs, st)
                                                             : launch_step_pp<OUT_FLAGS>(A, n_envs, st)) != SS_OK)
            return SS_ERR_CUDA;
    } else if (carry) {
        if (A.stats) {
            if (speeds) step_kernel<false, true, true, 1, true><<<grid, block, 0, st>>>(A);
            else step_kernel<false, true, false, 1, true><<<grid, block, 0, st>>>(A);
        } else {
            if (speeds) step_kernel<false, true, true><<<grid, block, 0, st>>>(A);
            else step_kernel<false, true, false><<<grid, block, 0, st>>>(A);
        }
    } else {
        // One physics tick per launch: a ~2 us kernel behind ~2 us of launch latency.  Launched with programmatic stream
        // serialization, the grid is scheduled while its predecessor drains and waits (griddepcontrol.wait) before its
        // first global access: back-to-back one-tick launches overlap their launch latency with the previous tick's tail.
        if (!A.stats && !speeds) {
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = 0; cfg.stream = st;
            cudaLaunchAttribute attr[1];
            attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
            attr[0].val.programmaticStreamSerializationAllowed = 1;
            cfg.attrs = attr; cfg.numAttrs = 1;
            // CTA size: when the whole batch is ONE wave of one 448-thread CTA per SM (65,536 envs on 148 SMs: 147 CTAs) the
            // launch measured 3.53 us against 4.11 us with two-warp CTAs (0.57 against 0.49 of the HBM roofline of the
            // 202-byte model, profiles/r2_step1_blk_sweep.txt); with more than one wave the small CTAs win (9.7 against
            // 12.2 us at 262,144 envs).  SS_STEP1_BLK = 64 / 448 forces one.
            int blk1 = 64;
            {
                const char *xe = getenv("SS_STEP1_BLK");
                const int xb = xe ? atoi(xe) : 0;
                const int sms = sm_count();
                const int64_t c448 = (n_envs + 447) / 448;
                if (xb == 64 || xb == 448) blk1 = xb;
                else if (c448 <= sms && c448 * 20 >= (int64_t)sms * 19) blk1 = 448;
            }
            if (blk1 == 448) {
                cfg.gridDim = dim3(blocks_for(n_envs, 448)); cfg.blockDim = dim3(448);
                if (cudaLaunchKernelEx(&cfg, step_kernel<false, false, false, 1, false, true, 448>, A) != cudaSuccess) return SS_ERR_CUDA;
            } else
            if (cudaLaunchKernelEx(&cfg, step_kernel<false, false, false, 1, false, true>, A) != cudaSuccess) return SS_ERR_CUDA;
        } else if (A.stats) {
            if (speeds) step_kernel<false, false, true, 1, true><<<grid, block, 0, st>>>(A);
            else step_kernel<false, false, false, 1, true><<<grid, block, 0, st>>>(A);
        } else {
            step_kernel<false, false, true><<<grid, block, 0, st>>>(A);
        }
    }
    return check_launch();
}

// ss_env_step_pool (blocks false: PoolRows), ss_env_step_pool_blocks (blocks true: BlockPoolRows from opp_envs) and
// ss_env_step_pool_speeds (blocks true, speeds not NULL: pool_step_speeds_kernel under BlockPoolRows)
static int step_pool(void *state, int64_t n_envs, int64_t pool_envs, int n_opponents, const float *actions,
                     const float *opp_actions, float *obs_out, float *obs_out2, float *reward_out, uint8_t *done_rows_out,
                     float *opp_obs_out, uint8_t *done_out, uint8_t *winner_out, int reward_mode, int64_t tick_limit,
                     int reset_mode, uint64_t seed, uint64_t counter, uint32_t *status, int flags, uint64_t *pool_stats,
                     bool blocks, const int64_t *opp_envs, const void *speeds, void *stream) {
    if (!state || !actions || !obs_out || n_envs <= 0 || pool_envs < 0 || pool_envs > n_envs) return SS_ERR_INVALID_ARG;
    if (pool_envs > 0 && (n_opponents < 1 || n_opponents > SS_LEAGUE_MAX_POLICIES || !opp_actions || !opp_obs_out))
        return SS_ERR_INVALID_ARG;
    BlockPoolRows B{};
    if (blocks && !pool_block_table(n_envs, pool_envs, n_opponents, opp_envs, B)) return SS_ERR_INVALID_ARG;
    if (!blocks && pool_envs > 0 && pool_envs % (2 * n_opponents) != 0) return SS_ERR_INVALID_ARG;
    if (reward_mode != SS_REWARD_NONE && reward_mode != SS_REWARD_LOOKING && reward_mode != SS_REWARD_TERMINAL) return SS_ERR_INVALID_ARG;
    if (reset_mode != SS_RESET_FIXED && reset_mode != SS_RESET_RANDOM) return SS_ERR_INVALID_ARG;
    if ((((uintptr_t)state | (uintptr_t)obs_out | (uintptr_t)obs_out2 | (uintptr_t)opp_obs_out) & 15) ||
        (((uintptr_t)actions | (uintptr_t)opp_actions | (uintptr_t)pool_stats) & 7) || (((uintptr_t)reward_out | (uintptr_t)status) & 3))
        return SS_ERR_INVALID_ARG;
    StepArgs A{};
    A.state = state; A.n = n_envs; A.actions = (const float4 *)actions; A.obs_out = (float4 *)obs_out; A.obs_out2 = (float4 *)obs_out2;
    A.reward_out = (float2 *)reward_out; A.done_out = done_out; A.winner_out = winner_out; A.done_rows_out = (uint16_t *)done_rows_out;
    A.status = status;
    A.stats = (status && (flags & SS_STEP_EPISODE_STATS)) ? reinterpret_cast<unsigned long long *>(status) + 1 : nullptr;
    if (A.stats && ((uintptr_t)status & 7)) return SS_ERR_INVALID_ARG;
    A.P.seed = seed; A.P.counter = counter; A.P.tick_limit = tick_limit; A.P.reward_mode = reward_mode; A.P.auto_reset = 1;
    A.P.reset_mode = reset_mode; A.n_ticks = 1;
    const dim3 grid(blocks_for(2 * n_envs, kBlockPP));
    if (blocks) {
        B.opp_actions = (const float2 *)opp_actions; B.opp_obs = (float4 *)opp_obs_out; B.pool_stats = (unsigned long long *)pool_stats;
        if (speeds) {
            A.speeds = speeds;
            // the staging tile is step_kernel's: the same carve-out
            static bool configured = false;
            if (!configured) {
                cudaFuncSetAttribute(pool_step_speeds_kernel<false>, cudaFuncAttributePreferredSharedMemoryCarveout, 50);
                cudaFuncSetAttribute(pool_step_speeds_kernel<true>, cudaFuncAttributePreferredSharedMemoryCarveout, 50);
                configured = true;
            }
            const dim3 grid_env(blocks_for(n_envs, kBlock));
            if ((A.stats ? sslaunch::launch(pool_step_speeds_kernel<true>, grid_env, dim3(kBlock), 0, (cudaStream_t)stream, A, B)
                         : sslaunch::launch(pool_step_speeds_kernel<false>, grid_env, dim3(kBlock), 0, (cudaStream_t)stream, A, B)) !=
                cudaSuccess)
                return SS_ERR_CUDA;
            return SS_OK;
        }
        if ((A.stats ? sslaunch::launch(step_pp_obs_kernel<true, BlockPoolRows>, grid, dim3(kBlockPP), 0, (cudaStream_t)stream, A, B)
                     : sslaunch::launch(step_pp_obs_kernel<false, BlockPoolRows>, grid, dim3(kBlockPP), 0, (cudaStream_t)stream, A, B)) !=
            cudaSuccess)
            return SS_ERR_CUDA;
        return SS_OK;
    }
    PoolRows R{n_envs - pool_envs, pool_envs > 0 ? pool_envs / n_opponents : 2, (const float2 *)opp_actions, (float4 *)opp_obs_out,
               pool_envs > 0 ? (unsigned long long *)pool_stats : nullptr};
    if ((A.stats ? sslaunch::launch(step_pp_obs_kernel<true, PoolRows>, grid, dim3(kBlockPP), 0, (cudaStream_t)stream, A, R)
                 : sslaunch::launch(step_pp_obs_kernel<false, PoolRows>, grid, dim3(kBlockPP), 0, (cudaStream_t)stream, A, R)) != cudaSuccess)
        return SS_ERR_CUDA;
    return SS_OK;
}

int ss_env_step_pool(void *state, int64_t n_envs, int64_t pool_envs, int n_opponents, const float *actions,
                     const float *opp_actions, float *obs_out, float *obs_out2, float *reward_out, uint8_t *done_rows_out,
                     float *opp_obs_out, uint8_t *done_out, uint8_t *winner_out, int reward_mode, int64_t tick_limit,
                     int reset_mode, uint64_t seed, uint64_t counter, uint32_t *status, int flags, uint64_t *pool_stats,
                     void *stream) {
    return step_pool(state, n_envs, pool_envs, n_opponents, actions, opp_actions, obs_out, obs_out2, reward_out, done_rows_out,
                     opp_obs_out, done_out, winner_out, reward_mode, tick_limit, reset_mode, seed, counter, status, flags, pool_stats,
                     false, nullptr, nullptr, stream);
}

int ss_env_step_pool_blocks(void *state, int64_t n_envs, int64_t pool_envs, int n_opponents, const float *actions,
                            const float *opp_actions, float *obs_out, float *obs_out2, float *reward_out, uint8_t *done_rows_out,
                            float *opp_obs_out, uint8_t *done_out, uint8_t *winner_out, int reward_mode, int64_t tick_limit,
                            int reset_mode, uint64_t seed, uint64_t counter, uint32_t *status, int flags, uint64_t *pool_stats,
                            const int64_t *opp_envs, void *stream) {
    return step_pool(state, n_envs, pool_envs, n_opponents, actions, opp_actions, obs_out, obs_out2, reward_out, done_rows_out,
                     opp_obs_out, done_out, winner_out, reward_mode, tick_limit, reset_mode, seed, counter, status, flags, pool_stats,
                     true, opp_envs, nullptr, stream);
}

int ss_env_step_pool_speeds(void *state, int64_t n_envs, int64_t pool_envs, int n_opponents, const float *actions,
                            const float *opp_actions, float *obs_out, float *obs_out2, float *reward_out, uint8_t *done_rows_out,
                            float *opp_obs_out, uint8_t *done_out, uint8_t *winner_out, int reward_mode, int64_t tick_limit,
                            int reset_mode, uint64_t seed, uint64_t counter, uint32_t *status, int flags, uint64_t *pool_stats,
                            const int64_t *opp_envs, const void *speeds, void *stream) {
    if (!speeds || ((uintptr_t)speeds & 15)) return SS_ERR_INVALID_ARG;
    return step_pool(state, n_envs, pool_envs, n_opponents, actions, opp_actions, obs_out, obs_out2, reward_out, done_rows_out,
                     opp_obs_out, done_out, winner_out, reward_mode, tick_limit, reset_mode, seed, counter, status, flags, pool_stats,
                     true, opp_envs, speeds, stream);
}

int ss_pool_restart(void *state, int64_t n_envs, int64_t pool_envs, int n_opponents, const int64_t *opp_envs, int reset_mode,
                    uint64_t seed, uint64_t counter, float *obs, float *opp_obs, uint32_t *status, void *stream) {
    (void)status;          // a restart ends no game: nothing is counted or flagged
    if (!state || !obs || !opp_obs || n_envs <= 0 || pool_envs <= 0 || pool_envs > n_envs) return SS_ERR_INVALID_ARG;
    if (reset_mode != SS_RESET_FIXED && reset_mode != SS_RESET_RANDOM) return SS_ERR_INVALID_ARG;
    if (((uintptr_t)state | (uintptr_t)obs | (uintptr_t)opp_obs) & 15) return SS_ERR_INVALID_ARG;
    BlockPoolRows B{};
    if (!pool_block_table(n_envs, pool_envs, n_opponents, opp_envs, B)) return SS_ERR_INVALID_ARG;
    B.opp_obs = (float4 *)opp_obs;
    pool_restart_kernel<<<blocks_for(2 * pool_envs, kBlockPP), kBlockPP, 0, (cudaStream_t)stream>>>(state, n_envs, (float4 *)obs,
                                                                                                  reset_mode, seed, counter, B);
    return check_launch();
}

int ss_env_step_tiles(void *state, int64_t n_envs, const float *actions, float *obs_out, float *obs_out2,
                      float *reward_out, uint8_t *done_out, uint8_t *done_rows_out, uint8_t *winner_out,
                      int reward_mode, int64_t tick_limit, int reset_mode, uint64_t seed, uint64_t counter,
                      uint32_t *status, int flags, int *tile_ready, int64_t units, int grid_fwd, void *stream) {
    if (!state || !actions || !obs_out || n_envs <= 0 || !tile_ready || units <= 0 || grid_fwd <= 0) return SS_ERR_INVALID_ARG;
    if (units < (2 * n_envs + 127) / 128) return SS_ERR_INVALID_ARG;      // (a noisy forward pads its last group with empty tiles)
    if (reward_mode != SS_REWARD_NONE && reward_mode != SS_REWARD_LOOKING && reward_mode != SS_REWARD_TERMINAL) return SS_ERR_INVALID_ARG;
    if (reset_mode != SS_RESET_FIXED && reset_mode != SS_RESET_RANDOM) return SS_ERR_INVALID_ARG;
    if (((uintptr_t)state | (uintptr_t)actions | (uintptr_t)obs_out | (uintptr_t)obs_out2) & 15) return SS_ERR_INVALID_ARG;
    TilesArgs T{};
    StepArgs &A = T.S;
    A.state = state; A.n = n_envs; A.actions = (const float4 *)actions; A.obs_out = (float4 *)obs_out; A.obs_out2 = (float4 *)obs_out2;
    A.reward_out = (float2 *)reward_out; A.done_out = done_out; A.winner_out = winner_out; A.done_rows_out = (uint16_t *)done_rows_out;
    A.status = status;
    A.stats = (status && (flags & SS_STEP_EPISODE_STATS)) ? reinterpret_cast<unsigned long long *>(status) + 1 : nullptr;
    if (A.stats && ((uintptr_t)status & 7)) return SS_ERR_INVALID_ARG;
    A.P.seed = seed; A.P.counter = counter; A.P.tick_limit = tick_limit; A.P.reward_mode = reward_mode; A.P.auto_reset = 1;
    A.P.reset_mode = reset_mode; A.n_ticks = 1;
    T.tile_ready = tile_ready; T.units = units; T.grid_fwd = grid_fwd;
    // The forward kernel needs the SM's shared-memory carve-out at its maximum (222 KB per CTA), and an SM cannot change its
    // carve-out while anything is resident on it: this kernel, which uses no shared memory at all, must ask for the same
    // carve-out, or the first of the two to reach an SM locks the other out until it exits (measured: every tile timed out).
    static bool configured = false;
    if (!configured) {
        cudaFuncSetAttribute(step_pp_tiles_kernel<true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        cudaFuncSetAttribute(step_pp_tiles_kernel<false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        configured = true;
    }
    const int64_t steps = (units + grid_fwd - 1) / grid_fwd + 1;          // tiles per forward CTA, rounded up
    const unsigned grid = (unsigned)(steps * 4 * grid_fwd);
    if (A.stats) step_pp_tiles_kernel<true><<<grid, 32, 0, (cudaStream_t)stream>>>(T);
    else step_pp_tiles_kernel<false><<<grid, 32, 0, (cudaStream_t)stream>>>(T);
    return check_launch();
}

int ss_env_step(void *state, int64_t n_envs, const float *actions, float *obs_out,
                float *reward_out, uint8_t *done_out, uint8_t *winner_out,
                int n_ticks, int reward_mode, int64_t tick_limit, int auto_reset,
                int reset_mode, uint64_t seed, uint64_t counter, const void *speeds,
                uint32_t *status, int flags, void *stream) {
    return ss_env_step_ring(state, n_envs, actions, obs_out, nullptr, reward_out, done_out, nullptr, winner_out, n_ticks,
                            reward_mode, tick_limit, auto_reset, reset_mode, seed, counter, speeds, status, flags, stream);
}

int ss_env_step_packed(void *state, int64_t n_envs, const float *actions, uint8_t *packed_out, int n_ticks,
                       int64_t tick_limit, int auto_reset, int reset_mode, uint64_t seed, uint64_t counter,
                       uint32_t *status, void *stream) {
    if (!state || !actions || !packed_out || n_envs <= 0 || n_ticks <= 0) return SS_ERR_INVALID_ARG;
    if (auto_reset && reset_mode != SS_RESET_FIXED && reset_mode != SS_RESET_RANDOM) return SS_ERR_INVALID_ARG;
    if (((uintptr_t)state | (uintptr_t)actions) & 15) return SS_ERR_INVALID_ARG;
    if (2 * n_envs * ((int64_t)n_ticks + 2) >= (int64_t)0x7fffffff) return SS_ERR_INVALID_ARG;
    StepArgs A{};
    A.state = state; A.n = n_envs; A.actions = (const float4 *)actions; A.packed_out = packed_out; A.status = status;
    A.P.seed = seed; A.P.counter = counter; A.P.tick_limit = tick_limit; A.P.reward_mode = SS_REWARD_TERMINAL;
    A.P.auto_reset = auto_reset ? 1 : 0; A.P.reset_mode = reset_mode; A.n_ticks = n_ticks;
    return launch_step_pp<OUT_PACKED>(A, n_envs, (cudaStream_t)stream);
}

int ss_env_features(const void *state, int64_t n_envs, double *feat_out, double *obs_out,
                    int32_t *general_out, const void *speeds, void *stream) {
    if (!state || n_envs <= 0) return SS_ERR_INVALID_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    if (speeds) features_kernel<true><<<blocks_for(n_envs, 128), 128, 0, st>>>(state, n_envs, feat_out, obs_out, general_out, speeds);
    else features_kernel<false><<<blocks_for(n_envs, 128), 128, 0, st>>>(state, n_envs, feat_out, obs_out, general_out, speeds);
    return check_launch();
}

int ss_env_export(const void *state, int64_t n_envs, int64_t first, int64_t count,
                  int32_t *ints, double *rots, void *stream) {
    if (!state || !ints || !rots || first < 0 || count <= 0 || first + count > n_envs) return SS_ERR_INVALID_ARG;
    export_kernel<<<blocks_for(count, 128), 128, 0, (cudaStream_t)stream>>>(state, n_envs, first, count, ints, rots);
    return check_launch();
}

int ss_env_import(void *state, int64_t n_envs, int64_t first, int64_t count,
                  const int32_t *ints, const double *rots, void *stream) {
    if (!state || !ints || !rots || first < 0 || count <= 0 || first + count > n_envs) return SS_ERR_INVALID_ARG;
    import_kernel<<<blocks_for(count, 128), 128, 0, (cudaStream_t)stream>>>(state, n_envs, first, count, ints, rots);
    return check_launch();
}

int ss_env_apply(void *state, int64_t n_envs, int64_t env, int player, int op, double value,
                 const void *speeds, uint32_t *status, void *stream) {
    if (!state || env < 0 || env >= n_envs || player < 0 || player > 1 || op < 0 || op > SS_OP_GAME_TICK)
        return SS_ERR_INVALID_ARG;
    apply_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(state, n_envs, env, player, op, value, speeds, status);
    return check_launch();
}

int ss_env_step_match(void *state, int64_t n_envs, int64_t split, const float *actions, float *obs_out, int64_t tick_limit,
                      const void *speeds, uint32_t *status, void *stream) {
    if (!state || !actions || !obs_out || n_envs <= 0 || split < 0 || split > n_envs || tick_limit <= 0) return SS_ERR_INVALID_ARG;
    if ((((uintptr_t)state | (uintptr_t)obs_out | (uintptr_t)speeds) & 15) || ((uintptr_t)actions & 7) || ((uintptr_t)status & 3))
        return SS_ERR_INVALID_ARG;
    MatchStepArgs A{state, n_envs, split, tick_limit, (const float2 *)actions, (float4 *)obs_out, speeds, status};
    cudaStream_t st = (cudaStream_t)stream;
    if (speeds) match_step_kernel<true, SplitSeats><<<blocks_for(n_envs, kBlock), kBlock, 0, st>>>(A);
    else match_step_kernel<false, SplitSeats><<<blocks_for(n_envs, kBlock), kBlock, 0, st>>>(A);
    return check_launch();
}

int ss_match_summary(const void *state, int64_t n_envs, int64_t split, int64_t tick_limit, uint64_t *out, void *stream) {
    if (!state || !out || n_envs <= 0 || split < 0 || split > n_envs || tick_limit <= 0) return SS_ERR_INVALID_ARG;
    if (((uintptr_t)state & 15) || ((uintptr_t)out & 7)) return SS_ERR_INVALID_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    if (cudaMemsetAsync(out, 0, SS_MATCH_STATS * sizeof(uint64_t), st) != cudaSuccess) return SS_ERR_CUDA;
    match_summary_kernel<<<blocks_for(n_envs, 256), 256, 0, st>>>(state, n_envs, split, tick_limit, (unsigned long long *)out);
    return check_launch();
}

int ss_env_step_seated(void *state, int64_t n_envs, const void *seat_rows, int64_t n_rows, const float *actions, float *obs_out,
                       int64_t tick_limit, const void *speeds, uint32_t *status, void *stream) {
    if (!state || !seat_rows || !actions || !obs_out || n_envs <= 0 || n_rows <= 0 || n_rows > INT32_MAX || tick_limit <= 0)
        return SS_ERR_INVALID_ARG;
    if ((((uintptr_t)state | (uintptr_t)obs_out | (uintptr_t)speeds) & 15) || (((uintptr_t)actions | (uintptr_t)seat_rows) & 7) ||
        ((uintptr_t)status & 3))
        return SS_ERR_INVALID_ARG;
    SeatedStepArgs A{state, n_envs, n_rows, tick_limit, (const int2 *)seat_rows, (const float2 *)actions, (float4 *)obs_out, speeds, status};
    cudaStream_t st = (cudaStream_t)stream;
    if (speeds) match_step_kernel<true, TableSeats><<<blocks_for(n_envs, kBlock), kBlock, 0, st>>>(A);
    else match_step_kernel<false, TableSeats><<<blocks_for(n_envs, kBlock), kBlock, 0, st>>>(A);
    return check_launch();
}

int ss_league_summary(const void *state, int64_t n_envs, const uint8_t *seat_policy, int n_policies, int64_t tick_limit, uint64_t *out,
                      void *stream) {
    if (!state || !seat_policy || !out || n_envs <= 0 || n_policies < 2 || n_policies > SS_LEAGUE_MAX_POLICIES || tick_limit <= 0)
        return SS_ERR_INVALID_ARG;
    if (((uintptr_t)state & 15) || ((uintptr_t)seat_policy & 1) || ((uintptr_t)out & 7)) return SS_ERR_INVALID_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t bytes = (size_t)n_policies * n_policies * 8 * sizeof(uint64_t);
    if (cudaMemsetAsync(out, 0, bytes, st) != cudaSuccess) return SS_ERR_CUDA;
    league_summary_kernel<<<blocks_for(n_envs, 256), 256, 0, st>>>(state, n_envs, seat_policy, n_policies, tick_limit,
                                                                    (unsigned long long *)out);
    return check_launch();
}

}  // extern "C"
