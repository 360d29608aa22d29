// ss_env_pp.cuh -- one SkillshotGame tick WITH its observation, one thread per PLAYER (device only).
//
// Lanes 2i and 2i+1 of a warp are players 1 and 2 of env i (see step_pp_kernel in ss_env.cu for the physics-only fused
// form).  This header holds the single-tick form that also produces the 12-float observation and the shaped reward: the
// rollout's env step.  It is written to be inlined into TWO places and to give the same bits in both:
//   * step_pp_obs_kernel (ss_env.cu), the stand-alone env step of a rollout tick;
//   * the output stage of the tensor-core actor forward (ss_mlp_tc.cu, ss_actor_forward_step_tc), where the lane that has
//     just computed a player's action plays that player's tick on the spot -- no action round trip, no second kernel.
// Those translation units are compiled with different floating-point contraction settings, so every multiply / add /
// subtract here goes through the explicit round-to-nearest wrappers of ss_env_core.cuh (mul / add / sub) and every fused
// multiply-add is an explicit fma(): nothing is left for the compiler to contract.  The arithmetic is, expression for
// expression, that of tick_env<OBS = true, CARRY = true> / fast_view / fast_obs in ss_env_core.cuh (the one-thread-per-env
// kernels), so both forms produce bit-identical states, observations and rewards.
//
// All 32 lanes of the warp must call lane_obs_tick together (one shuffle, one ballot).
#pragma once
#include "ss_env_core.cuh"

namespace sspp {

using namespace ss;

struct LaneState {
    double rot, qrot;                       // Player.rotation, Projectile.rotation
    int px, py, qx, qy, cd, age, valid;     // this player and its projectile
    int live, winner, ticks;                // the env's, replicated in both lanes
};

__device__ __forceinline__ double i2d(int x) { return __dsub_rn(__hiloint2double(0x43300000, x), 4503599627370496.0); }   // exact, 0 <= x < 2^32
__device__ __forceinline__ int d2i_rn(double v) { return __double2loint(__dadd_rn(v, 6755399441055744.0)); }              // == cvt.rni, |v| < 2^31
__device__ __forceinline__ bool nan2(double a, double b) {
    int p;
    asm("{ .reg .pred q; setp.nan.f64 q, %1, %2; selp.s32 %0, 1, 0, q; }" : "=r"(p) : "d"(a), "d"(b));
    return p != 0;
}
__device__ __forceinline__ float clipf_nan(float v) {        // Player.py:36-37, 60-61; a NaN falls through
    float r;
    asm("max.NaN.f32 %0, %1, 0fBF800000;" : "=f"(r) : "f"(v));
    asm("min.NaN.f32 %0, %1, 0f3F800000;" : "=f"(r) : "f"(r));
    return r;
}

// this lane's half of the env's packed state (include/skillshot_b200.h); gl = 2 * env + player
__device__ __forceinline__ void lane_load(const char *base, int64_t n, int64_t gl, LaneState &L) {
    const int P = (int)(gl & 1);
    const int64_t env = gl >> 1;
    L.rot = ((const double *)base)[gl];
    L.qrot = ((const double *)(base + 16 * n))[gl];
    const int4 a = ((const int4 *)(base + 32 * n))[env], b = ((const int4 *)(base + 48 * n))[env];
    const uint32_t pp = (uint32_t)a.x >> (16 * P), qq = (uint32_t)a.y >> (16 * P), f = (uint32_t)b.w;
    L.px = pp & 255; L.py = (pp >> 8) & 255; L.qx = qq & 255; L.qy = (qq >> 8) & 255;
    L.cd = P ? a.w : a.z; L.age = P ? b.y : b.x; L.ticks = b.z;
    L.valid = (f >> P) & 1; L.live = (f >> 2) & 1; L.winner = (f >> 4) & 3;
}
// v_other = the partner lane's valid bit (the env's flag word holds both)
__device__ __forceinline__ void lane_store(char *base, int64_t n, int64_t gl, const LaneState &L, int v_other) {
    const int P = (int)(gl & 1);
    const int64_t env = gl >> 1;
    ((double *)base)[gl] = L.rot;
    ((double *)(base + 16 * n))[gl] = L.qrot;
    char *ia = base + 32 * n + env * 16, *ib = base + 48 * n + env * 16;
    ((uint16_t *)ia)[P] = (uint16_t)(L.px | (L.py << 8));
    ((uint16_t *)ia)[2 + P] = (uint16_t)(L.qx | (L.qy << 8));
    ((int *)ia)[2 + P] = L.cd;
    ((int *)ib)[P] = L.age;
    if (!P) ((int2 *)ib)[1] = make_int2(L.ticks, L.valid | (v_other << 1) | (L.live << 2) | (L.winner << 4));
}

// get_dist_line_point / get_dist_point_point / check_future_collision of one player's view (fast_view of
// ss_env_core.cuh, same expressions); (ox, oy) = the opponent's position
struct LaneView { double player_path_dist, proj_path_dist, player_dist, proj_dist; int future_collision; };

__device__ __forceinline__ LaneView lane_view(const LaneState &L, int ox, int oy, double ps, double pc, double qs, double qc) {
    LaneView v;
    const int dx = ox - L.px, dy = oy - L.py;
    v.player_path_dist = fabs(sub(mul(pc, (double)dx), mul(ps, (double)dy)));
    v.player_dist = (double)sqrtf((float)(dx * dx + dy * dy));
    const int ex = ox - L.qx, ey = oy - L.qy;
    v.proj_path_dist = fabs(sub(mul(qc, (double)ex), mul(qs, (double)ey)));
    v.proj_dist = (double)sqrtf((float)(ex * ex + ey * ey));
    int fc = 0;
    if (L.valid) {                                       // check_future_collision, SkillshotGame.py:96-113
        const int d0 = ex, d1 = d0 + kPlayerSize, l = ey, h = l + kPlayerSize;
        if (fmin(fabs(qs), fabs(qc)) < 1e-6) {
            // axis-aligned shots keep the reference's own expression with g = tan(-rot + pi/2)
            const double g = tan(add(-L.qrot, kHalfPi));
            const double yint = sub((double)L.qy, mul(g, (double)L.qx));
            const double lo = (double)oy, hi = (double)(oy + kPlayerSize);
            const double v0 = add(mul(g, (double)ox), yint);
            const double v1 = add(mul(g, (double)(ox + kPlayerSize)), yint);
            fc = ((lo <= v0 && v0 <= hi) || (lo <= v1 && v1 <= hi)) ? 1 : 0;
        } else {
            const double ls = mul((double)l, qs), hs = mul((double)h, qs);
            const double lo = fmin(ls, hs), hi = fmax(ls, hs);
            const double c0 = mul(qc, (double)d0), c1 = mul(qc, (double)d1);
            fc = ((lo <= c0 && c0 <= hi) || (lo <= c1 && c1 <= hi)) ? 1 : 0;
        }
    }
    v.future_collision = fc;
    return v;
}

__device__ __forceinline__ double mod2_fast(double v) { return sub(v, mul(2.0, floor(mul(v, 0.5)))); }   // Python float % 2

// prepare_states (SkillshotLearner.py:525-539): the player's 12 floats as three float4 (fast_obs of ss_env_core.cuh)
__device__ __forceinline__ void lane_obs(const LaneState &L, const LaneView &v, float4 (&o)[3]) {
    constexpr float kInvBoard = 1.0f / 250.0f, kInvCooldown = 1.0f / 15.0f;
    o[0] = make_float4((float)mul(v.player_path_dist, kInvMaxDist), (float)mul(v.player_dist, kInvMaxDist),
                       (float)L.px * kInvBoard, (float)L.py * kInvBoard);
    o[1] = make_float4((float)mul(mod2_fast(L.rot), kHalfPiSq), (float)L.cd * kInvCooldown,
                       (float)mul(v.proj_dist, kInvMaxDist), (float)L.qx * kInvBoard);
    o[2] = make_float4((float)L.qy * kInvBoard, (float)mul(mod2_fast(L.qrot), kHalfPiSq),
                       (float)mul(v.proj_path_dist, kInvMaxDist), (float)v.future_collision);
}

struct LaneTrig { double ps, pc, qs, qc; };     // sin / cos of the player's and of the projectile's rotation (pre-tick)
__device__ __forceinline__ void lane_trig(const LaneState &L, LaneTrig &T) {
    sincos_d(L.rot, &T.ps, &T.pc);
    sincos_d(L.qrot, &T.qs, &T.qc);
}

// one finished game into the episode statistics block (SS_STEP_EPISODE_STATS, include/skillshot_b200.h)
__device__ __forceinline__ void count_episode_pp(unsigned long long *stats, int len, int winner, int tick_limit) {
    const int width = tick_limit > 0 ? (tick_limit + 63) / 64 : 32;
    atomicAdd(stats + 0, 1ull);
    atomicAdd(stats + (winner == 1 ? 1 : winner == 2 ? 2 : 3), 1ull);
    atomicAdd(stats + 4, (unsigned long long)len);
    atomicAdd(stats + 8 + min(63, len / width), 1ull);
}

// game_reset (SkillshotGame.py:168-169) of this lane's player: the start state, and in (ox, oy) the partner's start
// position.  SS_RESET_RANDOM draws from Philox4x32-10(key = seed, counter = (env, tick_counter)), as ss_env_reset does.
// The same statements as the auto-reset in lane_obs_tick below, which keeps its own copy: calling this helper there moves
// the register allocation of the kernels that inline it.
__device__ __forceinline__ void lane_reset(LaneState &L, int P, uint64_t env, uint64_t tick_counter, int reset_mode, uint64_t seed,
                                           int &ox, int &oy) {
    int x = P ? 200 : 50, y = x;
    ox = P ? 50 : 200; oy = ox;
    if (reset_mode == SS_RESET_RANDOM) {
        const U4 u = philox4x32_10(U4{(uint32_t)env, (uint32_t)(env >> 32), (uint32_t)tick_counter, (uint32_t)(tick_counter >> 32)},
                                   (uint32_t)seed, (uint32_t)(seed >> 32));
        x = rand_coord(P ? u.z : u.x); y = rand_coord(P ? u.w : u.y);
        ox = rand_coord(P ? u.x : u.z); oy = rand_coord(P ? u.y : u.w);
    }
    L.px = x; L.py = y; L.rot = 0.0; L.qx = 0; L.qy = 0; L.qrot = 0.0; L.cd = 0; L.age = 0; L.valid = 0;
    L.ticks = 0; L.live = 1; L.winner = 0;
}

struct LaneTickOut {
    float4 obs[3];          // the observation the actor sees next (post-reset if the game restarted)
    float reward;           // of the post-tick state
    int done, winner;       // of the post-tick state, before a reset
    int episode_len;        // >= 0: a game ended on this tick after this many ticks (episode statistics), else -1
};

// One model_train tick (SkillshotLearner.py:304-315) for this lane's player: do_actions, game_tick, reward, auto-reset,
// next observation.  reward_mode: SS_REWARD_NONE / LOOKING / TERMINAL (the `simple` shaper stays on the per-env kernel).
// T = lane_trig(L) of the pre-tick state: it does not depend on the action, so a caller that is still waiting for the
// action (the fused forward kernel) computes it ahead.
__device__ __forceinline__ void lane_obs_tick(LaneState &L, const LaneTrig &T, float a_move, float a_look, const TickParams &TP,
                                              uint64_t env, uint64_t tick_counter, int lane, int P, uint32_t &status,
                                              LaneTickOut &out) {
    const int limit = TP.tick_limit > 0 ? (int)min((int64_t)0x7fffffff, TP.tick_limit) : 0x7fffffff;
    double ps = T.ps, pc = T.pc, qs = T.qs, qc = T.qc;
    const int was_live = L.live;
    const int ticks_before = (!L.live || L.ticks >= limit) ? -1 : L.ticks;
    // ---- do_actions (SkillshotLearner.py:206-213): move with the rotation BEFORE the turn, turn, shoot ----
    const double speed = (double)clipf_nan(a_move), angle = (double)clipf_nan(a_look);
    const double vx = sub(i2d(L.px), mul(mul(ps, 3.0), speed));       // Player.py:63
    const double vy = sub(i2d(L.py), mul(mul(pc, 3.0), speed));       // Player.py:64
    if (nan2(vx, vy)) {
        status |= kStatusNaN;                                         // int(round(nan)) raises
    } else {
        const int nx = d2i_rn(vx), ny = d2i_rn(vy);
        if ((unsigned)nx <= (unsigned)(kBoard - kPlayerSize) && (unsigned)ny <= (unsigned)(kBoard - kPlayerSize)) { L.px = nx; L.py = ny; }
    }
    L.rot = fma(angle, 0.25, L.rot);                                  // rot + angle * 0.25: the product is exact
    sincos_d(L.rot, &ps, &pc);
    if (L.cd <= 0) {                                                  // Player.move_shoot_projectile, Player.py:78-89
        L.qx = L.px; L.qy = L.py; L.qrot = L.rot; qs = ps; qc = pc;
        L.valid = 1; L.cd = 15; L.age = 0;
    }
    // ---- game_tick (SkillshotGame.py:115-122), gated on game_live ----
    if (L.live) {
        L.ticks += 1;
        double wx = sub(i2d(L.qx), mul(qs, 5.0));                     // Projectile.py:40
        double wy = sub(i2d(L.qy), mul(qc, 5.0));                     // Projectile.py:41
        bool inb = false;
        if (nan2(wx, wy)) {
            status |= kStatusNaN;
        } else {
            const int mx = d2i_rn(wx), my = d2i_rn(wy);
            inb = (unsigned)mx <= (unsigned)(kBoard - kProjSize) && (unsigned)my <= (unsigned)(kBoard - kProjSize);
            if (L.valid && inb) { L.qx = mx; L.qy = my; }
        }
        if (!(L.valid && inb)) L.valid = 0;                           // Projectile.py:43-47
        L.cd -= 1; L.age += 1;                                        // Projectile.py:52-53
    }
    // my position and projectile to the partner lane, the partner's to me
    const uint32_t mine = (uint32_t)L.px | ((uint32_t)L.py << 8) | ((uint32_t)L.qx << 16) | ((uint32_t)L.qy << 24);
    const uint32_t theirs = __shfl_xor_sync(0xffffffffu, mine, 1);
    const uint32_t valids = __ballot_sync(0xffffffffu, L.valid != 0);
    int ox = theirs & 255, oy = (theirs >> 8) & 255;
    const int jx = (theirs >> 16) & 255, jy = theirs >> 24, jvalid = (valids >> (lane ^ 1)) & 1;
    // check_collision (SkillshotGame.py:58-94): my player against the OTHER player's projectile
    const bool in_x = (unsigned)(jx + kProjSize - L.px) <= (unsigned)kPlayerSize || (unsigned)(jx - L.px) <= (unsigned)kPlayerSize;
    const bool in_y = (unsigned)(jy - L.py) <= (unsigned)kPlayerSize || (unsigned)(jy - kProjSize - L.py) <= (unsigned)kPlayerSize;  // :72 minus
    const bool hit = was_live && jvalid && in_x && in_y;
    const uint32_t pair = (__ballot_sync(0xffffffffu, hit) >> (lane & 30)) & 3u;
    if (pair) { L.winner = (pair & 1u) ? 1 : 2; L.live = 0; }          // player 1 first; the first hit breaks
    out.done = (!L.live || L.ticks >= limit) ? 1 : 0;
    out.winner = L.winner;
    out.episode_len = (out.done && ticks_before >= 0) ? ticks_before + 1 : -1;
    const bool will_reset = TP.auto_reset && out.done;
    float r = 0.f;
    if (TP.reward_mode == SS_REWARD_TERMINAL && pair) r = (L.winner - 1 == P) ? -1.f : 1.f;      // readme.md:10
    if (TP.reward_mode == SS_REWARD_LOOKING && will_reset) {           // rare: the reward belongs to the pre-reset state
        const LaneView v = lane_view(L, ox, oy, ps, pc, qs, qc);
        r = (float)mul(v.player_path_dist, -0.004);                    // calculate_rewards_looking, SkillshotLearner.py:584
    }
    if (will_reset) {                                                  // game_reset (SkillshotGame.py:168-169)
        int x = P ? 200 : 50, y = x;
        ox = P ? 50 : 200; oy = ox;
        if (TP.reset_mode == SS_RESET_RANDOM) {
            const U4 u = philox4x32_10(U4{(uint32_t)env, (uint32_t)(env >> 32), (uint32_t)tick_counter, (uint32_t)(tick_counter >> 32)},
                                       (uint32_t)TP.seed, (uint32_t)(TP.seed >> 32));
            x = rand_coord(P ? u.z : u.x); y = rand_coord(P ? u.w : u.y);
            ox = rand_coord(P ? u.x : u.z); oy = rand_coord(P ? u.y : u.w);
        }
        L.px = x; L.py = y; L.rot = 0.0; L.qx = 0; L.qy = 0; L.qrot = 0.0; L.cd = 0; L.age = 0; L.valid = 0;
        L.ticks = 0; L.live = 1; L.winner = 0;
        ps = 0.0; pc = 1.0; qs = 0.0; qc = 1.0;                        // sin 0, cos 0
    }
    const LaneView v = lane_view(L, ox, oy, ps, pc, qs, qc);
    if (TP.reward_mode == SS_REWARD_LOOKING && !will_reset) r = (float)mul(v.player_path_dist, -0.004);
    out.reward = r;
    lane_obs(L, v, out.obs);
}

}  // namespace sspp
