// ss_rng.cuh -- counter-based random draws of the learner path (Philox4x32-10).
//
// The reference draws from numpy's global MT19937 (SkillshotLearner.py:238,
// 263-265, 427); that stream is not part of the contract (SURVEY.md hard part
// 10), the distributions are.  Every draw here is a pure function of
// (seed, tag, a, b, counter), so results do not depend on grid shape, launch
// order or the number of GPUs, and a host restatement (tests/philox_ref.py) can
// reproduce them.
#pragma once
#include "ss_env_core.cuh"

namespace ss {

constexpr uint32_t kTagParamNoise = 1;   // model_act_param_noise, SkillshotLearner.py:260-265
constexpr uint32_t kTagDropout = 2;      // Dropout(0.2) during critic.fit, SkillshotLearner.py:105, 434
constexpr uint32_t kTagActionNoise = 3;  // model_act_action_noise, SkillshotLearner.py:238
constexpr uint32_t kTagReplay = 4;       // minibatch row choice (np.random.shuffle at :427 in the reference)
constexpr uint32_t kTagTargetNoise = 5;  // TD3 target policy smoothing (no reference code, DESIGN.md section 6.14)

SS_HD U4 draw4(uint64_t seed, uint32_t tag, uint32_t a, uint32_t b, uint64_t counter) {
    return philox4x32_10(U4{a, b, (uint32_t)counter, tag ^ (uint32_t)(counter >> 32)},
                         (uint32_t)seed, (uint32_t)(seed >> 32));
}

// uniform in (0, 1): 24 random bits, never 0 or 1
SS_HD float unit_open(uint32_t x) { return ((float)(x >> 8) + 0.5f) * (1.0f / 16777216.0f); }

// Box-Muller: two uniforms -> two N(0,1)
SS_HD void box_muller(uint32_t x, uint32_t y, float *z0, float *z1) {
    const float r = sqrtf(-2.0f * logf(unit_open(x)));
    float s, c;
#ifdef __CUDA_ARCH__
    sincosf(6.283185307179586f * unit_open(y), &s, &c);
#else
    s = sinf(6.283185307179586f * unit_open(y));
    c = cosf(6.283185307179586f * unit_open(y));
#endif
    *z0 = r * c;
    *z1 = r * s;
}

SS_HD void normal4(uint64_t seed, uint32_t tag, uint32_t a, uint32_t b, uint64_t counter, float *z) {
    const U4 u = draw4(seed, tag, a, b, counter);
    box_muller(u.x, u.y, z + 0, z + 1);
    box_muller(u.z, u.w, z + 2, z + 3);
}

// TD3 target policy smoothing of one row's target action, in place: a_m = clamp(a_m + clamp(sigma z_m, -c, c), -1, 1)
// with z_0, z_1 the first two normals of normal4(seed, kTagTargetNoise, row, row >> 32, counter) -- keyed by the GLOBAL
// row, as dropout is, so a shard of a batch draws what the whole batch draws.  Every TD3 target entry point applies it.
SS_HD void td3_smooth(uint64_t seed, uint64_t counter, int64_t row, float sigma, float clip, float *a0, float *a1) {
    float z[4];
    normal4(seed, kTagTargetNoise, (uint32_t)row, (uint32_t)((uint64_t)row >> 32), counter, z);
    *a0 = fminf(fmaxf(*a0 + fminf(fmaxf(sigma * z[0], -clip), clip), -1.0f), 1.0f);
    *a1 = fminf(fmaxf(*a1 + fminf(fmaxf(sigma * z[1], -clip), clip), -1.0f), 1.0f);
}

#ifdef __CUDACC__
// The same four normals from the hardware approximations (ex2 / lg2 / sin / cos units): within ~3e-6 of normal4.
// The angle is shifted into (-pi, pi), where __sincosf is accurate to 2^-21, and the signs are flipped back.
// For bulk parameter noise, where the draw is rounded to bf16 or scaled by sd * w afterwards.
__device__ __forceinline__ void normal4_fast(uint64_t seed, uint32_t tag, uint32_t a, uint32_t b, uint64_t counter, float *z) {
    const U4 u = draw4(seed, tag, a, b, counter);
    const float r0 = sqrtf(-2.0f * __logf(unit_open(u.x))), r1 = sqrtf(-2.0f * __logf(unit_open(u.z)));
    float s0, c0, s1, c1;
    __sincosf(6.283185307179586f * unit_open(u.y) - 3.14159265358979f, &s0, &c0);
    __sincosf(6.283185307179586f * unit_open(u.w) - 3.14159265358979f, &s1, &c1);
    z[0] = -r0 * c0; z[1] = -r0 * s0; z[2] = -r1 * c1; z[3] = -r1 * s1;
}
#endif

}  // namespace ss
