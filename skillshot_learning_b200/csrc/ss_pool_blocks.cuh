// ss_pool_blocks.cuh -- the block table of a pool (include/skillshot_b200.h, "training against a pool"), host only:
// opponent k owns the b_k consecutive pool envs from S + B_k, B_k = b_0 + ... + b_{k-1}.
#pragma once
#include <stdint.h>

#include "../../include/skillshot_b200.h"

namespace sspool {

// start[0..K] = B_0 .. B_K from opp_envs [K] (NULL: M / K each).  false when K is out of range or a size is odd, below 2,
// or the sizes do not sum to M.
inline bool block_starts(int64_t M, int K, const int64_t *opp_envs, int64_t *start) {
    if (K < 1 || K > SS_LEAGUE_MAX_POLICIES || M <= 0) return false;
    if (!opp_envs && M % (2 * K) != 0) return false;
    start[0] = 0;
    for (int k = 0; k < K; ++k) {
        const int64_t b = opp_envs ? opp_envs[k] : M / K;
        if (b < 2 || (b & 1) || b > M - start[k]) return false;
        start[k + 1] = start[k] + b;
    }
    return start[K] == M;
}

}  // namespace sspool
