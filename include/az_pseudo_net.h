/*
 * az_pseudo_net.h — deterministic pseudo policy/value "network" used ONLY for MCTS
 * parity testing.  north_star asks for bit-exact visit counts "given identical
 * network outputs"; a real fp32 forward differs in the last bits between a CPU and a
 * GPU, so the search-parity tests plug this exactly-representable evaluator into
 * both the compiled reference (oracle/ref/ref_shim.cpp), the C oracle
 * (oracle/risk_oracle.c) and the CUDA search (evaluator = AZ_EVAL_PSEUDO).
 *
 * Every output is a small dyadic rational, so masking, summation and the
 * normalising division (NNOutputData::normalize,
 * /root/reference/src/risk_game/player/alpha_zero/neural_network/alphazero_nn_data.cpp:3-27)
 * round identically everywhere; the 16-level policy produces frequent exact prior
 * ties, which is what exercises the tie-breaking rules of PUCT.
 *
 * Inputs are fields present both in the game state and in the reference's
 * NNInputData (alphazero_nn_data.h:81-103): the 42 land bytes (army | owner << 6),
 * side to move, round and phase.
 */
#ifndef AZ_PSEUDO_NET_H
#define AZ_PSEUDO_NET_H

#include <stdint.h>

#if defined(__CUDACC__)
#define AZ_PN_HD __host__ __device__ __forceinline__
#else
#define AZ_PN_HD static inline
#endif

AZ_PN_HD uint64_t az_pn_mix(uint64_t x)
{
    x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ull;
    x ^= x >> 27; x *= 0x94D049BB133111EBull;
    x ^= x >> 31;
    return x;
}

AZ_PN_HD uint64_t az_pn_key(const uint8_t* land42, int cur, int round, int phase)
{
    uint64_t h = 0x9E3779B97F4A7C15ull ^ (uint64_t)(uint32_t)cur ^ ((uint64_t)(uint32_t)round << 8) ^
                 ((uint64_t)(uint32_t)phase << 24);
    for (int i = 0; i < 42; ++i) h = (h ^ land42[i]) * 0x100000001B3ull;
    return az_pn_mix(h);
}

AZ_PN_HD float az_pn_policy(uint64_t key, int move)
{
    uint64_t m = az_pn_mix(key + 0x9E3779B97F4A7C15ull * (uint64_t)(move + 1));
    return (float)((int)(m & 15u) + 1) * (1.0f / 16.0f);
}

AZ_PN_HD float az_pn_value(uint64_t key)
{
    uint64_t m = az_pn_mix(key ^ 0xD6E8FEB86659FD93ull);
    return (float)((int)((m >> 7) & 255u) - 128) * (1.0f / 128.0f);
}

/* component k (0..5) of the six-seat value vector (SIXPLAYER.md §2): the value of seat (cur + k) % 6.  Component 0 is
   az_pn_value; the others come from their own mix, dyadic like the rest, and their sum is not constrained. */
AZ_PN_HD float az_pn_value6(uint64_t key, int k)
{
    if (k == 0) return az_pn_value(key);
    uint64_t m = az_pn_mix((key ^ 0xD6E8FEB86659FD93ull) + 0xA0761D6478BD642Full * (uint64_t)k);
    return (float)((int)((m >> 7) & 255u) - 128) * (1.0f / 128.0f);
}

#endif /* AZ_PSEUDO_NET_H */
