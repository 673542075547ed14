// az_script6.cuh — the six-player scripted agent of SIXPLAYER.md §5 on the device (one thread per game), included by az_env6.cu for
// az_env6_script_actions and the scripted agents of k_arena6_advance.  The action is a pure function of the position (the game's
// AzGame6 masks and army column) and the rules: no randomness, no memory between plies.  The caller applies it with e6_move and the
// real-move dice of (seed, game, ply), like the random player's action.  The checker is oracle/risk6_script.c (same clauses, same
// tie-breaks, compared bit for bit).
#pragma once

#include "az_game6.cuh"

// continents NA, SA, EU, AF, AS, AU in index order (land/land_set.cpp:12-24)
__device__ __constant__ uint64_t E6_CONT_MASK[6] = { 0x1ffull, 0x1e00ull, 0xfe000ull, 0x3f00000ull, 0x3ffc000000ull, 0x3c000000000ull };
#define E6_SCRIPT_MARGIN 2              // an optional attack needs a source at least this many armies above its target
#define E6_SCRIPT_FORTIFY_BELOW 32      // a fortify target holds fewer armies than this (a full land takes nothing)

__device__ __forceinline__ int e6s_lowest(uint64_t m) { return __ffsll((long long)m) - 1; }

// the armies on the lands of N(l) & other
__device__ __forceinline__ int e6s_foreign_armies(const E6Ctx& c, const AzTables& T, int l, uint64_t other)
{
    int t = 0;
    for (uint64_t m = T.nbr[l] & other; m; m &= m - 1) t += (int)c.army.get(e6s_lowest(m));
    return t;
}

// strongest(t, S): the land of S among t's neighbours with the largest army, the first strict maximum in T.list6 order (the order
// e6_move picks an attack source in); -1 if no neighbour of t is in S
__device__ __forceinline__ int e6s_strongest(const E6Ctx& c, const AzTables& T, int t, uint64_t set)
{
    int best = -1, ba = 0;
    uint64_t lst = T.list6[t];
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        const int n = (int)(lst & 63u); lst >>= 6;
        if (n != 63 && ((set >> n) & 1ull)) {
            const int v = (int)c.army.get(n);
            if (v > ba) { ba = v; best = n; }
        }
    }
    return best;
}

// target(F): among the continents meeting F, the one with the fewest lands in other (ties: more lands of F, then the lower index);
// its land of F with the smallest army (ties: the lower index).  -1 if F is empty
__device__ __forceinline__ int e6s_target(const E6Ctx& c, uint64_t other, uint64_t f)
{
    uint64_t bc = 0;
    int bx = 0, bf = 0;
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        const uint64_t ck = E6_CONT_MASK[k];
        const int nf = __popcll(ck & f), nx = __popcll(ck & other);
        if (nf != 0 && (bc == 0 || nx < bx || (nx == bx && nf > bf))) { bc = ck; bx = nx; bf = nf; }
    }
    int t = -1, ta = AZ_ARMY_MAX + 1;
    for (uint64_t m = bc & f; m; m &= m - 1) {
        const int i = e6s_lowest(m), a = (int)c.army.get(i);
        if (a < ta) { ta = a; t = i; }
    }
    return t;
}

// the scripted action of the game's position (a land 0..41 or AZ_SKIP), always legal; the game must be running
__device__ __forceinline__ int e6_script_action(const E6Ctx& c, const AzTables& T, const AzRulesDev& r)
{
    const AzGame6& g = c.g;
    const uint64_t O = e6_own(g, g.cur), X = AZ_ALL_LANDS & ~O;
    if (g.phase == AZ_PH_MOBILIZATION) {
        const int from = (int)g.mob_from, to = (int)g.mob_to;
        return ((T.nbr[to] & X) == 0 && (T.nbr[from] & X) != 0) ? from : to;
    }
    const uint64_t valid = e6_valid(g, T, r), L = valid & AZ_ALL_LANDS;
    if (L == 0) return AZ_SKIP;
    if (g.phase == AZ_PH_ATTACK) {
        const int t = e6s_target(c, X, L);
        uint64_t cont = 0;
#pragma unroll
        for (int k = 0; k < 6; ++k) if ((E6_CONT_MASK[k] >> t) & 1ull) cont = E6_CONT_MASK[k];
        const uint64_t src = O & g.gt1;
        int best = -1, bm = 0, bin = 0, any = -1, am = 0;
        for (uint64_t m = L; m; m &= m - 1) {
            const int i = e6s_lowest(m), f = e6s_strongest(c, T, i, src);
            const int mg = (int)c.army.get(f) - (int)c.army.get(i), in = (int)((cont >> i) & 1ull);
            if (best < 0 || in > bin || (in == bin && mg > bm)) { best = i; bm = mg; bin = in; }
            if (any < 0 || mg > am) { any = i; am = mg; }
        }
        if (bm >= E6_SCRIPT_MARGIN || !(valid & AZ_SKIP_MASK)) return best;
        return am >= E6_SCRIPT_MARGIN ? any : AZ_SKIP;
    }
    if (g.phase == AZ_PH_FORTIFY) {                               // the source stays e6_move's rule
        int b = -1, bv = 0;
        for (uint64_t m = L & az_nbr_union(T, X); m; m &= m - 1) {
            const int i = e6s_lowest(m), a = (int)c.army.get(i);
            if (a >= E6_SCRIPT_FORTIFY_BELOW) continue;
            const int v = e6s_foreign_armies(c, T, i, X) - a;
            if (b < 0 || v > bv) { bv = v; b = i; }
        }
        return b >= 0 ? b : AZ_SKIP;
    }
    // SETUP, REINFORCEMENT
    const int t = e6s_target(c, X, az_nbr_union(T, O) & X);
    const int f = t >= 0 ? e6s_strongest(c, T, t, L) : -1;
    if (f >= 0) return f;
    int b = -1, bv = -1;
    for (uint64_t m = L; m; m &= m - 1) {
        const int i = e6s_lowest(m), v = e6s_foreign_armies(c, T, i, X);
        if (v > bv) { bv = v; b = i; }
    }
    return b;
}
