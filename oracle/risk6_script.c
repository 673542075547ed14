/*
 * TEST INFRASTRUCTURE — risk6_script.c: the six-player scripted agent of SIXPLAYER.md §5, the checker of az_env6_script_actions and
 * of the scripted agents of az_arena6_*.  The action is a pure function of the position and the rules: no randomness, no memory
 * between plies.  The chosen action is applied by r6_make_move with the real-move dice of (seed, game, ply), like the random player's.
 *
 * It builds on risk6_oracle.c unchanged (included here, so the legal-move mask and the neighbour tables are that file's own code).
 * Built as its own library by oracle/script6.py; never linked into the product.
 */
#include "risk6_oracle.c"

#define R6S_MARGIN 2            /* an optional attack needs a source at least this many armies above its target */
#define R6S_FORTIFY_BELOW 32    /* a fortify target holds fewer armies than this (RO_ARMY_MAX: a full land takes nothing) */

/* the armies on the lands of N(l) & other */
static int foreign_armies(const r6_state* s, int l, uint64_t other)
{
    int t = 0;
    uint64_t m = RO_NBR_MASK[l] & other;
    while (m) { int i = ctz(m); m &= m - 1; t += s->army[i]; }
    return t;
}

/* strongest(t, S): the land of S among t's neighbours with the largest army, the first strict maximum in RO_NBR_LIST order (the
   order r6_make_move picks an attack source in); -1 if no neighbour of t is in S */
static int strongest(const r6_state* s, int t, uint64_t set)
{
    int best = -1, ba = 0;
    for (int k = 0; k < 6 && RO_NBR_LIST[t][k] >= 0; ++k) {
        const int n = RO_NBR_LIST[t][k];
        if (((set >> n) & 1) && s->army[n] > ba) { ba = s->army[n]; best = n; }
    }
    return best;
}

/* target(F): among the continents meeting F, the one with the fewest lands in other (ties: more lands of F, then the lower index);
   its land of F with the smallest army (ties: the lower index).  -1 if F is empty */
static int target(const r6_state* s, uint64_t other, uint64_t f)
{
    int bk = -1, bx = 0, bf = 0;
    for (int k = 0; k < 6; ++k) {
        const int nf = popc(RO_CONTINENT_MASK[k] & f), nx = popc(RO_CONTINENT_MASK[k] & other);
        if (nf == 0) continue;
        if (bk < 0 || nx < bx || (nx == bx && nf > bf)) { bk = k; bx = nx; bf = nf; }
    }
    if (bk < 0) return -1;
    int t = -1, ta = RO_ARMY_MAX + 1;
    uint64_t m = RO_CONTINENT_MASK[bk] & f;
    while (m) { int i = ctz(m); m &= m - 1; if (s->army[i] < ta) { ta = s->army[i]; t = i; } }
    return t;
}

int r6_script_action(const r6_state* s, const ro_rules* r)
{
    const uint64_t valid = r6_valid_moves(s, r), L = valid & ALL_LANDS;
    uint64_t O = 0, gt1 = 0;
    for (int i = 0; i < RO_LANDS; ++i) {
        if (s->owner[i] == s->cur) O |= 1ull << i;
        if (s->army[i] > 1) gt1 |= 1ull << i;
    }
    const uint64_t X = ALL_LANDS & ~O;
    switch (s->phase) {
    case R6_SETUP:
    case R6_REINFORCEMENT: {
        if (!L) return R6_SKIP;
        const int t = target(s, X, nbr_union(O) & X);
        const int f = t >= 0 ? strongest(s, t, L) : -1;
        if (f >= 0) return f;
        int b = -1, bv = -1;
        for (uint64_t m = L; m; m &= m - 1) {
            const int i = ctz(m), v = foreign_armies(s, i, X);
            if (v > bv) { bv = v; b = i; }
        }
        return b;
    }
    case R6_ATTACK: {
        if (!L) return R6_SKIP;
        const int t = target(s, X, L);
        uint64_t cont = 0;
        for (int k = 0; k < 6; ++k) if ((RO_CONTINENT_MASK[k] >> t) & 1) cont = RO_CONTINENT_MASK[k];
        int best = -1, bm = 0, bin = 0, any = -1, am = 0;
        for (uint64_t m = L; m; m &= m - 1) {
            const int i = ctz(m), f = strongest(s, i, O & gt1);
            const int mg = (int)s->army[f] - (int)s->army[i], in = (int)((cont >> i) & 1);
            if (best < 0 || in > bin || (in == bin && mg > bm)) { best = i; bm = mg; bin = in; }
            if (any < 0 || mg > am) { any = i; am = mg; }
        }
        if (bm >= R6S_MARGIN || !(valid & SKIP_MASK)) return best;
        return am >= R6S_MARGIN ? any : R6_SKIP;
    }
    case R6_MOBILIZATION:
        if ((RO_NBR_MASK[s->mob_to] & X) == 0 && (RO_NBR_MASK[s->mob_from] & X) != 0) return s->mob_from;
        return s->mob_to;
    default: {                                                    /* FORTIFY: the source stays r6_make_move's rule */
        int b = -1, bv = 0;
        for (uint64_t m = L & nbr_union(X); m; m &= m - 1) {
            const int i = ctz(m);
            if (s->army[i] >= R6S_FORTIFY_BELOW) continue;
            const int v = foreign_armies(s, i, X) - (int)s->army[i];
            if (b < 0 || v > bv) { bv = v; b = i; }
        }
        return b >= 0 ? b : R6_SKIP;
    }
    }
}

/* the library's constants, for the binding's agreement check */
int r6s_margin(void) { return R6S_MARGIN; }
int r6s_fortify_below(void) { return R6S_FORTIFY_BELOW; }
