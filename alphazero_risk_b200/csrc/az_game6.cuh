// az_game6.cuh — device-side rules of the SIX-PLAYER extension (SIXPLAYER.md; BASELINE.json configs[3]), shared by the environment
// kernels (az_env6.cu, one thread per game) and the search (az_mcts6.cu, lane 0 of a game's warp).  No reference parity exists for
// this game (PLAYER_COUNT = 2 upstream); the checker is oracle/risk6_oracle.c.  Everything with a two-player counterpart follows
// az_game.cuh's arithmetic and reuses its tables, neighbour-union lookup, fortify-source search and Philox contract.
//
// State words (28 per game):
//   words 0..10   army bytes of the 42 lands            words 11..21  owner bytes (seat 0..5)
//   word 22       cards of seats 0..3 (a byte each)     word 23       cards of seats 4, 5 | allow_draw << 16 | attacks << 24
//   word 24       round | cur << 16 | card_sets << 24   word 25       reinf | phase << 8 | mob_from << 16 | mob_to << 24
//   word 26       set-up pools of the six seats (4 bits each)          word 27       ply
#pragma once

#include "az_game.cuh"

#define E6_WORDS 28
#define E6_IMG 108                      // sizeof(r6_state), oracle/risk6_oracle.h: the host image of one game
#define E6_PLAYERS 6

struct AzGame6 {
    uint64_t own[E6_PLAYERS];           // only ever indexed with compile-time constants (see e6_own): stays in registers
    uint64_t gt1, full;
    uint32_t round, cur, card_sets, reinf, phase, mob_from, mob_to, allow_draw, attacks;
    uint32_t cards_lo, cards_hi, pools; // a byte per seat (0..3 | 4, 5), four bits per seat
};

__device__ __forceinline__ uint64_t e6_own(const AzGame6& g, uint32_t p)
{
    uint64_t v = g.own[0];
#pragma unroll
    for (int k = 1; k < E6_PLAYERS; ++k) v = p == (uint32_t)k ? g.own[k] : v;
    return v;
}
__device__ __forceinline__ void e6_move_land(AzGame6& g, uint32_t from_p, uint32_t to_p, uint64_t m)
{
#pragma unroll
    for (int k = 0; k < E6_PLAYERS; ++k) {
        if (from_p == (uint32_t)k) g.own[k] &= ~m;
        if (to_p == (uint32_t)k) g.own[k] |= m;
    }
}
__device__ __forceinline__ uint32_t e6_cards(const AzGame6& g, uint32_t p) { return p < 4 ? (g.cards_lo >> (8 * p)) & 0xffu : (g.cards_hi >> (8 * (p - 4))) & 0xffu; }
__device__ __forceinline__ void e6_set_cards(AzGame6& g, uint32_t p, uint32_t v)
{
    v &= 0xffu;
    if (p < 4) g.cards_lo = (g.cards_lo & ~(0xffu << (8 * p))) | (v << (8 * p));
    else g.cards_hi = (g.cards_hi & ~(0xffu << (8 * (p - 4)))) | (v << (8 * (p - 4)));
}
__device__ __forceinline__ uint32_t e6_pool(const AzGame6& g, uint32_t p) { return (g.pools >> (4 * p)) & 0xfu; }

struct E6Ctx {
    AzGame6 g;
    AzLandColumn army, owner, scratch;
    uint32_t ply;
};

__device__ __forceinline__ void e6_masks(E6Ctx& c)
{
#pragma unroll
    for (int k = 0; k < E6_PLAYERS; ++k) c.g.own[k] = 0;
    c.g.gt1 = c.g.full = 0;
    for (int i = 0; i < AZ_LANDS; ++i) {
        const uint32_t a = c.army.get(i), o = c.owner.get(i);
        const uint64_t m = 1ull << i;
#pragma unroll
        for (int k = 0; k < E6_PLAYERS; ++k) if (o == (uint32_t)k) c.g.own[k] |= m;
        if (a > 1) c.g.gt1 |= m;
        if (a == AZ_ARMY_MAX) c.g.full |= m;
    }
}
__device__ __forceinline__ void e6_unpack(AzGame6& g, uint32_t w22, uint32_t w23, uint32_t w24, uint32_t w25, uint32_t w26)
{
    g.cards_lo = w22; g.cards_hi = w23 & 0xffffu; g.allow_draw = (w23 >> 16) & 0xffu; g.attacks = (w23 >> 24) & 0xffu;
    g.round = w24 & 0xffffu; g.cur = (w24 >> 16) & 0xffu; g.card_sets = (w24 >> 24) & 0xffu;
    g.reinf = w25 & 0xffu; g.phase = (w25 >> 8) & 0xffu; g.mob_from = (w25 >> 16) & 0xffu; g.mob_to = (w25 >> 24) & 0xffu;
    g.pools = w26 & 0xffffffu;
}
// ---------------------------------------------------------------- rules (SIXPLAYER.md; oracle/risk6_oracle.c states the same)
__device__ __forceinline__ void e6_set_army(E6Ctx& c, int i, uint32_t army)
{
    c.army.set(i, army);
    const uint64_t m = 1ull << i;
    c.g.gt1 = army > 1 ? (c.g.gt1 | m) : (c.g.gt1 & ~m);
    c.g.full = army == AZ_ARMY_MAX ? (c.g.full | m) : (c.g.full & ~m);
}

// winner seat 0..5, AZ_STATUS_DRAW, AZ_STATUS_RUNNING (State::gameStatus, state/state.cpp:518-565, for six seats)
__device__ __forceinline__ int e6_status(const AzGame6& g, const AzRulesDev& r)
{
    int alive = 0, last = -1, best = -1, best_n = -1, tie = 0;
#pragma unroll
    for (int p = 0; p < E6_PLAYERS; ++p) {
        const int n = __popcll(g.own[p]);
        if (n > 0) { alive++; last = p; }
        if (n > best_n) { best_n = n; best = p; tie = 0; } else if (n == best_n) tie = 1;
    }
    if (alive == 1) return last;
    if (r.allow_yield && best_n >= 30) return best;
    if ((int)g.round > r.max_game_rounds) return tie ? AZ_STATUS_DRAW : best;
    return AZ_STATUS_RUNNING;
}

__device__ __forceinline__ uint64_t e6_attack_army(const AzGame6& g, const AzTables& T, uint64_t oc) { return az_nbr_union(T, oc & g.gt1) & ~oc; }

// UtilityNN::getValidMoves (alphazero_moves.cpp:3-70): "the enemy" = every other seat
__device__ __forceinline__ uint64_t e6_valid(const AzGame6& g, const AzTables& T, const AzRulesDev& r)
{
    const uint64_t oc = e6_own(g, g.cur);
    if (g.phase == AZ_PH_MOBILIZATION) return (1ull << (g.mob_from & 63u)) | (1ull << (g.mob_to & 63u));
    if (g.phase == AZ_PH_ATTACK) {
        const uint64_t aa = e6_attack_army(g, T, oc);
        return r.limit_attack ? (aa ? aa : AZ_SKIP_MASK) : (aa | AZ_SKIP_MASK);
    }
    const uint64_t border = az_nbr_union(T, AZ_ALL_LANDS & ~oc);
    if (g.phase == AZ_PH_FORTIFY) return (r.limit_reinforcement ? (oc & border) : oc) | AZ_SKIP_MASK;
    const uint64_t o = oc & ~g.full;                              // SETUP / REINFORCEMENT
    if (o == 0) return AZ_SKIP_MASK;
    return (r.limit_reinforcement && (o & border)) ? (o & border) : o;
}

__device__ __forceinline__ void e6_goto_attack(AzGame6& g, const AzTables& T)
{
    g.phase = AZ_PH_ATTACK; g.mob_from = AZ_NONE; g.mob_to = AZ_NONE; g.reinf = 0;
    if (e6_attack_army(g, T, e6_own(g, g.cur)) == 0) g.phase = AZ_PH_FORTIFY;
}

// State::nextPlayerGameTurn (state.cpp:748-766): next seat that still owns a land; the round advances when the order wraps
__device__ __forceinline__ void e6_end_turn(AzGame6& g)
{
    if (g.allow_draw) { e6_set_cards(g, g.cur, e6_cards(g, g.cur) + 1); g.allow_draw = 0; }
    uint32_t next = g.cur;
    for (int k = 0; k < E6_PLAYERS; ++k) {
        next = next + 1 == E6_PLAYERS ? 0u : next + 1;
        if (next == 0) g.round = (g.round + 1) & 0xffffu;
        if (e6_own(g, next)) break;
    }
    g.cur = next; g.attacks = 0; g.phase = AZ_PH_REINFORCEMENT;
    g.reinf = (uint32_t)az_reinforcement_value(e6_own(g, next));
}

// the dice of ONE real move: the base-6 digits of word 0 of the real-move block (at most five dice, include/az_philox.h)
struct E6DiceWord {
    uint32_t w;
    __device__ __forceinline__ int next() { const uint64_t p = (uint64_t)w * 6u; w = (uint32_t)p; return (int)(p >> 32) + 1; }
};

// UtilityNN::makeMove (alphazero_moves.cpp:72-233) for a LEGAL action; DiceT::next() yields the dice in the reference's order
// (attacker dice first): E6DiceWord for a real move, AzDicePhilox for a descent of the search (one running stream per simulation)
template <class DiceT>
__device__ __forceinline__ void e6_move(E6Ctx& c, const AzTables& T, const AzRulesDev& r, int action, DiceT& dice)
{
    AzGame6& g = c.g;
    const uint32_t cur = g.cur;
    if (action == AZ_SKIP) {
        if (g.phase == AZ_PH_REINFORCEMENT) e6_goto_attack(g, T);
        else if (g.phase == AZ_PH_ATTACK) g.phase = AZ_PH_FORTIFY;
        else if (g.phase == AZ_PH_FORTIFY) e6_end_turn(g);
        return;
    }
    const int li = action;
    const int at = (int)c.army.get(li);
    if (g.phase == AZ_PH_SETUP) {
        e6_set_army(c, li, (uint32_t)(at + 1));
        g.pools -= 1u << (4 * cur);
        g.cur = cur + 1 == E6_PLAYERS ? 0u : cur + 1;
        if (g.cur == 0) g.round = (g.round + 1) & 0xffffu;
        if (e6_pool(g, g.cur) == 0) { g.phase = AZ_PH_REINFORCEMENT; g.reinf = (uint32_t)az_reinforcement_value(e6_own(g, g.cur)); }
    } else if (g.phase == AZ_PH_REINFORCEMENT) {
        uint32_t cards = e6_cards(g, cur);
        if (cards >= 3) {
            e6_set_cards(g, cur, cards - 3);
            g.card_sets = (g.card_sets + 1) & 0xffu;
            const int cs = (int)g.card_sets;
            g.reinf = (g.reinf + (uint32_t)(cs <= 5 ? 2 + 2 * cs : 15 + (cs - 6) * 5)) & 0xffu;
        }
        int rf = (int)g.reinf / 2;
        if (rf < r.min_unit_move) rf = r.min_unit_move < (int)g.reinf ? r.min_unit_move : (int)g.reinf;
        const int space = AZ_ARMY_MAX - at;
        if (space < rf) rf = space;
        g.reinf = (g.reinf - (uint32_t)rf) & 0xffu;
        e6_set_army(c, li, (uint32_t)(at + rf));
        if (g.reinf == 0) e6_goto_attack(g, T);
    } else if (g.phase == AZ_PH_ATTACK) {
        const uint64_t oc = e6_own(g, cur), cand = oc & g.gt1;
        int best = 0, from = li;
        uint64_t lst = T.list6[li];
#pragma unroll
        for (int k = 0; k < 6; ++k) {
            const int n = (int)(lst & 63u); lst >>= 6;
            const bool ok = n != 63 && ((cand >> n) & 1ull);
            const int v = ok ? (int)c.army.get(ok ? n : li) - 1 : 0;
            if (v > best) { best = v; from = n; }
        }
        g.attacks = (g.attacks + 1) & 0xffu;
        int a = best + 1, d = at, units;
        const uint32_t defender = c.owner.get(li);
        {
            const int na = a >= 4 ? 3 : (a == 3 ? 2 : 1), nd = d >= 2 ? 2 : 1;
            units = na;
            const int a0 = dice.next();
            int a1 = 0, a2 = 0, d1 = 0;
            if (na > 1) a1 = dice.next();
            if (na > 2) a2 = dice.next();
            const int d0 = dice.next();
            if (nd > 1) d1 = dice.next();
            const int hi = max(a0, max(a1, a2));
            int lo = min(a0, max(a1, a2)); lo = max(lo, min(a1, a2));
            const int dh = max(d0, d1), dl = min(d0, d1);
            if (hi > dh) d--; else { a--; units--; }
            if (na >= 2 && nd == 2) { if (lo > dl) d--; else { a--; units--; } }
        }
        if (d == 0) {
            a -= units;
            if (a > 1) { g.phase = AZ_PH_MOBILIZATION; g.mob_from = (uint32_t)from; g.mob_to = (uint32_t)li; }
            g.allow_draw = 1;
            e6_set_army(c, from, (uint32_t)a); e6_set_army(c, li, (uint32_t)units);
            c.owner.set(li, cur);
            e6_move_land(g, defender, cur, 1ull << li);
            if (e6_own(g, defender) == 0) {                       // elimination: the eliminator takes the cards
                e6_set_cards(g, cur, e6_cards(g, cur) + e6_cards(g, defender));
                e6_set_cards(g, defender, 0);
            }
        } else { e6_set_army(c, from, (uint32_t)a); e6_set_army(c, li, (uint32_t)d); }
        if (g.phase == AZ_PH_ATTACK && e6_attack_army(g, T, e6_own(g, cur)) == 0) g.phase = AZ_PH_FORTIFY;
    } else if (g.phase == AZ_PH_MOBILIZATION) {
        if ((uint32_t)li == g.mob_from) e6_goto_attack(g, T);
        else {
            const int from = (int)g.mob_from;
            const int af = (int)c.army.get(from), v = af - 1;
            int rf = v / 2;
            if (rf < r.min_unit_move) rf = r.min_unit_move < v ? r.min_unit_move : v;
            e6_set_army(c, from, (uint32_t)(af - rf)); e6_set_army(c, li, (uint32_t)(at + rf));
            if (af - rf == 1) e6_goto_attack(g, T);
        }
    } else {                                                      // FORTIFY
        if (at != AZ_ARMY_MAX) {
            AzGame t; t.cur = 0; t.own0 = e6_own(g, cur); t.own1 = 0; t.gt1 = g.gt1; t.full = g.full;   // the two-player search on the mover's lands
            int from, amount;
            az_fortify_source(t, c.army, c.scratch, T, li, from, amount);
            if (from >= 0) {
                const int space = AZ_ARMY_MAX - at, mv = space < amount ? space : amount;
                const int af = (int)c.army.get(from);
                e6_set_army(c, from, (uint32_t)(af - mv)); e6_set_army(c, li, (uint32_t)(at + mv));
            }
        }
        e6_end_turn(g);
    }
}

// State::newGame for six seats: the 42 draws of the deal stream go to seats 0..5 in turn, one army each; 13 armies to place per seat
__device__ __forceinline__ void e6_new_game(E6Ctx& c, uint64_t seed, uint32_t game, uint32_t ply)
{
    AzGame6& g = c.g;
#pragma unroll
    for (int k = 0; k < E6_PLAYERS; ++k) g.own[k] = 0;
    g.gt1 = g.full = 0;
    g.round = 1; g.cur = 0; g.card_sets = 0; g.reinf = 0; g.phase = AZ_PH_SETUP; g.mob_from = AZ_NONE; g.mob_to = AZ_NONE;
    g.allow_draw = 0; g.attacks = 0; g.cards_lo = g.cards_hi = 0; g.pools = 0xDDDDDDu;                 // 13 per seat
    uint64_t avail = AZ_ALL_LANDS;
    az_u32x4 blk;
    for (uint32_t i = 0; i < 42; ++i) {
        if ((i & 3u) == 0) blk = az_rng_block(seed, game, ply, AZ_STREAM_DEAL, i >> 2);
        const uint32_t k = az_mulhi32(az_u32x4_word(blk, (int)(i & 3u)), 42u - i);
        const int l = az_nth_set_bit(avail, k);
        avail &= ~(1ull << l);
        const uint32_t seat = i % E6_PLAYERS;
        c.army.set(l, 1u); c.owner.set(l, seat);
#pragma unroll
        for (int s = 0; s < E6_PLAYERS; ++s) if (seat == (uint32_t)s) g.own[s] |= 1ull << l;
    }
}

// the six-seat network input of one position (SIXPLAYER.md; r6_encode of the oracle, same expressions): the reference's [7][6][13]
// planes with "enemy" = the seat that moves next and "neutral" = every other seat.  One thread writes the position's
// AZ_INPUT_FLOATS floats; shared by the search's leaf batches (k_env6_encode) and the training unpack of six-player records.
// P = 16: the seat planes (SIXPLAYER.md §2; r6_encode16 of the oracle), AZ_INPUT6_FLOATS floats — plane k (k = 0..5) holds the armies
// of seat (cur + k) % 6, planes 6..15 are planes 3..12 of the 13-plane form.
template <int P = 13>
__device__ __forceinline__ void e6_encode_position(const uint8_t* army, const uint8_t* owner, uint32_t cur, uint32_t phase, uint32_t attacks,
                                                   uint32_t allow_draw, float* __restrict__ out)
{
    static_assert(P == 13 || P == 16, "13 or 16 input planes");
    uint64_t own[E6_PLAYERS] = { 0, 0, 0, 0, 0, 0 };
    int own_total = 0, other_total = 0;
    for (int i = 0; i < AZ_LANDS; ++i) {
        own[owner[i]] |= 1ull << i;
        if (owner[i] == cur) own_total += army[i]; else other_total += army[i];
    }
    uint32_t nx = cur;
    for (int k = 0; k < E6_PLAYERS; ++k) { nx = nx + 1 == E6_PLAYERS ? 0u : nx + 1; if (own[nx]) break; }
    const float ref = (float)az_reinforcement_value(own[cur]);
    float oref = 0.0f;
    for (uint32_t p = 0; p < E6_PLAYERS; ++p) if (p != cur && own[p]) oref = __fadd_rn(oref, (float)az_reinforcement_value(own[p]));
    const float army_share = __fdiv_rn((float)own_total, __fadd_rn((float)own_total, (float)other_total));
    const float reinf_share = __fdiv_rn(ref, __fadd_rn(ref, oref));
    float att = __fdiv_rn((float)attacks, 8.0f); att = att > 1.0f ? 1.0f : att;
    for (int i = 0; i < AZ_LANDS; ++i) {
        float* f = out + i * P;
        const float a = __fdiv_rn((float)army[i], 32.0f);
        if constexpr (P == 13) {
            f[0] = owner[i] == cur ? a : 0.0f;
            f[1] = (owner[i] == nx && nx != cur) ? a : 0.0f;
            f[2] = (owner[i] != cur && owner[i] != nx) ? a : 0.0f;
            f[3] = army_share; f[4] = reinf_share; f[5] = att; f[6] = allow_draw ? 1.0f : 0.0f;
            for (uint32_t k = 0; k < 6; ++k) f[7 + k] = phase == k ? 1.0f : 0.0f;
        } else {
            for (uint32_t k = 0; k < E6_PLAYERS; ++k) f[k] = owner[i] == (cur + k) % E6_PLAYERS ? a : 0.0f;
            f[6] = army_share; f[7] = reinf_share; f[8] = att; f[9] = allow_draw ? 1.0f : 0.0f;
            for (uint32_t k = 0; k < 6; ++k) f[10 + k] = phase == k ? 1.0f : 0.0f;
        }
    }
}
