// az_env6.cu — the SIX-PLAYER extension of the lockstep Risk environment (BASELINE.json configs[3]) and its az_env6_* C ABI.
//
// The reference has no six-player game (PLAYER_COUNT = 2, /root/reference/src/risk_game/state/state.h:13), so this is a
// throughput-only extension with NO reference parity: its rules are SIXPLAYER.md, its only checker is oracle/risk6_oracle.c
// (tests/test_env6_gpu.py compares bit for bit).  Everything that has a two-player counterpart follows that counterpart's
// arithmetic (az_game.cuh) and shares its map tables, neighbour-union lookup, fortify-source search and Philox contract.  The
// two-player path (az_env_*) is untouched.
//
// Layout: one thread per game; 28 words per game in HBM as a structure of arrays (word w of game g at state[w * n + g]):
//   words 0..10   army bytes of the 42 lands            words 11..21  owner bytes (seat 0..5)
//   word 22       cards of seats 0..3 (a byte each)     word 23       cards of seats 4, 5 | allow_draw << 16 | attacks << 24
//   word 24       round | cur << 16 | card_sets << 24   word 25       reinf | phase << 8 | mob_from << 16 | mob_to << 24
//   word 26       set-up pools of the six seats (4 bits each)          word 27       ply
// Inside a kernel the land bytes sit in shared-memory columns (bank = lane), six ownership masks + army > 1 + army == 32 in registers.
#include <cstring>
#include <new>

#include "az_common.cuh"
#include "az_arena.cuh"

#define E6_BLOCK 128                    // configs[3] has 16384 games per GPU: 128 blocks = four warps on 128 of the 148 SMs (256: 64 SMs)
#include "az_game6.cuh"
#include "az_script6.cuh"
#include "az_samples6.cuh"

struct E6Smem {
    uint64_t tab[AZ_TABLE_U64];
    uint32_t col[33 * E6_BLOCK];        // 11 army words + 11 owner words + 11 fortify-DFS parent words per thread
};
__device__ __forceinline__ void e6_bind(E6Ctx& c, E6Smem& sm)
{
    c.army.base = (uint8_t*)(sm.col) + 4 * threadIdx.x; c.army.stride_bytes = 4 * E6_BLOCK;
    c.owner.base = (uint8_t*)(sm.col + 11 * E6_BLOCK) + 4 * threadIdx.x; c.owner.stride_bytes = 4 * E6_BLOCK;
    c.scratch.base = (uint8_t*)(sm.col + 22 * E6_BLOCK) + 4 * threadIdx.x; c.scratch.stride_bytes = 4 * E6_BLOCK;
}
__device__ __forceinline__ void e6_load(E6Ctx& c, E6Smem& sm, const uint32_t* __restrict__ st, int n, int gi)
{
    e6_bind(c, sm);
    for (int w = 0; w < 22; ++w) sm.col[w * E6_BLOCK + threadIdx.x] = st[(size_t)w * n + gi];
    e6_masks(c);
    e6_unpack(c.g, st[(size_t)22 * n + gi], st[(size_t)23 * n + gi], st[(size_t)24 * n + gi], st[(size_t)25 * n + gi], st[(size_t)26 * n + gi]);
    c.ply = st[(size_t)27 * n + gi];
}
__device__ __forceinline__ void e6_store(const E6Ctx& c, E6Smem& sm, uint32_t* __restrict__ st, int n, int gi)
{
    for (int w = 0; w < 22; ++w) st[(size_t)w * n + gi] = sm.col[w * E6_BLOCK + threadIdx.x];
    const AzGame6& g = c.g;
    st[(size_t)22 * n + gi] = g.cards_lo;
    st[(size_t)23 * n + gi] = (g.cards_hi & 0xffffu) | ((g.allow_draw & 0xffu) << 16) | ((g.attacks & 0xffu) << 24);
    st[(size_t)24 * n + gi] = (g.round & 0xffffu) | (g.cur << 16) | (g.card_sets << 24);
    st[(size_t)25 * n + gi] = (g.reinf & 0xffu) | (g.phase << 8) | (g.mob_from << 16) | (g.mob_to << 24);
    st[(size_t)26 * n + gi] = g.pools & 0xffffffu;
    st[(size_t)27 * n + gi] = c.ply;
}

// ---------------------------------------------------------------- kernels
__device__ __forceinline__ AzTables e6_stage(E6Smem& sm, const uint64_t* __restrict__ g_tab)
{
    for (int i = threadIdx.x; i < AZ_TABLE_U64; i += blockDim.x) sm.tab[i] = g_tab[i];
    __syncthreads();
    return az_tables_from_smem(sm.tab);
}

__global__ void __launch_bounds__(E6_BLOCK) k_env6_reset(uint32_t* __restrict__ st, int n, uint64_t seed, uint32_t first_game)
{
    __shared__ E6Smem sm;
    const int gi = blockIdx.x * E6_BLOCK + threadIdx.x;
    if (gi >= n) return;
    E6Ctx c; e6_bind(c, sm);
    for (int w = 0; w < 22; ++w) sm.col[w * E6_BLOCK + threadIdx.x] = 0;
    e6_new_game(c, seed, first_game + (uint32_t)gi, 0);
    c.ply = 0;
    e6_store(c, sm, st, n, gi);
}

// n_steps uniform-random legal moves per game (action = k-th set bit of the mask, k = mulhi(word 1 of the real-move block,
// popcount); dice = word 0), finished games re-dealt in place: the six-player form of az_env_rollout.  counters: steps, games,
// draws, wins of seats 0..5
__global__ void __launch_bounds__(E6_BLOCK) k_env6_rollout(uint32_t* __restrict__ st, int n, const uint64_t* __restrict__ g_tab, int n_steps,
                                                          uint64_t seed, uint32_t first_game, AzRulesDev rules,
                                                          unsigned long long* __restrict__ counters)
{
    __shared__ E6Smem sm;
    const AzTables T = e6_stage(sm, g_tab);
    const int gi = blockIdx.x * E6_BLOCK + threadIdx.x;
    if (gi >= n) return;
    E6Ctx c; e6_load(c, sm, st, n, gi);
    const uint32_t game = first_game + (uint32_t)gi;
    unsigned games = 0, draws = 0;
    for (int s = 0; s < n_steps; ++s) {
        const int stt = e6_status(c.g, rules);
        if (stt != AZ_STATUS_RUNNING) {
            games++;
            if (stt == AZ_STATUS_DRAW) draws++; else atomicAdd(&counters[3 + stt], 1ull);
            e6_new_game(c, seed, game, c.ply);
        }
        const uint64_t valid = e6_valid(c.g, T, rules);
        const az_u32x4 blk = az_rng_block(seed, game, c.ply, AZ_STREAM_REAL, 0);
        const int action = az_nth_set_bit(valid, az_mulhi32(blk.y, (uint32_t)__popcll(valid)));
        { E6DiceWord dice; dice.w = blk.x; e6_move(c, T, rules, action, dice); }
        c.ply++;
    }
    e6_store(c, sm, st, n, gi);
    atomicAdd(&counters[0], (unsigned long long)n_steps);
    if (games) atomicAdd(&counters[1], (unsigned long long)games);
    if (draws) atomicAdd(&counters[2], (unsigned long long)draws);
}

// one host-chosen action per game (the lockstep tests): status byte = AZ_STATUS_ILLEGAL / AZ_STATUS_OVER (state untouched) or the
// game status after the move
__global__ void __launch_bounds__(E6_BLOCK) k_env6_step(uint32_t* __restrict__ st, int n, const uint64_t* __restrict__ g_tab,
                                                       const uint8_t* __restrict__ action, uint64_t seed, uint32_t first_game,
                                                       AzRulesDev rules, int8_t* __restrict__ status)
{
    __shared__ E6Smem sm;
    const AzTables T = e6_stage(sm, g_tab);
    const int gi = blockIdx.x * E6_BLOCK + threadIdx.x;
    if (gi >= n) return;
    E6Ctx c; e6_load(c, sm, st, n, gi);
    if (e6_status(c.g, rules) != AZ_STATUS_RUNNING) { status[gi] = AZ_STATUS_OVER; return; }
    const int a = action[gi];
    const uint64_t valid = e6_valid(c.g, T, rules);
    if (a > AZ_SKIP || !((valid >> a) & 1ull)) { status[gi] = AZ_STATUS_ILLEGAL; return; }
    const az_u32x4 blk = az_rng_block(seed, first_game + (uint32_t)gi, c.ply, AZ_STREAM_REAL, 0);
    { E6DiceWord dice; dice.w = blk.x; e6_move(c, T, rules, a, dice); }
    c.ply++;
    e6_store(c, sm, st, n, gi);
    status[gi] = (int8_t)e6_status(c.g, rules);
}

__global__ void __launch_bounds__(E6_BLOCK) k_env6_query(const uint32_t* __restrict__ st, int n, const uint64_t* __restrict__ g_tab,
                                                        AzRulesDev rules, uint64_t* __restrict__ valid, int8_t* __restrict__ status)
{
    __shared__ E6Smem sm;
    const AzTables T = e6_stage(sm, g_tab);
    const int gi = blockIdx.x * E6_BLOCK + threadIdx.x;
    if (gi >= n) return;
    E6Ctx c; e6_load(c, sm, st, n, gi);
    if (valid) valid[gi] = e6_valid(c.g, T, rules);
    if (status) status[gi] = (int8_t)e6_status(c.g, rules);
}

// the scripted action of every game (SIXPLAYER.md §5), 0xff for a finished game
__global__ void __launch_bounds__(E6_BLOCK) k_env6_script(const uint32_t* __restrict__ st, int n, const uint64_t* __restrict__ g_tab,
                                                         AzRulesDev rules, uint8_t* __restrict__ action)
{
    __shared__ E6Smem sm;
    const AzTables T = e6_stage(sm, g_tab);
    const int gi = blockIdx.x * E6_BLOCK + threadIdx.x;
    if (gi >= n) return;
    E6Ctx c; e6_load(c, sm, st, n, gi);
    action[gi] = e6_status(c.g, rules) != AZ_STATUS_RUNNING ? (uint8_t)0xff : (uint8_t)e6_script_action(c, T, rules);
}

// ---------------------------------------------------------------- generated games (SIXPLAYER.md §6)
// state words 22..26 of the game's scalars, packed as e6_store packs them (e6_store keeps its own copy: the SASS of the kernels that
// existed before generated games stays as it was)
__device__ __forceinline__ void e6_pack_scalars(const AzGame6& g, uint32_t w[5])
{
    w[0] = g.cards_lo;
    w[1] = (g.cards_hi & 0xffffu) | ((g.allow_draw & 0xffu) << 16) | ((g.attacks & 0xffu) << 24);
    w[2] = (g.round & 0xffffu) | (g.cur << 16) | (g.card_sets << 24);
    w[3] = (g.reinf & 0xffu) | (g.phase << 8) | (g.mob_from << 16) | (g.mob_to << 24);
    w[4] = g.pools & 0xffffffu;
}
// recording of az_env6_play (az_env6_record): the samples of each slot's running game are staged until the game ends
struct E6RecDev {
    uint32_t* stage = nullptr;                  // [n][max][28]  state words 0..26 before the ply, then the played action
    uint32_t* len = nullptr;                    // [n]           staged samples of the running game (> max = overflowed)
    uint8_t* out = nullptr;                     // [cap][288]    records of finished games
    unsigned long long* count = nullptr;        // [2]           records in out, samples dropped (staging or queue full)
    int max = 0;
    unsigned long long cap = 0;
};
#define E6_STAGE_WORDS 28

// the `len` staged samples of slot gi's game, which ended with `status` -> one contiguous block of records (az_rec_reserve: a game
// that overflowed its staging or does not fit is dropped whole and counted).  The game's own thread writes its block, 16 bytes a store.
__device__ __noinline__ void e6_rec_flush(E6RecDev r, int gi, uint32_t len, int status)
{
    unsigned long long base = 0;
    if (!az_rec_reserve(r.count, r.cap, len, len <= (uint32_t)r.max, &base)) return;
    const uint4* src = (const uint4*)(r.stage + (size_t)gi * r.max * E6_STAGE_WORDS);
    uint4* dst = (uint4*)(r.out + base * S6_BYTES);
    for (uint32_t i = 0; i < len; ++i, src += E6_STAGE_WORDS / 4, dst += S6_BYTES / 16) {
        uint32_t w[E6_STAGE_WORDS];
#pragma unroll
        for (int q = 0; q < E6_STAGE_WORDS / 4; ++q) { const uint4 v = src[q]; w[4 * q] = v.x; w[4 * q + 1] = v.y; w[4 * q + 2] = v.z; w[4 * q + 3] = v.w; }
        const int action = (int)w[E6_STAGE_WORDS - 1];
#pragma unroll
        for (int q = 0; q < S6_BYTES / 16; ++q)
            dst[q] = make_uint4(s6_onehot_record_word(w, action, status, 4 * q), s6_onehot_record_word(w, action, status, 4 * q + 1),
                                s6_onehot_record_word(w, action, status, 4 * q + 2), s6_onehot_record_word(w, action, status, 4 * q + 3));
    }
}

// n_plies plies of every game, the seat to move playing by `script` (bit s set: seat s is the scripted agent, e6_script_action; clear:
// the uniform-random player, k_env6_rollout's rule), both with the real-move dice of (seed, game, ply); finished games are counted
// and re-dealt in place on k_env6_rollout's schedule, so six random seats are k_env6_rollout bit for bit.  REC: every ply of a seat
// in `record_seats` stages (state before the ply, action); a game's samples become records by the end of the call in which it ends.
template <bool REC>
__global__ void __launch_bounds__(E6_BLOCK) k_env6_play(uint32_t* __restrict__ st, int n, const uint64_t* __restrict__ g_tab, int n_plies,
                                                       uint64_t seed, uint32_t first_game, AzRulesDev rules, uint32_t script,
                                                       uint32_t record_seats, E6RecDev rec, unsigned long long* __restrict__ counters)
{
    __shared__ E6Smem sm;
    const AzTables T = e6_stage(sm, g_tab);
    const int gi = blockIdx.x * E6_BLOCK + threadIdx.x;
    if (gi >= n) return;
    E6Ctx c; e6_load(c, sm, st, n, gi);
    const uint32_t game = first_game + (uint32_t)gi;
    unsigned games = 0, draws = 0;
    uint32_t len = REC ? rec.len[gi] : 0u;
    for (int s = 0; s < n_plies; ++s) {
        const int stt = e6_status(c.g, rules);
        if (stt != AZ_STATUS_RUNNING) {
            games++;
            if (stt == AZ_STATUS_DRAW) draws++; else atomicAdd(&counters[3 + stt], 1ull);
            if (REC && len) { e6_rec_flush(rec, gi, len, stt); len = 0; }
            e6_new_game(c, seed, game, c.ply);
        }
        const az_u32x4 blk = az_rng_block(seed, game, c.ply, AZ_STREAM_REAL, 0);
        int action;
        if ((script >> c.g.cur) & 1u) action = e6_script_action(c, T, rules);
        else {
            const uint64_t valid = e6_valid(c.g, T, rules);
            action = az_nth_set_bit(valid, az_mulhi32(blk.y, (uint32_t)__popcll(valid)));
        }
        if (REC && ((record_seats >> c.g.cur) & 1u)) {
            if (len < (uint32_t)rec.max) {
                uint32_t w[E6_STAGE_WORDS];
#pragma unroll
                for (int k = 0; k < 22; ++k) w[k] = sm.col[k * E6_BLOCK + threadIdx.x];
                e6_pack_scalars(c.g, w + 22);
                w[E6_STAGE_WORDS - 1] = (uint32_t)action;
                uint4* d = (uint4*)(rec.stage + ((size_t)gi * rec.max + len) * E6_STAGE_WORDS);
#pragma unroll
                for (int q = 0; q < E6_STAGE_WORDS / 4; ++q) d[q] = make_uint4(w[4 * q], w[4 * q + 1], w[4 * q + 2], w[4 * q + 3]);
            }
            len++;
        }
        { E6DiceWord dice; dice.w = blk.x; e6_move(c, T, rules, action, dice); }
        c.ply++;
    }
    if (REC) {
        if (len && e6_status(c.g, rules) != AZ_STATUS_RUNNING) { e6_rec_flush(rec, gi, len, e6_status(c.g, rules)); len = 0; }
        rec.len[gi] = len;
    }
    e6_store(c, sm, st, n, gi);
    atomicAdd(&counters[0], (unsigned long long)n_plies);
    if (games) atomicAdd(&counters[1], (unsigned long long)games);
    if (draws) atomicAdd(&counters[2], (unsigned long long)draws);
}

// 108-byte host image (== r6_state of the oracle): army[42], owner[42], cards[6], pool[6], round u16, cur, card_sets, reinf,
// phase, mob_from, mob_to, allow_draw, attacks, 2 pad bytes
__global__ void __launch_bounds__(E6_BLOCK) k_env6_export(const uint32_t* __restrict__ st, int n, uint8_t* __restrict__ img)
{
    __shared__ E6Smem sm;
    const int gi = blockIdx.x * E6_BLOCK + threadIdx.x;
    if (gi >= n) return;
    E6Ctx c; e6_load(c, sm, st, n, gi);
    uint8_t* d = img + (size_t)gi * E6_IMG;
    for (int i = 0; i < AZ_LANDS; ++i) { d[i] = (uint8_t)c.army.get(i); d[42 + i] = (uint8_t)c.owner.get(i); }
    for (uint32_t p = 0; p < E6_PLAYERS; ++p) { d[84 + p] = (uint8_t)e6_cards(c.g, p); d[90 + p] = (uint8_t)e6_pool(c.g, p); }
    d[96] = (uint8_t)(c.g.round & 0xffu); d[97] = (uint8_t)(c.g.round >> 8);
    d[98] = (uint8_t)c.g.cur; d[99] = (uint8_t)c.g.card_sets; d[100] = (uint8_t)c.g.reinf; d[101] = (uint8_t)c.g.phase;
    d[102] = (uint8_t)c.g.mob_from; d[103] = (uint8_t)c.g.mob_to; d[104] = (uint8_t)c.g.allow_draw; d[105] = (uint8_t)c.g.attacks;
    d[106] = 0; d[107] = 0;
}
__global__ void __launch_bounds__(E6_BLOCK) k_env6_import(uint32_t* __restrict__ st, int n, const uint8_t* __restrict__ img, int* __restrict__ bad)
{
    __shared__ E6Smem sm;
    const int gi = blockIdx.x * E6_BLOCK + threadIdx.x;
    if (gi >= n) return;
    const uint8_t* d = img + (size_t)gi * E6_IMG;
    E6Ctx c; e6_bind(c, sm);
    for (int w = 0; w < 22; ++w) sm.col[w * E6_BLOCK + threadIdx.x] = 0;
    bool ok = true;
    for (int i = 0; i < AZ_LANDS; ++i) {
        ok = ok && d[i] >= 1 && d[i] <= AZ_ARMY_MAX && d[42 + i] < E6_PLAYERS;
        c.army.set(i, d[i]); c.owner.set(i, d[42 + i]);
    }
    e6_masks(c);
    AzGame6& g = c.g;
    g.cards_lo = g.cards_hi = 0; g.pools = 0;
    for (uint32_t p = 0; p < E6_PLAYERS; ++p) { e6_set_cards(g, p, d[84 + p]); g.pools |= (uint32_t)(d[90 + p] & 0xfu) << (4 * p); ok = ok && d[90 + p] <= 13; }
    g.round = (uint32_t)d[96] | ((uint32_t)d[97] << 8); g.cur = d[98]; g.card_sets = d[99]; g.reinf = d[100]; g.phase = d[101];
    g.mob_from = d[102]; g.mob_to = d[103]; g.allow_draw = d[104]; g.attacks = d[105];
    ok = ok && g.cur < E6_PLAYERS && g.phase <= AZ_PH_FORTIFY && g.phase != AZ_PH_SETUP_NEUTRAL;
    if (!ok) { atomicAdd(bad, 1); return; }
    c.ply = st[(size_t)27 * n + gi];                              // the slot's move counter is not part of the image
    e6_store(c, sm, st, n, gi);
}

// ---------------------------------------------------------------- six-player arena (SIXPLAYER.md §4): everything between two searches
// One thread per slot: tally the slot's finished game (per-game status and plies on the device), claim the next match game from
// the shared counter and deal it (deal of game id g - g % 6 with rotation, else g; ply 0), play the plies of the uniform-random player
// (az_env6_rollout's rule keyed by the match game id) and of the scripted agent (e6_script_action, SIXPLAYER.md §5; the same dice),
// and stop when a searcher's seat is to move: to_move = that agent.  At most 64 iterations per launch, like k_arena_advance.
// res[A6_ACTIVE] counts the slots that hold a game afterwards, res[A6_WAIT0 + a] those waiting for agent a's search.
__global__ void __launch_bounds__(E6_BLOCK) k_arena6_advance(Arena6Dev a, const uint64_t* __restrict__ g_tab, AzRulesDev rules)
{
    __shared__ E6Smem sm;
    __shared__ unsigned s_cnt[1 + 2 * E6_PLAYERS];    // active slots, waiting slots per agent, random / scripted plies per agent
    if (threadIdx.x < 1 + 2 * E6_PLAYERS) s_cnt[threadIdx.x] = 0;
    const AzTables T = e6_stage(sm, g_tab);           // (its barrier also orders the zeroing above)
    const int gi = blockIdx.x * E6_BLOCK + threadIdx.x;
    int slot = gi < a.n ? a.slot[gi] : A6_DONE;
    if (slot != A6_DONE) {
        E6Ctx c;
        uint32_t game = 0, r = 0;
        int wait = 0xff;
        if (slot == A6_PLAYING) { e6_load(c, sm, a.state, a.n, gi); game = a.slot_game[gi]; r = a.rotate ? game % E6_PLAYERS : 0u; }
        else e6_bind(c, sm);
        for (int it = 0; it < 64; ++it) {
            if (slot == A6_PLAYING) {
                const int st = e6_status(c.g, rules);
                if (st != AZ_STATUS_RUNNING) {
                    const uint32_t k = game - a.first_game;
                    atomicAdd(&a.res[A6_COUNT], 1ull);
                    if (st == AZ_STATUS_DRAW) atomicAdd(&a.res[A6_DRAW], 1ull);
                    else {
                        atomicAdd(&a.res[A6_WIN0 + ((a.seat_agent >> (4 * (((uint32_t)st + r) % E6_PLAYERS))) & 0xfu)], 1ull);
                        atomicAdd(&a.res[A6_WIN_SEAT0 + st], 1ull);
                    }
                    a.out_status[k] = (int8_t)st; a.out_plies[k] = c.ply;
                    slot = A6_FREE;
                }
            }
            if (slot == A6_FREE) {
                const unsigned long long k = atomicAdd(&a.res[A6_CLAIMED], 1ull);
                if (k >= a.n_games) { slot = A6_DONE; break; }
                game = a.first_game + (uint32_t)k;
                r = a.rotate ? game % E6_PLAYERS : 0u;
                for (int w = 0; w < 22; ++w) sm.col[w * E6_BLOCK + threadIdx.x] = 0;
                e6_new_game(c, a.seed, game - r, 0);
                c.ply = 0;
                slot = A6_PLAYING;
                continue;
            }
            const uint32_t agent = (a.seat_agent >> (4 * ((c.g.cur + r) % E6_PLAYERS))) & 0xfu;
            if ((a.searcher >> agent) & 1u) { wait = (int)agent; break; }
            const az_u32x4 blk = az_rng_block(a.seed, game, c.ply, AZ_STREAM_REAL, 0);
            int action;
            if ((a.script >> agent) & 1u) action = e6_script_action(c, T, rules);
            else {
                const uint64_t valid = e6_valid(c.g, T, rules);
                action = az_nth_set_bit(valid, az_mulhi32(blk.y, (uint32_t)__popcll(valid)));
            }
            { E6DiceWord dice; dice.w = blk.x; e6_move(c, T, rules, action, dice); }
            c.ply++;
            atomicAdd(&s_cnt[1 + E6_PLAYERS + agent], 1u);
        }
        if (slot == A6_PLAYING) {
            e6_store(c, sm, a.state, a.n, gi);
            a.slot_game[gi] = game;
            atomicAdd(&s_cnt[0], 1u);
            if (wait != 0xff) atomicAdd(&s_cnt[1 + wait], 1u);
        }
        a.slot[gi] = (uint8_t)slot;
        a.to_move[gi] = (uint8_t)wait;
    }
    __syncthreads();
    if (threadIdx.x < 1 + 2 * E6_PLAYERS && s_cnt[threadIdx.x]) {
        const int i = threadIdx.x;
        const int dst = i == 0 ? A6_ACTIVE : i <= E6_PLAYERS ? A6_WAIT0 + i - 1 : A6_MOVES0 + i - 1 - E6_PLAYERS;
        atomicAdd(&a.res[dst], (unsigned long long)s_cnt[i]);
    }
}

// ---------------------------------------------------------------- C ABI
struct az_env6 {
    int n = 0, device = 0;
    uint32_t first_game = 0;
    uint64_t seed = 0;
    az_rules rules;
    uint32_t* d_state = nullptr;
    unsigned long long* d_counters = nullptr;   // steps, games, draws, wins[6]
    uint8_t* d_img = nullptr; uint8_t* d_action = nullptr; int8_t* d_status = nullptr; uint64_t* d_valid = nullptr; int* d_bad = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    bool timed = false;
    uint64_t generation = 0;    // bumped by reset / import: a search's staged samples of the games before it are abandoned
    E6RecDev rec;               // recording of az_env6_play (az_env6_record); enabled iff rec.out != NULL
};

// accessors for az_mcts6.cu
uint32_t* az_env6_state_ptr(az_env6* e) { return e->d_state; }
int az_env6_n(const az_env6* e) { return e->n; }
int az_env6_device(const az_env6* e) { return e->device; }
uint64_t az_env6_seed(const az_env6* e) { return e->seed; }
uint32_t az_env6_first_game(const az_env6* e) { return e->first_game; }
const az_rules* az_env6_rules(const az_env6* e) { return &e->rules; }
uint64_t az_env6_generation(const az_env6* e) { return e->generation; }

static AzRulesDev e6_rules(const az_rules& r)
{
    AzRulesDev d; d.allow_yield = r.allow_yield; d.limit_reinforcement = r.limit_reinforcement; d.limit_attack = r.limit_attack;
    d.max_game_rounds = r.max_game_rounds; d.min_unit_move = r.min_unit_move; return d;
}
static inline int e6_grid(int n) { return (n + E6_BLOCK - 1) / E6_BLOCK; }

int az_launch_arena6_advance(const Arena6Dev& a, const az_rules* rules, cudaStream_t s)
{
    k_arena6_advance<<<e6_grid(a.n), E6_BLOCK, 0, s>>>(a, az_device_tables(), e6_rules(*rules));
    AZ_CUDA(cudaGetLastError());
    return AZ_OK;
}

extern "C" int az_env6_create(int n_games, const az_rules* rules, int device, uint32_t first_game_id, az_env6** out)
{
    AZ_REQUIRE(out != nullptr, "out is NULL");
    AZ_REQUIRE(n_games > 0, "n_games must be positive");
    int have = 0;
    if (cudaGetDeviceCount(&have) != cudaSuccess || have == 0) { az_set_error("no CUDA device: libaz_b200 has no CPU fallback"); return AZ_ERR_NO_DEVICE; }
    AZ_REQUIRE(device >= 0 && device < have, "device index out of range");
    AzDeviceGuard guard(device);
    int rc = az_upload_tables(); if (rc) return rc;
    az_env6* e = new (std::nothrow) az_env6();
    AZ_REQUIRE(e != nullptr, "out of host memory");
    e->n = n_games; e->device = device; e->first_game = first_game_id;
    if (rules) e->rules = *rules; else az_default_rules(&e->rules);
    const size_t n = (size_t)n_games;
    cudaError_t ce = cudaMalloc(&e->d_state, sizeof(uint32_t) * E6_WORDS * n);
    if (ce == cudaSuccess) ce = cudaMemset(e->d_state, 0, sizeof(uint32_t) * E6_WORDS * n);
    if (ce == cudaSuccess) ce = cudaMalloc(&e->d_counters, sizeof(unsigned long long) * 16);
    if (ce == cudaSuccess) ce = cudaMemset(e->d_counters, 0, sizeof(unsigned long long) * 16);
    if (ce == cudaSuccess) ce = cudaMalloc(&e->d_img, n * E6_IMG);
    if (ce == cudaSuccess) ce = cudaMalloc(&e->d_action, n);
    if (ce == cudaSuccess) ce = cudaMalloc(&e->d_status, n);
    if (ce == cudaSuccess) ce = cudaMalloc(&e->d_valid, sizeof(uint64_t) * n);
    if (ce == cudaSuccess) ce = cudaMalloc(&e->d_bad, sizeof(int));
    if (ce == cudaSuccess) ce = cudaEventCreate(&e->ev0);
    if (ce == cudaSuccess) ce = cudaEventCreate(&e->ev1);
    if (ce != cudaSuccess) { az_set_error("az_env6_create: %s", cudaGetErrorString(ce)); az_env6_destroy(e); return AZ_ERR_CUDA; }
    *out = e;
    return AZ_OK;
}

extern "C" int az_env6_destroy(az_env6* e)
{
    if (!e) return AZ_OK;
    AzDeviceGuard guard(e->device);
    cudaFree(e->d_state); cudaFree(e->d_counters); cudaFree(e->d_img); cudaFree(e->d_action); cudaFree(e->d_status); cudaFree(e->d_valid); cudaFree(e->d_bad);
    cudaFree(e->rec.stage); cudaFree(e->rec.len); cudaFree(e->rec.out); cudaFree(e->rec.count);
    if (e->ev0) cudaEventDestroy(e->ev0);
    if (e->ev1) cudaEventDestroy(e->ev1);
    delete e;
    return AZ_OK;
}

extern "C" int az_env6_reset(az_env6* e, uint64_t seed, void* stream)
{
    AZ_REQUIRE(e != nullptr, "env is NULL");
    AzDeviceGuard guard(e->device);
    e->seed = seed;
    e->generation++;
    if (e->rec.out) AZ_CUDA(cudaMemsetAsync(e->rec.len, 0, sizeof(uint32_t) * (size_t)e->n, (cudaStream_t)stream));   // staged samples go
    k_env6_reset<<<e6_grid(e->n), E6_BLOCK, 0, (cudaStream_t)stream>>>(e->d_state, e->n, seed, e->first_game);
    AZ_CUDA(cudaGetLastError());
    return AZ_OK;
}

extern "C" int az_env6_rollout(az_env6* e, int n_steps, void* stream)
{
    AZ_REQUIRE(e != nullptr, "env is NULL");
    AZ_REQUIRE(n_steps >= 0, "n_steps must be >= 0");
    AzDeviceGuard guard(e->device);
    cudaStream_t s = (cudaStream_t)stream;
    AZ_CUDA(cudaEventRecord(e->ev0, s));
    k_env6_rollout<<<e6_grid(e->n), E6_BLOCK, 0, s>>>(e->d_state, e->n, az_device_tables(), n_steps, e->seed, e->first_game, e6_rules(e->rules),
                                                     e->d_counters);
    AZ_CUDA(cudaGetLastError());
    AZ_CUDA(cudaEventRecord(e->ev1, s));
    e->timed = true;
    return AZ_OK;
}

extern "C" int az_env6_last_kernel_ms(az_env6* e, float* ms)
{
    AZ_REQUIRE(e && ms, "NULL argument");
    AZ_REQUIRE(e->timed, "no timed launch yet");
    AzDeviceGuard guard(e->device);
    AZ_CUDA(cudaEventSynchronize(e->ev1));
    AZ_CUDA(cudaEventElapsedTime(ms, e->ev0, e->ev1));
    return AZ_OK;
}

extern "C" int az_env6_step(az_env6* e, const uint8_t* h_action, int8_t* h_status, void* stream)
{
    AZ_REQUIRE(e && h_action && h_status, "NULL argument");
    AzDeviceGuard guard(e->device);
    cudaStream_t s = (cudaStream_t)stream;
    AZ_CUDA(cudaMemcpyAsync(e->d_action, h_action, (size_t)e->n, cudaMemcpyHostToDevice, s));
    k_env6_step<<<e6_grid(e->n), E6_BLOCK, 0, s>>>(e->d_state, e->n, az_device_tables(), e->d_action, e->seed, e->first_game, e6_rules(e->rules), e->d_status);
    AZ_CUDA(cudaGetLastError());
    AZ_CUDA(cudaMemcpyAsync(h_status, e->d_status, (size_t)e->n, cudaMemcpyDeviceToHost, s));
    AZ_CUDA(cudaStreamSynchronize(s));
    return AZ_OK;
}

extern "C" int az_env6_query(az_env6* e, uint64_t* h_valid, int8_t* h_status, void* stream)
{
    AZ_REQUIRE(e && (h_valid || h_status), "NULL argument");
    AzDeviceGuard guard(e->device);
    cudaStream_t s = (cudaStream_t)stream;
    k_env6_query<<<e6_grid(e->n), E6_BLOCK, 0, s>>>(e->d_state, e->n, az_device_tables(), e6_rules(e->rules), h_valid ? e->d_valid : nullptr,
                                                   h_status ? e->d_status : nullptr);
    AZ_CUDA(cudaGetLastError());
    if (h_valid) AZ_CUDA(cudaMemcpyAsync(h_valid, e->d_valid, sizeof(uint64_t) * (size_t)e->n, cudaMemcpyDeviceToHost, s));
    if (h_status) AZ_CUDA(cudaMemcpyAsync(h_status, e->d_status, (size_t)e->n, cudaMemcpyDeviceToHost, s));
    AZ_CUDA(cudaStreamSynchronize(s));
    return AZ_OK;
}

extern "C" int az_env6_script_actions(az_env6* e, uint8_t* h_action, void* stream)
{
    AZ_REQUIRE(e && h_action, "NULL argument");
    AzDeviceGuard guard(e->device);
    cudaStream_t s = (cudaStream_t)stream;
    k_env6_script<<<e6_grid(e->n), E6_BLOCK, 0, s>>>(e->d_state, e->n, az_device_tables(), e6_rules(e->rules), e->d_action);
    AZ_CUDA(cudaGetLastError());
    AZ_CUDA(cudaMemcpyAsync(h_action, e->d_action, (size_t)e->n, cudaMemcpyDeviceToHost, s));
    AZ_CUDA(cudaStreamSynchronize(s));
    return AZ_OK;
}

extern "C" int az_env6_export(az_env6* e, uint8_t* h_images, void* stream)
{
    AZ_REQUIRE(e && h_images, "NULL argument");
    AzDeviceGuard guard(e->device);
    cudaStream_t s = (cudaStream_t)stream;
    k_env6_export<<<e6_grid(e->n), E6_BLOCK, 0, s>>>(e->d_state, e->n, e->d_img);
    AZ_CUDA(cudaGetLastError());
    AZ_CUDA(cudaMemcpyAsync(h_images, e->d_img, (size_t)e->n * E6_IMG, cudaMemcpyDeviceToHost, s));
    AZ_CUDA(cudaStreamSynchronize(s));
    return AZ_OK;
}

extern "C" int az_env6_import(az_env6* e, const uint8_t* h_images, void* stream)
{
    AZ_REQUIRE(e && h_images, "NULL argument");
    AzDeviceGuard guard(e->device);
    cudaStream_t s = (cudaStream_t)stream;
    AZ_CUDA(cudaMemcpyAsync(e->d_img, h_images, (size_t)e->n * E6_IMG, cudaMemcpyHostToDevice, s));
    AZ_CUDA(cudaMemsetAsync(e->d_bad, 0, sizeof(int), s));
    e->generation++;
    if (e->rec.out) AZ_CUDA(cudaMemsetAsync(e->rec.len, 0, sizeof(uint32_t) * (size_t)e->n, s));                       // staged samples go
    k_env6_import<<<e6_grid(e->n), E6_BLOCK, 0, s>>>(e->d_state, e->n, e->d_img, e->d_bad);
    AZ_CUDA(cudaGetLastError());
    int bad = 0;
    AZ_CUDA(cudaMemcpyAsync(&bad, e->d_bad, sizeof(int), cudaMemcpyDeviceToHost, s));
    AZ_CUDA(cudaStreamSynchronize(s));
    if (bad) { az_set_error("az_env6_import: %d malformed game image(s)", bad); return AZ_ERR_BAD_STATE; }
    return AZ_OK;
}

extern "C" int az_env6_counters(az_env6* e, az_counters6* h_out, int reset, void* stream)
{
    AZ_REQUIRE(e && h_out, "NULL argument");
    AzDeviceGuard guard(e->device);
    cudaStream_t s = (cudaStream_t)stream;
    unsigned long long h[16];
    AZ_CUDA(cudaMemcpyAsync(h, e->d_counters, sizeof h, cudaMemcpyDeviceToHost, s));
    if (reset) AZ_CUDA(cudaMemsetAsync(e->d_counters, 0, sizeof h, s));
    AZ_CUDA(cudaStreamSynchronize(s));
    h_out->steps = h[0]; h_out->games = h[1]; h_out->draws = h[2];
    for (int p = 0; p < E6_PLAYERS; ++p) h_out->wins[p] = h[3 + p];
    return AZ_OK;
}

// ---- generated games (SIXPLAYER.md §6)
extern "C" int az_env6_play(az_env6* e, const int* seat_kind, uint32_t record_seats, int n_plies, void* stream)
{
    AZ_REQUIRE(e != nullptr, "env is NULL");
    AZ_REQUIRE(seat_kind != nullptr, "seat_kind is NULL");
    AZ_REQUIRE(n_plies >= 0, "n_plies must be >= 0");
    AZ_REQUIRE(record_seats < (1u << E6_PLAYERS), "record_seats has a bit above seat 5");
    AZ_REQUIRE(record_seats == 0 || e->rec.out != nullptr, "record_seats != 0 needs az_env6_record first");
    uint32_t script = 0;
    for (int p = 0; p < E6_PLAYERS; ++p) {
        AZ_REQUIRE(seat_kind[p] == AZ_AGENT6_RANDOM || seat_kind[p] == AZ_AGENT6_SCRIPT,
                   "seat_kind entries must be AZ_AGENT6_RANDOM or AZ_AGENT6_SCRIPT (a searcher cannot play here)");
        if (seat_kind[p] == AZ_AGENT6_SCRIPT) script |= 1u << p;
    }
    AzDeviceGuard guard(e->device);
    cudaStream_t s = (cudaStream_t)stream;
    AZ_CUDA(cudaEventRecord(e->ev0, s));
    // With recording enabled every call runs the recording kernel, record_seats == 0 included: a game with samples staged by an
    // earlier call may end in this one, and its block must be queued (and its staging cleared) before the re-deal.
    if (e->rec.out)
        k_env6_play<true><<<e6_grid(e->n), E6_BLOCK, 0, s>>>(e->d_state, e->n, az_device_tables(), n_plies, e->seed, e->first_game,
                                                           e6_rules(e->rules), script, record_seats, e->rec, e->d_counters);
    else if (script == 0)                                // six random seats, nothing staged: exactly the rollout, at its speed
        k_env6_rollout<<<e6_grid(e->n), E6_BLOCK, 0, s>>>(e->d_state, e->n, az_device_tables(), n_plies, e->seed, e->first_game,
                                                         e6_rules(e->rules), e->d_counters);
    else
        k_env6_play<false><<<e6_grid(e->n), E6_BLOCK, 0, s>>>(e->d_state, e->n, az_device_tables(), n_plies, e->seed, e->first_game,
                                                            e6_rules(e->rules), script, 0u, E6RecDev(), e->d_counters);
    AZ_CUDA(cudaGetLastError());
    AZ_CUDA(cudaEventRecord(e->ev1, s));
    e->timed = true;
    return AZ_OK;
}

extern "C" int az_env6_record(az_env6* e, size_t capacity_samples, int max_samples_per_game)
{
    AZ_REQUIRE(e != nullptr, "env is NULL");
    AZ_REQUIRE(capacity_samples > 0 && max_samples_per_game > 0, "capacity_samples and max_samples_per_game must be positive");
    AZ_REQUIRE(e->rec.out == nullptr, "recording is already enabled on this env");
    AzDeviceGuard guard(e->device);
    const size_t n = (size_t)e->n;
    E6RecDev r;
    cudaError_t ce = cudaMalloc(&r.stage, sizeof(uint32_t) * n * (size_t)max_samples_per_game * E6_STAGE_WORDS);
    if (ce == cudaSuccess) ce = cudaMalloc(&r.len, sizeof(uint32_t) * n);
    if (ce == cudaSuccess) ce = cudaMemset(r.len, 0, sizeof(uint32_t) * n);
    if (ce == cudaSuccess) ce = cudaMalloc(&r.count, 2 * sizeof(unsigned long long));
    if (ce == cudaSuccess) ce = cudaMemset(r.count, 0, 2 * sizeof(unsigned long long));
    if (ce == cudaSuccess) ce = cudaMalloc(&r.out, capacity_samples * (size_t)S6_BYTES);
    if (ce != cudaSuccess) {
        cudaFree(r.stage); cudaFree(r.len); cudaFree(r.count); cudaFree(r.out);
        az_set_error("az_env6_record: %s", cudaGetErrorString(ce));
        return AZ_ERR_CUDA;
    }
    r.max = max_samples_per_game; r.cap = capacity_samples;
    e->rec = r;                                        // rec.out != NULL: recording enabled
    return AZ_OK;
}

extern "C" int az_env6_samples(az_env6* e, uint8_t* h_records, size_t max_records, size_t* n_out, uint64_t* h_dropped, void* stream)
{
    AZ_REQUIRE(e && n_out, "NULL argument");
    AZ_REQUIRE(e->rec.out != nullptr, "az_env6_record has not been called");
    AzDeviceGuard guard(e->device);
    cudaStream_t s = (cudaStream_t)stream;
    unsigned long long h[2];
    AZ_CUDA(cudaMemcpyAsync(h, e->rec.count, sizeof h, cudaMemcpyDeviceToHost, s));
    AZ_CUDA(cudaStreamSynchronize(s));
    AZ_REQUIRE(h[0] <= e->rec.cap, "sample queue corrupted: committed count exceeds the capacity");
    const size_t have = (size_t)h[0];                  // committed records: az_rec_reserve never reserves past the capacity
    if (h_dropped) *h_dropped = h[1];
    *n_out = have;
    if (!h_records && have) return AZ_OK;              // size query; with an empty queue the call drains (resets the dropped count)
    AZ_REQUIRE(max_records >= have, "h_records is too small: query the size with h_records = NULL first");
    if (have) AZ_CUDA(cudaMemcpyAsync(h_records, e->rec.out, have * (size_t)S6_BYTES, cudaMemcpyDeviceToHost, s));
    AZ_CUDA(cudaMemsetAsync(e->rec.count, 0, sizeof h, s));
    AZ_CUDA(cudaStreamSynchronize(s));
    return AZ_OK;
}
