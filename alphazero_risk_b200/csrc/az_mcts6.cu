// az_mcts6.cu — lockstep MCTS for the SIX-PLAYER extension (SIXPLAYER.md; BASELINE.json configs[3]) and the az_mcts6_* C ABI.
//
// No reference parity exists for this game (PLAYER_COUNT = 2 upstream, /root/reference/src/risk_game/state/state.h:13); the
// checker is oracle/risk6_oracle.c (r6_mcts_search), compared bit for bit by tests/test_mcts6_gpu.py.  The search is the
// reference's AlphaZeroMCTS (player/alpha_zero/alphazero_mcts.cpp: PUCT :67-119, search :322-377, addValue :8-21, policy from the
// visit counts :121-148, move choice :379-412) with the two changes SIXPLAYER.md states: the table is cleared before every search
// (no trimNodes carry-over), and a leaf's scalar value belongs to the seat to move there — on the way up a node whose mover is
// that seat receives +v, every other node -v / 5.  az_rules.concurrent_descents = K descents per tree per leaf batch in the two-player
// lockstep schedule (az_mcts.cu, SIXPLAYER.md §2; checker oracle/risk6_lockstep.c): descent j of round r uses the dice of simulation
// r * K + j and selects after descents 0..j-1 under the active_N rule; the round's leaves are evaluated as one batch of K * n positions,
// then expanded and backed up in descent order.  K = 1 is the one-descent search (THREADS_PER_MCTS = 1 semantics).
// An evaluator with a six-seat value vector (a 6-output network, AZ_EVAL_PSEUDO6; SIXPLAYER.md §2) gives each leaf v[6] relative to its
// seat to move L, and a path node whose mover is s receives v[(s - L + 6) % 6] instead; a finished game backs up as above.
//
// Mapping: one warp per game.  The game logic of a descent (status, legal mask, transition: az_game6.cuh) runs on lane 0 over the
// warp's shared-memory state row — the six-seat rules are thread code, shared with the environment kernels —, the table work
// (hash-window probing, node records, PUCT argmax) uses all 32 lanes.  The leaf batch goes through the same policy / value tower
// as the two-player game (k_env6_encode -> az_nn_forward_dev).  Deliberately simpler than az_mcts.cu (one pool per game, no tree
// reuse between searches): the tower is what it spends its time in.  The six-player arena (az_arena6_*, end of this file) restricts a search to
// the games waiting for its searcher and compacts their leaf batch.
//
// Training samples (AZ_SAMPLE6_BYTES records, az_samples6.cuh): k_mcts6_finish stages (state words, pi) per real move; the game's warp
// turns them into records in k_mcts6_rec_end once the game has ended.
#include <algorithm>
#include <cstring>
#include <new>

#include "az_common.cuh"
#include "az_arena.cuh"
#include "az_game6.cuh"
#include "az_samples6.cuh"
#include "az_nn.cuh"
#include "az_pseudo_net.h"

#define M6_WARPS 4
#define M6_FULL 0xffffffffu
#define M6_KEY 27                       // state words 0..26 identify a position (word 27 = the slot's move counter)
#define M6_NODE_WORDS 192
#define M6_VALID 28
#define M6_SUMN 30
#define M6_VALUE 31
#define M6_P 32
#define M6_Q 76
#define M6_N 120
enum { M6_EVAL_NN = 0, M6_EVAL_PSEUDO = 1, M6_EVAL_UNIFORM = 2, M6_EVAL_PSEUDO6 = 3 };
enum { M6C_SIMS = 0, M6C_EVALS = 1, M6C_OVERFLOW = 2, M6C_STEPS = 3, M6C_GAMES = 4, M6C_DRAWS = 5, M6C_WIN0 = 6, M6C_N = 12 };

struct Mcts6Dev {
    int n, cap, H, dmax;
    int K;                  // descents per tree per round (az_rules.concurrent_descents); descent slot = j * n + game
    uint32_t* nodes;        // [n][cap][M6_NODE_WORDS]; the N word of a move: N in the low 24 bits, active_N in the top byte
    uint32_t* index;        // [n][H]   0 = empty, else tag16 << 16 | (node + 1)
    uint32_t* count;        // [n]
    uint32_t* path;         // [K*n][dmax]  node | move << 16 | mover << 22
    uint32_t* path_len;     // [K*n]
    uint32_t* leaf_state;   // [28][K*n]
    uint64_t* leaf_valid;   // [K*n]
    int32_t* pending;       // [K*n]
    float* term_value;      // [K*n]   value of a descent that ended in a finished game
    int32_t* term_seat;     // [K*n]   and the seat it belongs to
    float* nn_policy;       // [K*n][43]
    float* nn_value;        // [K*n][vo]   the evaluator's value (vector) per descent slot
    int vo;                 // value components per leaf: 1 (the scalar rule) or 6 (per-seat backup)
    uint32_t* root_state;   // the env6 state [28][n]
    uint32_t* out_visits; float* out_pi; uint8_t* out_move; int8_t* out_status; float* out_q; float* out_p; uint32_t* out_sumn; int32_t* out_table;
    unsigned long long* counters;
    float c1, c2, cpuct;
    uint64_t seed; uint32_t first_game;
    AzRulesDev rules;
    int eval_mode, temp_threshold;
    // sample recording (az_selfplay6_record): per-game staging until the game ends
    uint32_t* rec_state;    // [n][rec_moves][27]  state words 0..26 of the root before the move
    float* rec_pi;          // [n][rec_moves][43]  policy target
    uint32_t* rec_len;      // [n]                 staged samples of the running game (> rec_moves = overflowed)
    int8_t* rec_end;        // [n]                 status of a game that ended at the last real move, else AZ_STATUS_RUNNING
    uint8_t* rec_out;       // [rec_cap][288]      records of finished games
    unsigned long long* rec_count;   // [2]        records in rec_out, samples dropped (staging or queue full)
    int rec_moves; unsigned long long rec_cap;
    // six-player arena (az_arena6_play sets these around a search; NULL = every game, ids first_game + gi)
    const uint8_t* sel; int sel_value;    // only games with sel[gi] == sel_value search
    const uint32_t* game_id;              // [n] the game id of the descents' dice and the real move, replacing first_game + gi
};

struct M6Smem {
    uint64_t tab[AZ_TABLE_U64];
    uint32_t row[M6_WARPS][E6_WORDS];
    uint32_t scratch[M6_WARPS][12];
};

// lane-0 game context over the warp's row: the column accessors of az_game.cuh with a 4-byte stride are plain byte rows
__device__ __forceinline__ void m6_bind(E6Ctx& c, uint32_t* row, uint32_t* scratch)
{
    c.army.base = (uint8_t*)row; c.army.stride_bytes = 4;
    c.owner.base = (uint8_t*)(row + 11); c.owner.stride_bytes = 4;
    c.scratch.base = (uint8_t*)scratch; c.scratch.stride_bytes = 4;
}
__device__ __forceinline__ void m6_unpack_row(E6Ctx& c, const uint32_t* row)
{
    e6_masks(c);
    e6_unpack(c.g, row[22], row[23], row[24], row[25], row[26]);
    c.ply = row[27];
}
__device__ __forceinline__ void m6_pack_row(const E6Ctx& c, uint32_t* row)
{
    const AzGame6& g = c.g;
    row[22] = g.cards_lo;
    row[23] = (g.cards_hi & 0xffffu) | ((g.allow_draw & 0xffu) << 16) | ((g.attacks & 0xffu) << 24);
    row[24] = (g.round & 0xffffu) | (g.cur << 16) | (g.card_sets << 24);
    row[25] = (g.reinf & 0xffu) | (g.phase << 8) | (g.mob_from << 16) | (g.mob_to << 24);
    row[26] = g.pools & 0xffffffu;
}

__device__ __forceinline__ uint64_t m6_hash(uint32_t kw, int lane)
{
    uint64_t h = ((uint64_t)kw + 0x9E3779B97F4A7C15ull * (uint64_t)(lane + 1)) * 0xD6E8FEB86659FD93ull;
    h ^= h >> 29;
    if (lane >= M6_KEY) h = 0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        uint32_t lo = __shfl_xor_sync(M6_FULL, (uint32_t)h, o), hi = __shfl_xor_sync(M6_FULL, (uint32_t)(h >> 32), o);
        h += ((uint64_t)hi << 32) | lo;
    }
    return az_pn_mix(h);
}
__device__ __forceinline__ bool m6_skip(const Mcts6Dev& m, int gi) { return m.sel && m.sel[gi] != (uint8_t)m.sel_value; }
__device__ __forceinline__ uint32_t m6_game(const Mcts6Dev& m, int gi) { return m.game_id ? m.game_id[gi] : m.first_game + (uint32_t)gi; }
__device__ __forceinline__ uint32_t* m6_node(const Mcts6Dev& m, int gi, uint32_t idx) { return m.nodes + ((size_t)gi * m.cap + idx) * M6_NODE_WORDS; }

// the node of the position whose key words sit in lanes 0..26 (kw), or -1; empty_slot = where an insert would go
__device__ __forceinline__ int m6_lookup(const Mcts6Dev& m, int gi, uint64_t h, uint32_t kw, int lane, int& empty_slot)
{
    const uint32_t* base = m.index + (size_t)gi * m.H;
    const uint32_t tag = (uint32_t)(h >> 48) & 0xffffu, start = (uint32_t)h & (uint32_t)(m.H - 1);
    empty_slot = -1;
    for (int win = 0; win < m.H; win += 32) {
        const uint32_t slot = (start + (uint32_t)win + (uint32_t)lane) & (uint32_t)(m.H - 1);
        const uint32_t e = base[slot];
        const uint32_t empties = __ballot_sync(M6_FULL, e == 0);
        uint32_t matches = __ballot_sync(M6_FULL, e != 0 && (e >> 16) == tag);
        const int first_empty = empties ? (__ffs((int)empties) - 1) : 32;
        if (first_empty < 32) matches &= (1u << first_empty) - 1u;
        while (matches) {
            const int l = __ffs((int)matches) - 1; matches &= matches - 1;
            const uint32_t idx = (__shfl_sync(M6_FULL, e, l) & 0xffffu) - 1u;
            const uint32_t* nd = m6_node(m, gi, idx);
            const uint32_t w = lane < M6_KEY ? nd[lane] : 0u;
            if (__ballot_sync(M6_FULL, w == kw) == M6_FULL) return (int)idx;
        }
        if (first_empty < 32) { empty_slot = (int)((start + (uint32_t)win + (uint32_t)first_empty) & (uint32_t)(m.H - 1)); return -1; }
    }
    return -1;
}

// getNextBestMoveAndSetVisited (alphazero_mcts.cpp:67-119), ascending move index on ties.  A move with N == 0 && active_N == 1 (one
// descent of the round is about to open it) is passed over (:91-93); if nothing else can be chosen the best such move is requested
// again (:108-111).  The chosen move's active_N is incremented.  With K = 1 no mark is ever 1 at selection: the plain argmax.
__device__ __forceinline__ int m6_select(const Mcts6Dev& m, uint32_t* nd, int lane)
{
    const uint64_t valid = (uint64_t)nd[M6_VALID] | ((uint64_t)nd[M6_VALID + 1] << 32);
    const float sq = __fsqrt_rn(__fadd_rn(1.0f, (float)nd[M6_SUMN]));
    float bu = -INFINITY, du = -INFINITY; int bi = 64, di = 64;
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const int i = lane + 32 * k;
        if (i < AZ_MOVES && ((valid >> i) & 1ull)) {
            const float P = __uint_as_float(nd[M6_P + i]), Q = __uint_as_float(nd[M6_Q + i]);
            const uint32_t nw = nd[M6_N + i], N = nw & 0xffffffu;
            const float noiseP = __fadd_rn(__fmul_rn(m.c1, P), m.c2);
            const float v = __fmul_rn(__fmul_rn(noiseP, m.cpuct), sq);
            const float u = __fadd_rn(Q, __fdiv_rn(v, __fadd_rn(1.0f, (float)N)));
            if (N == 0u && (nw >> 24) == 1u) { if (u > du) { du = u; di = i; } }
            else if (u > bu) { bu = u; bi = i; }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        float ou = __shfl_xor_sync(M6_FULL, bu, o); int oi = __shfl_xor_sync(M6_FULL, bi, o);
        if (ou > bu || (ou == bu && oi < bi)) { bu = ou; bi = oi; }
        ou = __shfl_xor_sync(M6_FULL, du, o); oi = __shfl_xor_sync(M6_FULL, di, o);
        if (ou > du || (ou == du && oi < di)) { du = ou; di = oi; }
    }
    if (bi == 64) bi = di;
    __syncwarp();
    if (lane == 0 && bi < AZ_MOVES) nd[M6_N + bi] += 1u << 24;
    return bi;
}

// addValue up the recorded path of descent slot `slot`: +v for the nodes of the seat the leaf value belongs to, -v / 5 for every other
// node; with a value vector vec (NULL: the scalar rule; seat = the leaf's seat to move) a node whose mover is s receives
// vec[(s - seat + 6) % 6].  Each step takes the descent's active_N mark off its move
__device__ __forceinline__ void m6_backup(const Mcts6Dev& m, int slot, int gi, float v, uint32_t seat, uint32_t len, int lane, const float* vec)
{
    __syncwarp();
    if (lane == 0) {
        const float other = __fdiv_rn(-v, 5.0f);
        for (int d = (int)len - 1; d >= 0; --d) {
            const uint32_t e = m.path[(size_t)slot * m.dmax + d];
            const uint32_t idx = e & 0xffffu, mv = (e >> 16) & 63u, mover = (e >> 22) & 7u;
            const float val = vec ? vec[(mover + E6_PLAYERS - seat) % E6_PLAYERS] : (mover == seat ? v : other);
            uint32_t* nd = m6_node(m, gi, idx);
            const uint32_t nw = nd[M6_N + mv], N = nw & 0xffffffu;
            const float Q = __uint_as_float(nd[M6_Q + mv]);
            const float q = N == 0 ? val : __fdiv_rn(__fadd_rn(__fmul_rn((float)N, Q), val), (float)(N + 1u));
            nd[M6_Q + mv] = __float_as_uint(q);
            nd[M6_N + mv] = (N + 1u) | (((nw >> 24) - 1u) << 24);
            nd[M6_SUMN] += 1u;
        }
        if (len > 0) atomicAdd(&m.counters[M6C_SIMS], 1ull);
        m.path_len[slot] = 0;
    }
    __syncwarp();
}

// a descent that overflowed the path: its marks come off without a backup (it is counted as an error, not as a simulation)
__device__ __forceinline__ void m6_unmark(const Mcts6Dev& m, int slot, int gi, uint32_t len, int lane)
{
    __syncwarp();
    if (lane == 0)
        for (uint32_t d = 0; d < len; ++d) {
            const uint32_t e = m.path[(size_t)slot * m.dmax + d];
            m6_node(m, gi, e & 0xffffu)[M6_N + ((e >> 16) & 63u)] -= 1u << 24;
        }
    __syncwarp();
}

__device__ __forceinline__ uint64_t m6_pn_key(const uint32_t* row)
{
    const uint8_t* army = (const uint8_t*)row; const uint8_t* owner = (const uint8_t*)(row + 11);
    uint8_t land[AZ_LANDS];
    for (int i = 0; i < AZ_LANDS; ++i) land[i] = (uint8_t)(army[i] + 40 * owner[i]);
    return az_pn_key(land, (int)((row[24] >> 16) & 0xffu), (int)(row[24] & 0xffffu), (int)((row[25] >> 8) & 0xffu));
}

// complete descent slot `slot` of the previous round: expand the queued leaf with the evaluator's output (StateSimulations ctor :26-42
// after NNOutputData::normalize, alphazero_nn_data.cpp:3-27), or take the finished game's value, and back it up.  A leaf an earlier
// descent of the round has added is not inserted again (StateSimulationsStorage::add :203-215); its own value is still backed up.
__device__ __forceinline__ void m6_complete(const Mcts6Dev& m, int slot, int gi, uint32_t* row, int lane)
{
    const uint32_t len = m.path_len[slot];
    float v = m.term_value[slot];
    uint32_t seat = (uint32_t)m.term_seat[slot];
    const float* vec = nullptr;
    if (m.pending[slot]) {
        __syncwarp();
        if (lane < E6_WORDS) row[lane] = m.leaf_state[(size_t)lane * m.K * m.n + slot];
        __syncwarp();
        const uint64_t valid = m.leaf_valid[slot];
        float p0 = 0.0f, p1 = 0.0f, value;
        if (m.eval_mode == M6_EVAL_NN) {
            p0 = m.nn_policy[(size_t)slot * AZ_MOVES + lane];
            if (lane + 32 < AZ_MOVES) p1 = m.nn_policy[(size_t)slot * AZ_MOVES + 32 + lane];
            value = m.nn_value[(size_t)slot * m.vo];
        } else if (m.eval_mode == M6_EVAL_PSEUDO || m.eval_mode == M6_EVAL_PSEUDO6) {
            const uint64_t key = m6_pn_key(row);
            p0 = az_pn_policy(key, lane);
            if (lane + 32 < AZ_MOVES) p1 = az_pn_policy(key, lane + 32);
            value = az_pn_value(key);
            if (m.eval_mode == M6_EVAL_PSEUDO6 && lane < E6_PLAYERS) m.nn_value[(size_t)slot * E6_PLAYERS + lane] = az_pn_value6(key, lane);
        } else { p0 = 1.0f / 43.0f; p1 = lane + 32 < AZ_MOVES ? 1.0f / 43.0f : 0.0f; value = 0.0f; }
        if (!((valid >> lane) & 1ull)) p0 = 0.0f;
        if (lane + 32 >= AZ_MOVES || !((valid >> (lane + 32)) & 1ull)) p1 = 0.0f;
        float sum = 0.0f;                                    // ascending-order sum; the masked entries are +0 and x + 0 == x exactly
#pragma unroll
        for (int i = 0; i < 32; ++i) sum = __fadd_rn(sum, __shfl_sync(M6_FULL, p0, i));
#pragma unroll
        for (int i = 0; i < AZ_MOVES - 32; ++i) sum = __fadd_rn(sum, __shfl_sync(M6_FULL, p1, i));
        if (p0 > 0.0f) p0 = __fdiv_rn(p0, sum);
        if (p1 > 0.0f) p1 = __fdiv_rn(p1, sum);
        const uint32_t kw = lane < M6_KEY ? row[lane] : 0u;
        const uint64_t h = m6_hash(kw, lane);
        int ins;
        const int found = m6_lookup(m, gi, h, kw, lane, ins);
        const uint32_t cnt = m.count[gi];
        if (found < 0 && (int)cnt < m.cap && ins >= 0) {
            uint32_t* nd = m6_node(m, gi, cnt);
            if (lane < M6_KEY) nd[lane] = kw;
            if (lane == 27) nd[M6_VALID] = (uint32_t)valid;
            if (lane == 28) nd[M6_VALID + 1] = (uint32_t)(valid >> 32);
            if (lane == 29) nd[M6_SUMN] = 0u;
            if (lane == 30) nd[M6_VALUE] = __float_as_uint(value);
            nd[M6_P + lane] = __float_as_uint(p0); nd[M6_Q + lane] = 0u; nd[M6_N + lane] = 0u;
            if (lane < AZ_MOVES - 32) { nd[M6_P + 32 + lane] = __float_as_uint(p1); nd[M6_Q + 32 + lane] = 0u; nd[M6_N + 32 + lane] = 0u; }
            __syncwarp();
            if (lane == 0) { m.count[gi] = cnt + 1; m.index[(size_t)gi * m.H + ins] = (((uint32_t)(h >> 48) & 0xffffu) << 16) | (cnt + 1u); }
            __syncwarp();
        } else if (found < 0 && lane == 0) atomicAdd(&m.counters[M6C_OVERFLOW], 1ull);
        v = value;
        seat = (row[24] >> 16) & 0xffu;                      // the seat to move at the leaf
        if (lane == 0) { m.pending[slot] = 0; atomicAdd(&m.counters[M6C_EVALS], 1ull); }
        if (m.vo == E6_PLAYERS) vec = m.nn_value + (size_t)slot * E6_PLAYERS;   // m6_backup's __syncwarp orders the lanes' writes
    }
    m6_backup(m, slot, gi, v, seat, len, lane, vec);
}

// one descent from the root into descent slot `slot` (AlphaZeroMCTS::search :322-377 as a loop); sim < 0: only make sure the root is
// in the table.  A descent that ends in a finished game backs up at once; one that reaches an unseen position queues it.
__device__ __forceinline__ void m6_descend(const Mcts6Dev& m, int slot, int gi, uint32_t* row, uint32_t* scratch, const AzTables& T, int sim, int lane)
{
    __syncwarp();
    if (lane < E6_WORDS) row[lane] = m.root_state[(size_t)lane * m.n + gi];
    __syncwarp();
    E6Ctx c; m6_bind(c, row, scratch);
    AzDicePhilox dice;
    if (lane == 0) { m6_unpack_row(c, row); dice.init(m.seed, m6_game(m, gi), c.ply, (uint32_t)(sim < 0 ? 0 : sim)); }
    uint32_t depth = 0;
    for (;;) {
        int st = 0; uint64_t valid = 0; uint32_t mover = 0;
        if (lane == 0) { st = e6_status(c.g, m.rules); valid = st == AZ_STATUS_RUNNING ? e6_valid(c.g, T, m.rules) : 0ull; mover = c.g.cur; }
        st = __shfl_sync(M6_FULL, st, 0);
        mover = __shfl_sync(M6_FULL, mover, 0);
        valid = ((uint64_t)__shfl_sync(M6_FULL, (uint32_t)(valid >> 32), 0) << 32) | __shfl_sync(M6_FULL, (uint32_t)valid, 0);
        if (st != AZ_STATUS_RUNNING) {                       // a finished game: its value belongs to the winner (a draw is worth 0 to everyone)
            const float tv = st == AZ_STATUS_DRAW ? 0.0f : 1.0f;
            const uint32_t seat = st == AZ_STATUS_DRAW ? mover : (uint32_t)st;
            if (lane == 0) { m.term_value[slot] = tv; m.term_seat[slot] = (int32_t)seat; m.pending[slot] = 0; }
            m6_backup(m, slot, gi, tv, seat, depth, lane, nullptr);
            depth = 0;
            break;
        }
        const uint32_t kw = lane < M6_KEY ? row[lane] : 0u;
        const uint64_t h = m6_hash(kw, lane);
        int ins;
        const int idx = m6_lookup(m, gi, h, kw, lane, ins);
        if (idx < 0) {                                       // unseen position: queue it for the evaluator
            if (lane < E6_WORDS) m.leaf_state[(size_t)lane * m.K * m.n + slot] = row[lane];
            if (lane == 0) { m.leaf_valid[slot] = valid; m.pending[slot] = 1; m.term_value[slot] = 0.0f; m.term_seat[slot] = (int32_t)mover; }
            break;
        }
        if (sim < 0) { if (lane == 0) m.pending[slot] = 0; break; }
        if ((int)depth >= m.dmax) {
            m6_unmark(m, slot, gi, depth, lane);
            if (lane == 0) { atomicAdd(&m.counters[M6C_OVERFLOW], 1ull); m.pending[slot] = 0; m.term_value[slot] = 0.0f; }
            depth = 0; break;
        }
        const int mv = m6_select(m, m6_node(m, gi, (uint32_t)idx), lane);
        if (lane == 0) {
            m.path[(size_t)slot * m.dmax + depth] = (uint32_t)idx | ((uint32_t)mv << 16) | (mover << 22);
            e6_move(c, T, m.rules, mv, dice);
            m6_pack_row(c, row);
        }
        __syncwarp();
        depth++;
    }
    if (lane == 0) m.path_len[slot] = depth;
    __syncwarp();
}

__global__ void __launch_bounds__(M6_WARPS * 32) k_mcts6_begin(Mcts6Dev m)
{
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int gi = blockIdx.x * M6_WARPS + warp;
    if (gi >= m.n || m6_skip(m, gi)) return;
    uint32_t* ix = m.index + (size_t)gi * m.H;
    for (int i = lane; i < m.H; i += 32) ix[i] = 0u;
    if (lane == 0) m.count[gi] = 0u;
    if (lane < m.K) {
        const size_t slot = (size_t)lane * m.n + gi;
        m.pending[slot] = 0; m.path_len[slot] = 0u; m.term_value[slot] = 0.0f; m.term_seat[slot] = 0;
    }
}

// one round: complete the K descents of the previous round in order, then (do_descent) start the K descents of this one in order;
// round < 0: the root round.  Bounded to the register budget of five blocks per SM, which K = 1 had without the bound.
__global__ void __launch_bounds__(M6_WARPS * 32, 5) k_mcts6_sim(Mcts6Dev m, const uint64_t* __restrict__ g_tab, int round, int do_descent)
{
    __shared__ M6Smem sm;
    for (int i = threadIdx.x; i < AZ_TABLE_U64; i += blockDim.x) sm.tab[i] = g_tab[i];
    __syncthreads();
    const AzTables T = az_tables_from_smem(sm.tab);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int gi = blockIdx.x * M6_WARPS + warp;
    if (gi >= m.n || m6_skip(m, gi)) return;
    for (int j = 0; j < m.K; ++j) m6_complete(m, j * m.n + gi, gi, sm.row[warp], lane);    // the previous round, in descent order
    if (!do_descent) return;
    if (round < 0) m6_descend(m, gi, gi, sm.row[warp], sm.scratch[warp], T, -1, lane);        // the root round: slot 0 only
    else for (int j = 0; j < m.K; ++j) m6_descend(m, j * m.n + gi, gi, sm.row[warp], sm.scratch[warp], T, round * m.K + j, lane);
}

// after the last simulation: root statistics (calculateMoveProbability :121-148), move choice (pickHigestWeightedMove :397-412 /
// pickRandomWeightedMove :379-395 under the temperature rule), optionally the real move on the env6 state (+ re-deal of finished
// games when auto_reset).  The float arithmetic runs on lane 0 in the oracle's order.
__global__ void __launch_bounds__(M6_WARPS * 32) k_mcts6_finish(Mcts6Dev m, const uint64_t* __restrict__ g_tab, int pick_mode, int apply_move, int auto_reset)
{
    __shared__ M6Smem sm;
    for (int i = threadIdx.x; i < AZ_TABLE_U64; i += blockDim.x) sm.tab[i] = g_tab[i];
    __syncthreads();
    const AzTables T = az_tables_from_smem(sm.tab);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int gi = blockIdx.x * M6_WARPS + warp;
    if (gi >= m.n || m6_skip(m, gi)) return;
    uint32_t* row = sm.row[warp];
    m6_complete(m, gi, gi, row, lane);          // slot 0; with K > 1 the host has completed the last round's slots already
    __syncwarp();
    if (lane < E6_WORDS) row[lane] = m.root_state[(size_t)lane * m.n + gi];
    __syncwarp();
    const uint32_t kw = lane < M6_KEY ? row[lane] : 0u;
    const uint64_t h = m6_hash(kw, lane);
    int ins;
    const int idx = m6_lookup(m, gi, h, kw, lane, ins);
    if (lane != 0) return;
    E6Ctx c; m6_bind(c, row, sm.scratch[warp]);
    m6_unpack_row(c, row);
    int status = e6_status(c.g, m.rules);
    int move = AZ_NONE;
    const uint32_t game = m6_game(m, gi);
    uint32_t* ov = m.out_visits + (size_t)gi * AZ_MOVES; float* op = m.out_pi + (size_t)gi * AZ_MOVES;
    float* oq = m.out_q + (size_t)gi * AZ_MOVES; float* opp = m.out_p + (size_t)gi * AZ_MOVES;
    for (int i = 0; i < AZ_MOVES; ++i) { ov[i] = 0u; op[i] = 0.0f; oq[i] = 0.0f; opp[i] = 0.0f; }
    m.out_sumn[gi] = 0u; m.out_table[gi] = (int32_t)m.count[gi];
    if (status == AZ_STATUS_RUNNING && idx >= 0) {
        const uint32_t* nd = m6_node(m, gi, (uint32_t)idx);
        const uint64_t valid = (uint64_t)nd[M6_VALID] | ((uint64_t)nd[M6_VALID + 1] << 32);
        float sum = 0.0f;
        for (int i = 0; i < AZ_MOVES; ++i) if ((valid >> i) & 1ull) {
            const uint32_t N = nd[M6_N + i] & 0xffffffu;         // the top byte is active_N
            ov[i] = N; oq[i] = __uint_as_float(nd[M6_Q + i]); opp[i] = __uint_as_float(nd[M6_P + i]);
            op[i] = (float)N; sum = __fadd_rn(sum, op[i]);
        }
        for (int i = 0; i < AZ_MOVES; ++i) op[i] = __fdiv_rn(op[i], sum);
        m.out_sumn[gi] = nd[M6_SUMN];
        const bool sample = pick_mode == 1 && (int)c.g.round <= m.temp_threshold;
        const az_u32x4 blk = az_rng_block(m.seed, game, c.ply, AZ_STREAM_REAL, 0);
        if (!sample) {
            float best = 0.0f;
            for (int i = 0; i < AZ_MOVES; ++i) if (op[i] > best) { best = op[i]; move = i; }
        } else {
            float tot = 0.0f;
            for (int i = 0; i < AZ_MOVES; ++i) tot = __fadd_rn(tot, op[i]);
            const float a = __fmul_rn(tot, az_rng_unit_float(blk.z));
            float it = 0.0f;
            for (int i = 0; i < AZ_MOVES; ++i) { it = __fadd_rn(it, op[i]); if (it >= a) { move = i; break; } }
        }
        if (apply_move && move != AZ_NONE) {
            if (m.rec_out) {                                 // stage (root before the move, pi); the records are written when the game ends
                const uint32_t k = m.rec_len[gi];
                if (k < (uint32_t)m.rec_moves) {
                    uint32_t* rs = m.rec_state + ((size_t)gi * m.rec_moves + k) * S6_IMG_WORDS;
                    float* rp = m.rec_pi + ((size_t)gi * m.rec_moves + k) * AZ_MOVES;
                    for (int w = 0; w < S6_IMG_WORDS; ++w) rs[w] = row[w];
                    for (int i = 0; i < AZ_MOVES; ++i) rp[i] = op[i];
                }
                m.rec_len[gi] = k + 1;                       // > rec_moves marks the game's samples as overflowed (dropped at the end)
            }
            E6DiceWord dice; dice.w = blk.x;
            e6_move(c, T, m.rules, move, dice);
            c.ply++;
            atomicAdd(&m.counters[M6C_STEPS], 1ull);
            status = e6_status(c.g, m.rules);
            if (status != AZ_STATUS_RUNNING) {
                atomicAdd(&m.counters[M6C_GAMES], 1ull);
                if (status == AZ_STATUS_DRAW) atomicAdd(&m.counters[M6C_DRAWS], 1ull); else atomicAdd(&m.counters[M6C_WIN0 + status], 1ull);
                if (m.rec_out) m.rec_end[gi] = (int8_t)status;    // before the re-deal: the staged samples belong to this result
                if (auto_reset) e6_new_game(c, m.seed, game, c.ply);
            }
            m6_pack_row(c, row);
            for (int w = 0; w < 27; ++w) m.root_state[(size_t)w * m.n + gi] = row[w];
            m.root_state[(size_t)27 * m.n + gi] = c.ply;
        }
    }
    m.out_move[gi] = (uint8_t)move;
    m.out_status[gi] = (int8_t)status;
}

// the staged samples of every game that ended at the last real move -> records with their value targets, one contiguous block per game
// in the output queue (az_rec_reserve: a game that overflowed its staging or does not fit is dropped whole and counted).  One warp per
// game; the lanes write the game's records word by word.
__global__ void __launch_bounds__(M6_WARPS * 32) k_mcts6_rec_end(Mcts6Dev m)
{
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int gi = blockIdx.x * M6_WARPS + warp;
    if (gi >= m.n) return;
    const int status = m.rec_end[gi];
    if (status == AZ_STATUS_RUNNING) return;
    const uint32_t len = m.rec_len[gi];
    unsigned long long base = 0;
    int ok = 0;
    if (lane == 0 && len > 0) ok = az_rec_reserve(m.rec_count, m.rec_cap, len, len <= (uint32_t)m.rec_moves, &base);
    ok = __shfl_sync(M6_FULL, ok, 0);
    base = ((unsigned long long)__shfl_sync(M6_FULL, (uint32_t)(base >> 32), 0) << 32) | __shfl_sync(M6_FULL, (uint32_t)base, 0);
    if (ok) {
        const uint32_t* rs = m.rec_state + (size_t)gi * m.rec_moves * S6_IMG_WORDS;
        const float* rp = m.rec_pi + (size_t)gi * m.rec_moves * AZ_MOVES;
        uint32_t* dst = (uint32_t*)(m.rec_out + base * S6_BYTES);
        for (uint32_t j = (uint32_t)lane; j < len * S6_WORDS; j += 32) {
            const uint32_t i = j / S6_WORDS, k = j % S6_WORDS;
            dst[j] = s6_record_word(rs + (size_t)i * S6_IMG_WORDS, rp + (size_t)i * AZ_MOVES, status, (int)k);
        }
    }
    if (lane == 0) { m.rec_len[gi] = 0; m.rec_end[gi] = AZ_STATUS_RUNNING; }
}

// the six-seat network input (SIXPLAYER.md, e6_encode_position) of column i of the SoA state st [28][stride], P = 13 or 16 planes
template <int P>
__device__ __forceinline__ void m6_encode_game(const uint32_t* __restrict__ st, int stride, int i, float* __restrict__ out)
{
    uint32_t row[E6_WORDS];
    for (int w = 0; w < E6_WORDS; ++w) row[w] = st[(size_t)w * stride + i];
    const uint32_t cur = (row[24] >> 16) & 0xffu, phase = (row[25] >> 8) & 0xffu, attacks = (row[23] >> 24) & 0xffu, allow = (row[23] >> 16) & 0xffu;
    e6_encode_position<P>((const uint8_t*)row, (const uint8_t*)(row + 11), cur, phase, attacks, allow, out);
}
// one thread per position: columns 0..count-1 of the SoA state st [28][stride]
template <int P>
__global__ void __launch_bounds__(128) k_env6_encode(const uint32_t* __restrict__ st, int stride, int count, float* __restrict__ x)
{
    const int i = blockIdx.x * 128 + threadIdx.x;
    if (i >= count) return;
    m6_encode_game<P>(st, stride, i, x + (size_t)i * 42 * P);
}

// arena leaf batches: row j * count + k = the leaf of descent slot j * n + games[k] (games = the games that search this tick, k_used =
// descent slots per game in the batch, leaf state stride K * n), and the network's outputs (policy [43], value [vo]) back to those slots
template <int P>
__global__ void __launch_bounds__(128) k_env6_encode_list(const uint32_t* __restrict__ st, int stride, int n, const int32_t* __restrict__ games,
                                                          int count, int k_used, float* __restrict__ x)
{
    const int i = blockIdx.x * 128 + threadIdx.x;
    if (i >= count * k_used) return;
    const int j = i / count, k = i - j * count;
    m6_encode_game<P>(st, stride, j * n + games[k], x + (size_t)i * 42 * P);
}
__global__ void __launch_bounds__(256) k_mcts6_scatter_evals(const float* __restrict__ pol_c, const float* __restrict__ val_c,
                                                             const int32_t* __restrict__ games, int count, int n, int k_used, int vo,
                                                             float* __restrict__ pol, float* __restrict__ val)
{
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= count * k_used * (AZ_MOVES + vo)) return;
    const int c = i / (AZ_MOVES + vo), e = i - c * (AZ_MOVES + vo);
    const int j = c / count, k = c - j * count;
    const size_t slot = (size_t)j * n + games[k];
    if (e < AZ_MOVES) pol[slot * AZ_MOVES + e] = pol_c[(size_t)c * AZ_MOVES + e];
    else val[slot * vo + (e - AZ_MOVES)] = val_c[(size_t)c * vo + (e - AZ_MOVES)];
}

// ---------------------------------------------------------------- host side
struct az_env6;
uint32_t* az_env6_state_ptr(az_env6* e); int az_env6_n(const az_env6* e); int az_env6_device(const az_env6* e);
uint64_t az_env6_seed(const az_env6* e); uint32_t az_env6_first_game(const az_env6* e); const az_rules* az_env6_rules(const az_env6* e);
uint64_t az_env6_generation(const az_env6* e);

struct az_mcts6 {
    az_env6* env = nullptr; az_nn* nn = nullptr;
    int evaluator = M6_EVAL_NN, precision = AZ_NN_FP32, device = 0, sims = 0;
    Mcts6Dev d;
    float* d_x = nullptr;
    uint64_t rec_generation = 0;    // the env's deal generation the staged samples belong to
    // arena: only the listed games go through the network (az_arena6_play sets these around a search; the buffers are the arena's)
    const int32_t* eval_games = nullptr;    // ascending list of the searching games
    int eval_count = 0;                     // its length; 0 = every game is evaluated
    float* eval_pol = nullptr; float* eval_val = nullptr;   // compacted outputs [count][43], [count][vo]
    std::vector<void*> allocs;
};

template <class T> static int m6_alloc(az_mcts6* mc, T** p, size_t count, bool zero = true)
{
    AZ_CUDA(cudaMalloc(p, sizeof(T) * count));
    if (zero) AZ_CUDA(cudaMemset(*p, 0, sizeof(T) * count));
    mc->allocs.push_back(*p);
    return AZ_OK;
}

extern "C" int az_mcts6_create(az_env6* env, az_nn* nn, int evaluator, int precision, az_mcts6** out)
{
    AZ_REQUIRE(env && out, "NULL argument");
    AZ_REQUIRE(evaluator >= M6_EVAL_NN && evaluator <= M6_EVAL_PSEUDO6, "unknown evaluator");
    AZ_REQUIRE(evaluator != M6_EVAL_NN || nn != nullptr, "evaluator AZ_EVAL_NN needs a network");
    AZ_REQUIRE(precision == AZ_NN_FP32 || precision == AZ_NN_BF16, "unknown precision");
    const az_rules* r = az_env6_rules(env);
    const int T = r->threads_per_mcts < 1 ? 1 : r->threads_per_mcts;
    const int sims = r->mcts_simulations - (r->mcts_simulations % T);
    AZ_REQUIRE(sims >= 1 && sims <= 60000, "mcts_simulations - mcts_simulations % threads_per_mcts must be in 1..60000");
    const int K = r->concurrent_descents < 1 ? 1 : r->concurrent_descents;
    AZ_REQUIRE(K <= 16, "concurrent_descents must be <= 16");
    AZ_REQUIRE(sims % K == 0, "the simulation count (mcts_simulations - mcts_simulations % threads_per_mcts) must be a multiple of concurrent_descents");
    AzDeviceGuard guard(az_env6_device(env));
    if (evaluator == M6_EVAL_NN && !nn->finalized) { int frc = az_nn_finalize(nn); if (frc) return frc; }
    az_mcts6* mc = new (std::nothrow) az_mcts6();
    AZ_REQUIRE(mc != nullptr, "out of host memory");
    mc->env = env; mc->nn = nn; mc->evaluator = evaluator; mc->precision = precision; mc->device = az_env6_device(env); mc->sims = sims;
    Mcts6Dev& d = mc->d;
    memset(&d, 0, sizeof d);
    d.n = az_env6_n(env); d.K = K;
    d.vo = evaluator == M6_EVAL_PSEUDO6 ? E6_PLAYERS : evaluator == M6_EVAL_NN ? nn->value_outputs : 1;
    d.cap = sims + 2;                                       // the table is cleared per search: the root + one node per simulation
    d.H = 64; while (d.H < 2 * d.cap) d.H <<= 1;
    d.dmax = 192;
    const size_t n = (size_t)d.n, ns = n * (size_t)K;     // ns = descent slots = the leaf batch of a simulation round
    int rc = 0;
    rc |= m6_alloc(mc, &d.nodes, n * d.cap * M6_NODE_WORDS, false);
    rc |= m6_alloc(mc, &d.index, n * d.H); rc |= m6_alloc(mc, &d.count, n);
    rc |= m6_alloc(mc, &d.path, ns * d.dmax); rc |= m6_alloc(mc, &d.path_len, ns);
    rc |= m6_alloc(mc, &d.leaf_state, ns * E6_WORDS); rc |= m6_alloc(mc, &d.leaf_valid, ns); rc |= m6_alloc(mc, &d.pending, ns);
    rc |= m6_alloc(mc, &d.term_value, ns); rc |= m6_alloc(mc, &d.term_seat, ns);
    rc |= m6_alloc(mc, &d.nn_policy, ns * AZ_MOVES); rc |= m6_alloc(mc, &d.nn_value, ns * (size_t)d.vo);
    rc |= m6_alloc(mc, &d.out_visits, n * AZ_MOVES); rc |= m6_alloc(mc, &d.out_pi, n * AZ_MOVES); rc |= m6_alloc(mc, &d.out_q, n * AZ_MOVES);
    rc |= m6_alloc(mc, &d.out_p, n * AZ_MOVES); rc |= m6_alloc(mc, &d.out_move, n); rc |= m6_alloc(mc, &d.out_status, n);
    rc |= m6_alloc(mc, &d.out_sumn, n); rc |= m6_alloc(mc, &d.out_table, n);
    rc |= m6_alloc(mc, &d.counters, (size_t)M6C_N);
    if (evaluator == M6_EVAL_NN) rc |= m6_alloc(mc, &mc->d_x, ns * 42 * (size_t)nn->input_planes);
    if (rc) { for (void* p : mc->allocs) cudaFree(p); delete mc; return AZ_ERR_CUDA; }
    d.root_state = az_env6_state_ptr(env);
    d.c1 = 1.0f - r->dir_noise_epsi; d.c2 = r->dir_noise_epsi * r->dir_noise_value; d.cpuct = r->cpuct;
    d.rules.allow_yield = r->allow_yield; d.rules.limit_reinforcement = r->limit_reinforcement; d.rules.limit_attack = r->limit_attack;
    d.rules.max_game_rounds = r->max_game_rounds; d.rules.min_unit_move = r->min_unit_move;
    d.eval_mode = evaluator; d.temp_threshold = r->temperature_threshold;
    *out = mc;
    return AZ_OK;
}

extern "C" int az_mcts6_destroy(az_mcts6* mc)
{
    if (!mc) return AZ_OK;
    AzDeviceGuard guard(mc->device);
    for (void* p : mc->allocs) cudaFree(p);
    delete mc;
    return AZ_OK;
}

// the leaves of the first k_used descent slots of every game (K for a simulation round, 1 for the root round: it uses slot 0 only)
static int m6_evaluate(az_mcts6* mc, cudaStream_t s, int k_used)
{
    if (mc->evaluator != M6_EVAL_NN) return AZ_OK;
    Mcts6Dev& d = mc->d;
    const int ns = d.K * d.n;                            // the stride of the SoA leaf state
    const bool seat_planes = mc->nn->input_planes == AZ_NN_IN_CH6;   // the leaves are encoded with the network's plane count
    if (mc->eval_count > 0 && mc->eval_count < d.n) {
        const int c = mc->eval_count, m = c * k_used;
        if (seat_planes) k_env6_encode_list<AZ_NN_IN_CH6><<<(m + 127) / 128, 128, 0, s>>>(d.leaf_state, ns, d.n, mc->eval_games, c, k_used, mc->d_x);
        else k_env6_encode_list<AZ_NN_IN_CH><<<(m + 127) / 128, 128, 0, s>>>(d.leaf_state, ns, d.n, mc->eval_games, c, k_used, mc->d_x);
        AZ_CUDA(cudaGetLastError());
        int rc = az_nn_forward_dev(mc->nn, mc->d_x, m, mc->eval_pol, mc->eval_val, mc->precision, s); if (rc) return rc;
        k_mcts6_scatter_evals<<<(m * (AZ_MOVES + d.vo) + 255) / 256, 256, 0, s>>>(mc->eval_pol, mc->eval_val, mc->eval_games, c, d.n, k_used,
                                                                                d.vo, d.nn_policy, d.nn_value);
        AZ_CUDA(cudaGetLastError());
        return AZ_OK;
    }
    const int m = d.n * k_used;                          // slots j * n + game: the first k_used * n of them
    if (seat_planes) k_env6_encode<AZ_NN_IN_CH6><<<(m + 127) / 128, 128, 0, s>>>(d.leaf_state, ns, m, mc->d_x);
    else k_env6_encode<AZ_NN_IN_CH><<<(m + 127) / 128, 128, 0, s>>>(d.leaf_state, ns, m, mc->d_x);
    AZ_CUDA(cudaGetLastError());
    return az_nn_forward_dev(mc->nn, mc->d_x, m, d.nn_policy, d.nn_value, mc->precision, s);
}

static int m6_search_once(az_mcts6* mc, int pick_mode, int apply_move, int auto_reset, cudaStream_t s)
{
    Mcts6Dev& d = mc->d;
    if (mc->evaluator == M6_EVAL_NN && !mc->nn->finalized) { int frc = az_nn_finalize(mc->nn); if (frc) return frc; }
    d.seed = az_env6_seed(mc->env); d.first_game = az_env6_first_game(mc->env);
    const int grid = (d.n + M6_WARPS - 1) / M6_WARPS;
    if (d.rec_out && mc->rec_generation != az_env6_generation(mc->env)) {    // games re-dealt or imported since: their staged samples go
        AZ_CUDA(cudaMemsetAsync(d.rec_len, 0, sizeof(uint32_t) * (size_t)d.n, s));
        mc->rec_generation = az_env6_generation(mc->env);
    }
    const uint64_t* tab = az_device_tables();
    k_mcts6_begin<<<grid, M6_WARPS * 32, 0, s>>>(d);
    k_mcts6_sim<<<grid, M6_WARPS * 32, 0, s>>>(d, tab, -1, 1);
    AZ_CUDA(cudaGetLastError());
    int rc = m6_evaluate(mc, s, 1); if (rc) return rc;
    for (int i = 0; i < mc->sims / d.K; ++i) {               // rounds of K descents per tree
        k_mcts6_sim<<<grid, M6_WARPS * 32, 0, s>>>(d, tab, i, 1);
        AZ_CUDA(cudaGetLastError());
        rc = m6_evaluate(mc, s, d.K); if (rc) return rc;
    }
    if (d.K > 1) k_mcts6_sim<<<grid, M6_WARPS * 32, 0, s>>>(d, tab, 0, 0);     // the last round's K completions; k_mcts6_finish does slot 0
    k_mcts6_finish<<<grid, M6_WARPS * 32, 0, s>>>(d, tab, pick_mode, apply_move, auto_reset);
    AZ_CUDA(cudaGetLastError());
    if (d.rec_out && apply_move) {
        k_mcts6_rec_end<<<grid, M6_WARPS * 32, 0, s>>>(d);
        AZ_CUDA(cudaGetLastError());
    }
    return AZ_OK;
}

extern "C" int az_mcts6_search(az_mcts6* mc, int pick_mode, int apply_move, uint32_t* h_visits, float* h_pi, uint8_t* h_move, int8_t* h_status,
                               void* stream)
{
    AZ_REQUIRE(mc != nullptr, "mcts is NULL");
    AZ_REQUIRE(pick_mode == 0 || pick_mode == 1, "pick_mode: 0 = argmax (play), 1 = self-play temperature rule");
    AzDeviceGuard guard(mc->device);
    cudaStream_t s = (cudaStream_t)stream;
    int rc = m6_search_once(mc, pick_mode, apply_move, 0, s); if (rc) return rc;
    const size_t n = (size_t)mc->d.n;
    if (h_visits) AZ_CUDA(cudaMemcpyAsync(h_visits, mc->d.out_visits, sizeof(uint32_t) * n * AZ_MOVES, cudaMemcpyDeviceToHost, s));
    if (h_pi) AZ_CUDA(cudaMemcpyAsync(h_pi, mc->d.out_pi, sizeof(float) * n * AZ_MOVES, cudaMemcpyDeviceToHost, s));
    if (h_move) AZ_CUDA(cudaMemcpyAsync(h_move, mc->d.out_move, n, cudaMemcpyDeviceToHost, s));
    if (h_status) AZ_CUDA(cudaMemcpyAsync(h_status, mc->d.out_status, n, cudaMemcpyDeviceToHost, s));
    AZ_CUDA(cudaStreamSynchronize(s));
    return AZ_OK;
}

extern "C" int az_mcts6_root_stats(az_mcts6* mc, float* h_q, float* h_p, uint32_t* h_sumn, int32_t* h_table, void* stream)
{
    AZ_REQUIRE(mc != nullptr, "mcts is NULL");
    AzDeviceGuard guard(mc->device);
    cudaStream_t s = (cudaStream_t)stream;
    const size_t n = (size_t)mc->d.n;
    if (h_q) AZ_CUDA(cudaMemcpyAsync(h_q, mc->d.out_q, sizeof(float) * n * AZ_MOVES, cudaMemcpyDeviceToHost, s));
    if (h_p) AZ_CUDA(cudaMemcpyAsync(h_p, mc->d.out_p, sizeof(float) * n * AZ_MOVES, cudaMemcpyDeviceToHost, s));
    if (h_sumn) AZ_CUDA(cudaMemcpyAsync(h_sumn, mc->d.out_sumn, sizeof(uint32_t) * n, cudaMemcpyDeviceToHost, s));
    if (h_table) AZ_CUDA(cudaMemcpyAsync(h_table, mc->d.out_table, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, s));
    AZ_CUDA(cudaStreamSynchronize(s));
    return AZ_OK;
}

// n_moves self-play moves of every game with no host synchronisation; finished games are re-dealt in place
extern "C" int az_selfplay6_run(az_mcts6* mc, int n_moves, void* stream)
{
    AZ_REQUIRE(mc != nullptr, "mcts is NULL");
    AZ_REQUIRE(n_moves >= 0, "n_moves must be >= 0");
    AzDeviceGuard guard(mc->device);
    for (int i = 0; i < n_moves; ++i) { int rc = m6_search_once(mc, 1, 1, 1, (cudaStream_t)stream); if (rc) return rc; }
    return AZ_OK;
}

// ---- six-player training samples (az_samples6.cuh)
extern "C" int az_selfplay6_record(az_mcts6* mc, size_t capacity_samples, int max_moves_per_game)
{
    AZ_REQUIRE(mc != nullptr, "mcts is NULL");
    AZ_REQUIRE(capacity_samples > 0 && max_moves_per_game > 0, "capacity_samples and max_moves_per_game must be positive");
    AZ_REQUIRE(mc->d.rec_out == nullptr, "recording is already enabled on this handle");
    AzDeviceGuard guard(mc->device);
    Mcts6Dev& d = mc->d;
    const size_t n = (size_t)d.n;
    int rc = 0;
    rc |= m6_alloc(mc, &d.rec_state, n * (size_t)max_moves_per_game * S6_IMG_WORDS, false);
    rc |= m6_alloc(mc, &d.rec_pi, n * (size_t)max_moves_per_game * AZ_MOVES, false);
    rc |= m6_alloc(mc, &d.rec_len, n);
    rc |= m6_alloc(mc, &d.rec_end, n, false);
    rc |= m6_alloc(mc, &d.rec_count, (size_t)2);
    uint8_t* out = nullptr;
    rc |= m6_alloc(mc, &out, capacity_samples * (size_t)S6_BYTES, false);
    if (rc) { d.rec_out = nullptr; return AZ_ERR_CUDA; }
    AZ_CUDA(cudaMemset(d.rec_end, 0xff, n));           // AZ_STATUS_RUNNING: no game has ended
    d.rec_moves = max_moves_per_game; d.rec_cap = capacity_samples;
    mc->rec_generation = az_env6_generation(mc->env);
    d.rec_out = out;                                   // set last: the kernels record iff rec_out != NULL
    return AZ_OK;
}

extern "C" int az_selfplay6_samples(az_mcts6* mc, uint8_t* h_records, size_t max_records, size_t* n_out, uint64_t* h_dropped, void* stream)
{
    AZ_REQUIRE(mc && n_out, "NULL argument");
    AZ_REQUIRE(mc->d.rec_out != nullptr, "az_selfplay6_record has not been called");
    AzDeviceGuard guard(mc->device);
    cudaStream_t s = (cudaStream_t)stream;
    unsigned long long h[2];
    AZ_CUDA(cudaMemcpyAsync(h, mc->d.rec_count, sizeof h, cudaMemcpyDeviceToHost, s));
    AZ_CUDA(cudaStreamSynchronize(s));
    AZ_REQUIRE(h[0] <= mc->d.rec_cap, "sample queue corrupted: committed count exceeds the capacity");
    const size_t have = (size_t)h[0];                  // committed records: az_rec_reserve never reserves past the capacity
    if (h_dropped) *h_dropped = h[1];
    *n_out = have;
    if (!h_records && have) return AZ_OK;              // size query; with an empty queue the call drains (resets the dropped count)
    AZ_REQUIRE(max_records >= have, "h_records is too small: query the size with h_records = NULL first");
    if (have) AZ_CUDA(cudaMemcpyAsync(h_records, mc->d.rec_out, have * (size_t)S6_BYTES, cudaMemcpyDeviceToHost, s));
    AZ_CUDA(cudaMemsetAsync(mc->d.rec_count, 0, sizeof h, s));
    AZ_CUDA(cudaStreamSynchronize(s));
    return AZ_OK;
}

extern "C" int az_mcts6_counters(az_mcts6* mc, az_counters6* h_out, uint64_t* h_sims, uint64_t* h_evals, uint64_t* h_errors, int reset, void* stream)
{
    AZ_REQUIRE(mc && h_out, "NULL argument");
    AzDeviceGuard guard(mc->device);
    cudaStream_t s = (cudaStream_t)stream;
    unsigned long long h[M6C_N];
    AZ_CUDA(cudaMemcpyAsync(h, mc->d.counters, sizeof h, cudaMemcpyDeviceToHost, s));
    if (reset) AZ_CUDA(cudaMemsetAsync(mc->d.counters, 0, sizeof h, s));
    AZ_CUDA(cudaStreamSynchronize(s));
    h_out->steps = h[M6C_STEPS]; h_out->games = h[M6C_GAMES]; h_out->draws = h[M6C_DRAWS];
    for (int p = 0; p < E6_PLAYERS; ++p) h_out->wins[p] = h[M6C_WIN0 + p];
    if (h_sims) *h_sims = h[M6C_SIMS];
    if (h_evals) *h_evals = h[M6C_EVALS];
    if (h_errors) *h_errors = h[M6C_OVERFLOW];
    return AZ_OK;
}

extern "C" int az_env6_encode_planes(az_env6* e, int input_planes, float* h_x, void* stream)
{
    AZ_REQUIRE(e && h_x, "NULL argument");
    AZ_REQUIRE(input_planes == AZ_NN_IN_CH || input_planes == AZ_NN_IN_CH6, "input_planes must be 13 or 16");
    AzDeviceGuard guard(az_env6_device(e));
    cudaStream_t s = (cudaStream_t)stream;
    const int n = az_env6_n(e);
    const size_t floats = (size_t)n * 42 * input_planes;
    float* d_x = nullptr;
    AZ_CUDA(cudaMalloc(&d_x, sizeof(float) * floats));
    if (input_planes == AZ_NN_IN_CH6) k_env6_encode<AZ_NN_IN_CH6><<<(n + 127) / 128, 128, 0, s>>>(az_env6_state_ptr(e), n, n, d_x);
    else k_env6_encode<AZ_NN_IN_CH><<<(n + 127) / 128, 128, 0, s>>>(az_env6_state_ptr(e), n, n, d_x);
    cudaError_t ce = cudaGetLastError();
    if (ce == cudaSuccess) ce = cudaMemcpyAsync(h_x, d_x, sizeof(float) * floats, cudaMemcpyDeviceToHost, s);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(s);
    cudaFree(d_x);
    if (ce != cudaSuccess) { az_set_error("az_env6_encode: %s", cudaGetErrorString(ce)); return AZ_ERR_CUDA; }
    return AZ_OK;
}
extern "C" int az_env6_encode(az_env6* e, float* h_x, void* stream) { return az_env6_encode_planes(e, AZ_NN_IN_CH, h_x, stream); }

// ---------------------------------------------------------------- six-player arena (SIXPLAYER.md §4)
// k_arena6_advance (az_env6.cu) tallies, deals and plays the random and scripted agents' plies; each tick then runs one search per searcher
// restricted to the slots waiting for it (Mcts6Dev::sel over to_move), with the slots' match game ids as the search's game ids, and
// its leaf batches compacted to those slots.  A searcher's move can hand the turn to another agent: that slot waits for the next tick.
struct az_arena6 {
    az_env6* env = nullptr;
    az_mcts6* agent[E6_PLAYERS] = {};    // NULL = the uniform-random player or the scripted agent (Arena6Dev::script)
    int n_agents = 0;
    Arena6Dev a;
    int32_t* d_list = nullptr;           // slots waiting for the searcher of this search (leaf-batch compaction)
    float* d_pol_c = nullptr; float* d_val_c = nullptr;   // compacted network outputs [K*n][43], [K*n][vo] (K = the searchers' descents per tree)
    int8_t* d_status = nullptr; uint32_t* d_plies = nullptr; uint64_t games_cap = 0;   // per match game
    std::vector<uint32_t> active;        // active slots of every tick of the last match
    std::vector<void*> allocs;
};

int az_launch_arena_list(const uint8_t* flags, int n, int want, int32_t* out, cudaStream_t s)
{
    k_arena_list<<<1, 1024, 0, s>>>(flags, n, want, out);
    AZ_CUDA(cudaGetLastError());
    return AZ_OK;
}

template <class T> static int a6_alloc(az_arena6* ar, T** p, size_t count)
{
    AZ_CUDA(cudaMalloc(p, sizeof(T) * count));
    AZ_CUDA(cudaMemset(*p, 0, sizeof(T) * count));
    ar->allocs.push_back(*p);
    return AZ_OK;
}

extern "C" int az_arena6_create_agents(az_env6* env, az_mcts6* const* agents, const int* kinds, int n_agents, const uint8_t* seat_agent,
                                       int rotate_seats, az_arena6** out)
{
    AZ_REQUIRE(env && agents && kinds && seat_agent && out, "NULL argument");
    AZ_REQUIRE(n_agents >= 1 && n_agents <= E6_PLAYERS, "n_agents must be in 1..6");
    for (int i = 0; i < n_agents; ++i) {
        AZ_REQUIRE(kinds[i] == AZ_AGENT6_SEARCHER || kinds[i] == AZ_AGENT6_RANDOM || kinds[i] == AZ_AGENT6_SCRIPT,
                   "unknown agent kind (AZ_AGENT6_SEARCHER, AZ_AGENT6_RANDOM or AZ_AGENT6_SCRIPT)");
        AZ_REQUIRE((kinds[i] == AZ_AGENT6_SEARCHER) == (agents[i] != nullptr),
                   "agents[i] must be an az_mcts6 handle for a searcher and NULL for the random or scripted agent");
    }
    for (int i = 0; i < n_agents; ++i) {
        if (!agents[i]) continue;
        AZ_REQUIRE(agents[i]->env == env, "every searcher must be built over the arena's env (the agents share its game states)");
        for (int j = 0; j < i; ++j) AZ_REQUIRE(agents[j] != agents[i], "the same az_mcts6 handle appears twice (each agent owns its tables)");
    }
    unsigned held = 0;
    for (int s = 0; s < E6_PLAYERS; ++s) {
        AZ_REQUIRE(seat_agent[s] < n_agents, "seat_agent entry out of range (must be < n_agents)");
        held |= 1u << seat_agent[s];
    }
    AZ_REQUIRE(held == (1u << n_agents) - 1u, "every agent must hold at least one seat");
    AzDeviceGuard guard(az_env6_device(env));
    az_arena6* ar = new (std::nothrow) az_arena6();
    AZ_REQUIRE(ar != nullptr, "out of host memory");
    ar->env = env; ar->n_agents = n_agents;
    Arena6Dev& a = ar->a;
    memset(&a, 0, sizeof a);
    a.n = az_env6_n(env); a.state = az_env6_state_ptr(env); a.rotate = rotate_seats ? 1 : 0;
    for (int s = 0; s < E6_PLAYERS; ++s) a.seat_agent |= (uint32_t)seat_agent[s] << (4 * s);
    for (int i = 0; i < n_agents; ++i) {
        ar->agent[i] = agents[i];
        if (kinds[i] == AZ_AGENT6_SEARCHER) a.searcher |= (uint8_t)(1u << i);
        if (kinds[i] == AZ_AGENT6_SCRIPT) a.script |= (uint8_t)(1u << i);
    }
    const size_t n = (size_t)a.n;
    size_t ns = n, nv = n;                                              // the largest compacted leaf batch: K * n, and its values K * n * vo
    for (int i = 0; i < n_agents; ++i) if (agents[i]) {
        ns = std::max(ns, n * (size_t)agents[i]->d.K);
        nv = std::max(nv, n * (size_t)agents[i]->d.K * (size_t)agents[i]->d.vo);
    }
    int rc = 0;
    rc |= a6_alloc(ar, &a.slot, n); rc |= a6_alloc(ar, &a.slot_game, n); rc |= a6_alloc(ar, &a.to_move, n);
    rc |= a6_alloc(ar, &a.res, (size_t)A6_N); rc |= a6_alloc(ar, &ar->d_list, n);
    rc |= a6_alloc(ar, &ar->d_pol_c, ns * AZ_MOVES); rc |= a6_alloc(ar, &ar->d_val_c, nv);
    if (rc) { for (void* p : ar->allocs) cudaFree(p); delete ar; return AZ_ERR_CUDA; }
    *out = ar;
    return AZ_OK;
}

extern "C" int az_arena6_create(az_env6* env, az_mcts6* const* agents, int n_agents, const uint8_t* seat_agent, int rotate_seats, az_arena6** out)
{
    AZ_REQUIRE(agents != nullptr, "NULL argument");
    AZ_REQUIRE(n_agents >= 1 && n_agents <= E6_PLAYERS, "n_agents must be in 1..6");
    int kinds[E6_PLAYERS];
    for (int i = 0; i < n_agents; ++i) kinds[i] = agents[i] ? AZ_AGENT6_SEARCHER : AZ_AGENT6_RANDOM;
    return az_arena6_create_agents(env, agents, kinds, n_agents, seat_agent, rotate_seats, out);
}

extern "C" int az_arena6_destroy(az_arena6* ar)
{
    if (!ar) return AZ_OK;
    AzDeviceGuard guard(az_env6_device(ar->env));
    for (void* p : ar->allocs) cudaFree(p);
    cudaFree(ar->d_status); cudaFree(ar->d_plies);
    delete ar;
    return AZ_OK;
}

extern "C" int az_arena6_play(az_arena6* ar, uint64_t first_game, uint64_t n_games, uint64_t seed, az_arena6_results* h_out,
                              int8_t* h_status, uint32_t* h_plies, void* stream)
{
    AZ_REQUIRE(ar && h_out, "NULL argument");
    Arena6Dev& a = ar->a;
    for (int i = 0; i < ar->n_agents; ++i)
        AZ_REQUIRE(!ar->agent[i] || !ar->agent[i]->d.rec_out, "a searcher with sample recording enabled cannot play in an arena");
    AZ_REQUIRE(!a.rotate || (first_game % E6_PLAYERS == 0 && n_games % E6_PLAYERS == 0),
               "with rotate_seats, first_game and n_games must be multiples of 6 (whole rotation groups)");
    AZ_REQUIRE(first_game <= (1ull << 32) && n_games <= (1ull << 32) - first_game, "first_game + n_games must not exceed 2^32 (32-bit game ids)");
    AzDeviceGuard guard(az_env6_device(ar->env));
    cudaStream_t s = (cudaStream_t)stream;
    if (n_games > ar->games_cap) {
        cudaFree(ar->d_status); cudaFree(ar->d_plies);
        ar->d_status = nullptr; ar->d_plies = nullptr; ar->games_cap = 0;
        AZ_CUDA(cudaMalloc(&ar->d_status, n_games));
        AZ_CUDA(cudaMalloc(&ar->d_plies, sizeof(uint32_t) * n_games));
        ar->games_cap = n_games;
    }
    int rc = az_env6_reset(ar->env, seed, stream); if (rc) return rc;
    a.seed = seed; a.first_game = (uint32_t)first_game; a.n_games = n_games; a.out_status = ar->d_status; a.out_plies = ar->d_plies;
    const size_t n = (size_t)a.n;
    AZ_CUDA(cudaMemsetAsync(a.slot, A6_FREE, n, s));
    AZ_CUDA(cudaMemsetAsync(a.res, 0, sizeof(unsigned long long) * A6_N, s));
    for (int i = 0; i < ar->n_agents; ++i)
        if (ar->agent[i]) AZ_CUDA(cudaMemsetAsync(ar->agent[i]->d.counters, 0, sizeof(unsigned long long) * M6C_N, s));
    const az_rules* rules = az_env6_rules(ar->env);
    unsigned long long cnt[1 + E6_PLAYERS];                              // A6_ACTIVE, A6_WAIT0 ..
    ar->active.clear();
    for (;;) {
        AZ_CUDA(cudaMemsetAsync(a.res + A6_ACTIVE, 0, sizeof cnt, s));
        rc = az_launch_arena6_advance(a, rules, s); if (rc) return rc;
        AZ_CUDA(cudaMemcpyAsync(cnt, a.res + A6_ACTIVE, sizeof cnt, cudaMemcpyDeviceToHost, s));
        AZ_CUDA(cudaStreamSynchronize(s));
        if (cnt[0] == 0) break;
        ar->active.push_back((uint32_t)cnt[0]);
        for (int i = 0; i < ar->n_agents; ++i) {
            az_mcts6* mc = ar->agent[i];
            if (!mc || !cnt[1 + i]) continue;
            if (mc->evaluator == M6_EVAL_NN && cnt[1 + i] < (unsigned long long)a.n) {
                rc = az_launch_arena_list(a.to_move, a.n, i, ar->d_list, s); if (rc) return rc;
                mc->eval_games = ar->d_list; mc->eval_count = (int)cnt[1 + i]; mc->eval_pol = ar->d_pol_c; mc->eval_val = ar->d_val_c;
            }
            mc->d.sel = a.to_move; mc->d.sel_value = i; mc->d.game_id = a.slot_game;
            rc = m6_search_once(mc, 0, 1, 0, s);                            // argmax, the move applied, no re-deal
            mc->d.sel = nullptr; mc->d.sel_value = 0; mc->d.game_id = nullptr;
            mc->eval_games = nullptr; mc->eval_count = 0; mc->eval_pol = nullptr; mc->eval_val = nullptr;
            if (rc) return rc;
        }
    }
    unsigned long long r[A6_N], c[E6_PLAYERS][M6C_N];
    memset(c, 0, sizeof c);
    AZ_CUDA(cudaMemcpyAsync(r, a.res, sizeof r, cudaMemcpyDeviceToHost, s));
    for (int i = 0; i < ar->n_agents; ++i)
        if (ar->agent[i]) AZ_CUDA(cudaMemcpyAsync(c[i], ar->agent[i]->d.counters, sizeof c[i], cudaMemcpyDeviceToHost, s));
    if (h_status && n_games) AZ_CUDA(cudaMemcpyAsync(h_status, ar->d_status, n_games, cudaMemcpyDeviceToHost, s));
    if (h_plies && n_games) AZ_CUDA(cudaMemcpyAsync(h_plies, ar->d_plies, sizeof(uint32_t) * n_games, cudaMemcpyDeviceToHost, s));
    AZ_CUDA(cudaStreamSynchronize(s));
    memset(h_out, 0, sizeof *h_out);
    h_out->count = r[A6_COUNT]; h_out->draw = r[A6_DRAW];
    for (int p = 0; p < E6_PLAYERS; ++p) {
        h_out->win[p] = r[A6_WIN0 + p]; h_out->win_seat[p] = r[A6_WIN_SEAT0 + p];
        h_out->moves[p] = ar->agent[p] ? c[p][M6C_STEPS] : r[A6_MOVES0 + p];
        h_out->sims += c[p][M6C_SIMS]; h_out->evals += c[p][M6C_EVALS]; h_out->errors += c[p][M6C_OVERFLOW];
    }
    h_out->ticks = ar->active.size();
    return AZ_OK;
}

extern "C" int az_arena6_active_slots(az_arena6* ar, uint32_t* h_active, size_t max_ticks, size_t* n_out)
{
    AZ_REQUIRE(ar && n_out, "NULL argument");
    *n_out = ar->active.size();
    if (!h_active) return AZ_OK;
    AZ_REQUIRE(max_ticks >= ar->active.size(), "h_active is too small: query the size with h_active = NULL first");
    if (!ar->active.empty()) memcpy(h_active, ar->active.data(), sizeof(uint32_t) * ar->active.size());
    return AZ_OK;
}
