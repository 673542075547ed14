// az_arena.cuh — device-side bookkeeping of the -m play arena, shared by az_env.cu (k_arena_advance) and az_mcts.cu (host loop)
#pragma once

#include <stdint.h>
#include <cuda_runtime.h>

#include "az_b200.h"

enum { ARENA_COUNT = 0, ARENA_DRAW = 1, ARENA_WIN0 = 2, ARENA_WIN1 = 3, ARENA_WAS0 = 4, ARENA_WAS1 = 5, ARENA_OPP_TURNS = 6,
       ARENA_CLAIMED = 7, ARENA_ACTIVE = 8, ARENA_TOMOVE0 = 9, ARENA_TOMOVE1 = 10, ARENA_N = 12 };

struct ArenaDev {
    int n;
    uint32_t first_game;
    uint64_t seed;
    uint32_t* state;            // env SoA [16][n]
    uint32_t* start_state;      // [16][n]  Game::previousStartState (game/game.h)
    uint32_t* script;           // [n][2]   packed ScriptPlayer members per side
    uint8_t* player_start;      // [n]      Game::playerStart
    uint8_t* fresh;             // [n]      slot has not started a game yet
    uint8_t* active;            // [n]      slot still plays
    uint8_t* last_mover;        // [n]      side that moved last in the running game (0xff = nobody yet)
    uint8_t* extra_trim;        // [n]      the MCTS handle's pending trimNodes counter
    uint8_t* extra_trim_opp;    // [n]      the same for the second searcher (AZ_OPPONENT_ALPHAZERO), else NULL
    uint8_t* ended;             // [n]      game that ended in this advance call: 0 none, 1 / 2 = winner 0 / 1, 3 = draw (sample flush)
    uint8_t* to_move;           // [n]      side whose searcher moves next in this slot (AZ_OPPONENT_ALPHAZERO; 0xff = slot is done)
    unsigned long long* res;    // [ARENA_N]
    unsigned long long total_games;
    int opponent, mirror;
};

int az_launch_arena_advance(const ArenaDev& a, const az_rules* rules, cudaStream_t s);   // az_env.cu
// ascending list of the slots with flags[slot] == want: the leaf-batch compaction of both arenas.  The kernel is defined in az_mcts.cu;
// az_launch_arena_list (az_mcts6.cu) launches it for the six-player arena.
__global__ void k_arena_list(const uint8_t* __restrict__ flags, int n, int want, int32_t* __restrict__ out);
int az_launch_arena_list(const uint8_t* flags, int n, int want, int32_t* out, cudaStream_t s);

// ---------------------------------------------------------------- six-player arena (az_arena6_*, SIXPLAYER.md §4)
// shared by az_env6.cu (k_arena6_advance) and az_mcts6.cu (host loop)
enum { A6_COUNT = 0, A6_DRAW = 1, A6_WIN0 = 2, A6_WIN_SEAT0 = 8, A6_MOVES0 = 14, A6_CLAIMED = 20, A6_ACTIVE = 21, A6_WAIT0 = 22, A6_N = 28 };
enum { A6_FREE = 0, A6_PLAYING = 1, A6_DONE = 2 };

struct Arena6Dev {
    int n;                      // slots of the env
    uint32_t first_game;        // match game ids first_game .. first_game + n_games - 1
    uint64_t n_games, seed;
    uint32_t* state;            // env6 SoA [28][n]
    uint8_t* slot;              // [n]  A6_FREE (claims a game next), A6_PLAYING, A6_DONE (no game left)
    uint32_t* slot_game;        // [n]  match game id of the slot's game
    uint8_t* to_move;           // [n]  agent whose searcher moves next in this slot (0xff = none this tick)
    int8_t* out_status;         // [n_games]  per match game: winner seat or AZ_STATUS_DRAW
    uint32_t* out_plies;        // [n_games]  and its plies
    unsigned long long* res;    // [A6_N]
    uint32_t seat_agent;        // agent index of seat s in bits 4s .. 4s + 3
    uint8_t searcher;           // bit a: agent a is a searcher
    uint8_t script;             // bit a: agent a is the scripted agent (SIXPLAYER.md §5); neither bit: the uniform-random player
    uint8_t rotate;
};

int az_launch_arena6_advance(const Arena6Dev& a, const az_rules* rules, cudaStream_t s);   // az_env6.cu
