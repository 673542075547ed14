// az_samples6.cuh — the six-player training-sample record (include/az_b200.h AZ_SAMPLE6_BYTES), shared by the recorder of the
// six-player search (az_mcts6.cu), the recorder of generated games (az_env6.cu) and the training unpack (az_nn_train.cu).  A format of this project: every field is 4-byte aligned,
// so both sides move whole 32-bit words.
//   bytes 0..107    the position before the move as its 108-byte image (k_env6_export's layout; seat to move = byte 98)
//   bytes 108..111  float value target of the seat to move there
//   bytes 112..283  float policy target[43]
//   byte  284       int8 final status of the game (winner seat 0..5 or AZ_STATUS_DRAW), bytes 285..287 zero
#pragma once

#include "az_game6.cuh"
#include "az_samples.cuh"

#define S6_BYTES AZ_SAMPLE6_BYTES
#define S6_WORDS (AZ_SAMPLE6_BYTES / 4)
#define S6_IMG_WORDS (E6_IMG / 4)       // 27
#define S6_VALUE 108
#define S6_PI 112
#define S6_STATUS 284
#define S6_CUR 98                       // image byte of the seat to move
#define S6_PHASE 101
#define S6_ALLOW_DRAW 104
#define S6_ATTACKS 105

// value target of a sample whose seat to move is `seat` in a game that ended with `status`: the six-seat rule the search backs up
// (m6_backup: +v for the winner's nodes, -v / 5 for every other seat, 0 for everyone after a draw) with v = 1
__device__ __forceinline__ float s6_value(int status, uint32_t seat)
{
    return status == AZ_STATUS_DRAW ? 0.0f : ((uint32_t)status == seat ? 1.0f : __fdiv_rn(-1.0f, 5.0f));
}

// byte b (0..107) of the 108-byte image of a game held as the device state words 0..26 (az_game6.cuh)
__device__ __forceinline__ uint32_t s6_image_byte(const uint32_t* __restrict__ st, int b)
{
    if (b < AZ_LANDS) return (st[b >> 2] >> (8 * (b & 3))) & 0xffu;                                      // army
    if (b < 2 * AZ_LANDS) { b -= AZ_LANDS; return (st[11 + (b >> 2)] >> (8 * (b & 3))) & 0xffu; }     // owner
    if (b < 90) { const int p = b - 84; return p < 4 ? (st[22] >> (8 * p)) & 0xffu : (st[23] >> (8 * (p - 4))) & 0xffu; }   // cards
    if (b < 96) return (st[26] >> (4 * (b - 90))) & 0xfu;                                                // set-up pools
    switch (b) {
    case 96: return st[24] & 0xffu;             // round (u16)
    case 97: return (st[24] >> 8) & 0xffu;
    case 98: return (st[24] >> 16) & 0xffu;     // cur
    case 99: return st[24] >> 24;               // card_sets
    case 100: return st[25] & 0xffu;            // reinf
    case 101: return (st[25] >> 8) & 0xffu;     // phase
    case 102: return (st[25] >> 16) & 0xffu;    // mob_from
    case 103: return st[25] >> 24;              // mob_to
    case 104: return (st[23] >> 16) & 0xffu;    // allow_draw
    case 105: return st[23] >> 24;              // attacks
    default: return 0u;                         // 2 pad bytes
    }
}

// word k (0..71) of the record of the sample staged as state words st[0..26] and policy pi[43], for a game that ended with `status`
__device__ __forceinline__ uint32_t s6_record_word(const uint32_t* __restrict__ st, const float* __restrict__ pi, int status, int k)
{
    if (k < S6_IMG_WORDS) {
        const int b = 4 * k;
        return s6_image_byte(st, b) | (s6_image_byte(st, b + 1) << 8) | (s6_image_byte(st, b + 2) << 16) | (s6_image_byte(st, b + 3) << 24);
    }
    if (k == S6_VALUE / 4) return __float_as_uint(s6_value(status, (st[24] >> 16) & 0xffu));
    if (k < S6_STATUS / 4) return __float_as_uint(pi[k - S6_PI / 4]);
    return (uint32_t)(uint8_t)(int8_t)status;
}

// the same word for a sample whose policy target is one-hot at the played `action` (the generated games of az_env6_play)
__device__ __forceinline__ uint32_t s6_onehot_record_word(const uint32_t* __restrict__ st, int action, int status, int k)
{
    if (k >= S6_PI / 4 && k < S6_STATUS / 4) return k - S6_PI / 4 == action ? __float_as_uint(1.0f) : 0u;
    return s6_record_word(st, nullptr, status, k);
}
