/*
 * TEST INFRASTRUCTURE — risk6_planes.c: the six-player seat planes (SIXPLAYER.md §2, "seat planes"), the checker of the 16-plane
 * encoding of az_env6_encode_planes, of the six-player search's leaf batches and of az_nn_train6 over a network with 16 input planes.
 * Tensor [7][6][16], cell (y, x) = land y*6 + x:
 *   planes 0..5    army / 32 on the lands of seat (cur + k) % 6, k = 0..5 (fixed seat order, eliminated seats included: an all-zero plane)
 *   planes 6..15   planes 3..12 of r6_encode: own / (own + all opponents') armies, own / (own + living opponents') reinforcement values,
 *                  min(attacks / 8, 1), may-draw-a-card, the phase one-hot (SETUP_NEUTRAL never set)
 * Stated here on its own (not through r6_encode) so that the tests can hold the two encodings against each other.  It builds on
 * risk6_oracle.c unchanged (included here); built as its own library by oracle/planes6.py, never linked into the product.
 */
#include "risk6_oracle.c"

#define R6_INPUT16_FLOATS 672
const int r6_input16_floats = R6_INPUT16_FLOATS;

void r6_encode16(const r6_state* s, float x[R6_INPUT16_FLOATS])
{
    derived6 d; derive(s, &d);
    const int c = s->cur;
    int own_total = 0, other_total = 0;
    for (int i = 0; i < RO_LANDS; ++i) { if (s->owner[i] == c) own_total += s->army[i]; else other_total += s->army[i]; }
    float ref = (float)ro_reinforcement_value(d.owned[c]), oref = 0.0f;
    for (int p = 0; p < R6_PLAYERS; ++p) if (p != c && d.owned[p]) oref += (float)ro_reinforcement_value(d.owned[p]);
    const float army_share = (float)own_total / ((float)own_total + (float)other_total);
    const float reinf_share = ref / (ref + oref);
    float att = (float)s->attacks / 8.0f; if (att > 1.0f) att = 1.0f;
    for (int i = 0; i < RO_LANDS; ++i) {
        float* f = x + i * 16;
        const float a = (float)s->army[i] / 32.0f;
        for (int k = 0; k < R6_PLAYERS; ++k) f[k] = s->owner[i] == (c + k) % R6_PLAYERS ? a : 0.0f;
        f[6] = army_share; f[7] = reinf_share; f[8] = att; f[9] = s->allow_draw ? 1.0f : 0.0f;
        for (int k = 0; k < 6; ++k) f[10 + k] = s->phase == k ? 1.0f : 0.0f;
    }
}
