// az_mcts_value6.cu — the translation unit of the two-player search: az_mcts.cu itself (included byte for byte: the ncu capture of
// k_mcts_sim in profiles/traffic.json is keyed by that file's hash) with az_mcts_create wrapped so that it rejects a network with six
// value outputs or 16 input planes (SIXPLAYER.md §2).  The two-player search backs up one value per leaf and reads value [n] from the
// forward, and it encodes its leaves with the 13 two-player planes.
#include "az_b200.h"

#define az_mcts_create az_mcts_create_one_value
#include "az_mcts.cu"
#undef az_mcts_create

extern "C" int az_mcts_create(az_env* env, az_nn* nn, int evaluator, int precision, az_mcts** out)
{
    AZ_REQUIRE(evaluator != EVAL_NN || nn == nullptr || nn->value_outputs == 1,
               "az_mcts_create: the two-player search backs up one value; this network has six value outputs");
    AZ_REQUIRE(evaluator != EVAL_NN || nn == nullptr || nn->input_planes == AZ_NN_IN_CH,
               "az_mcts_create: the two-player search encodes 13 input planes; this network has 16 (the six-player seat planes)");
    return az_mcts_create_one_value(env, nn, evaluator, precision, out);
}
