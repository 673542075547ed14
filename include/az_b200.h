/*
 * az_b200.h — C ABI of libaz_b200.so, the B200 (sm_100a) implementation of
 * JGasp/alphazero-risk's self-play hot path.
 *
 * The reference has no FFI: its plugin seams are C++ classes (SURVEY.md §8b).  Each entry
 * point below names the reference interface it replaces (paths relative to
 * /root/reference/src/risk_game); the C++ adapters that present those interfaces on top of
 * this ABI live in alphazero_risk_b200/host/, the binding a reference maintainer would add
 * is shown in INTEGRATION.md.
 *
 * Conventions: every call returns AZ_OK (0) or a negative az_error; the message of the last
 * failure on the calling thread is az_last_error().  No exception crosses the boundary: where
 * the reference throws for one game (illegal action, move on a finished game) the per-game
 * status byte carries the code and the game's state is left untouched.  Handles are opaque,
 * the library owns all device memory, the caller owns host buffers.  `stream` is a
 * cudaStream_t passed as void* (NULL = the legacy default stream).  Calls on different
 * handles are thread-safe; calls on one handle must be serialised by the caller.
 * Pointers named h_* are HOST buffers (copied inside the call), d_* are DEVICE buffers.
 */
#ifndef AZ_B200_H
#define AZ_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define AZ_API __attribute__((visibility("default")))
#else
#define AZ_API
#endif

#define AZ_LANDS 42
#define AZ_MOVES 43            /* 42 lands + skip; ALL_MOVES, player/alpha_zero/alphazero_mcts.h:13 */
#define AZ_SKIP 42             /* Land::SKIP_MOVE, land/land.cpp:312 */
#define AZ_NONE 43             /* LandIndex::None */
#define AZ_DATA_BYTES 160      /* sizeof(Data), state/state.h:86-105 */
#define AZ_INPUT_FLOATS 546    /* [7][6][13], neural_network/alphazero_nn_data.h:66 (INPUT_VECTOR_TYPE_2) */
#define AZ_INPUT6_FLOATS 672   /* [7][6][16]: the six-player seat planes (SIXPLAYER.md §2, az_nn_create_planes) */
#define AZ_STATE_WORDS 16      /* device SoA: 32-bit words per game (see DESIGN.md) */

typedef enum az_error {
    AZ_OK = 0,
    AZ_ERR_INVALID_ARG = -1,
    AZ_ERR_CUDA = -2,
    AZ_ERR_NO_DEVICE = -3,
    AZ_ERR_BAD_STATE = -4,     /* az_env_import_aos: masks / totals disagree with landArmy[] */
    AZ_ERR_CAPACITY = -5,      /* MCTS node pool exhausted */
    AZ_ERR_NOT_READY = -6
} az_error;

/* per-game status byte written by the step calls */
#define AZ_STATUS_RUNNING (-1) /* State::NOT_ENDED, state/state.h:124 */
#define AZ_STATUS_DRAW (-2)    /* State::DRAW, state/state.h:123; 0 / 1 = winner */
#define AZ_STATUS_ILLEGAL (-3) /* action not in the legal-move mask (reference: std::invalid_argument / logic_error) */
#define AZ_STATUS_OVER (-4)    /* game had already ended before the step */

/* runtime options of /root/reference/src/settings.h:40-62 that change the path's results;
   field names follow SETTINGS.* */
typedef struct az_rules {
    int32_t allow_yield;             /* ALLOW_YIELD               --allow-yield           default 1 */
    int32_t limit_reinforcement;     /* LIMIT_REINFORCEMENT_MOVES --limit-reinforcement   default 1 */
    int32_t limit_attack;            /* LIMIT_ATTACK_MOVES        --limit-attack          default 0 */
    int32_t max_game_rounds;         /* MAX_GAME_ROUNDS                                   default 58 */
    int32_t min_unit_move;           /* MIN_UNIT_MOVE                                     default 3 */
    int32_t mcts_simulations;        /* MCTS_SIMULATIONS          --mcts                  default 32 */
    int32_t threads_per_mcts;        /* THREADS_PER_MCTS          -t   (sims - sims % t)  default 2 */
    float cpuct;                     /* HP_EXPLORATION            --hp                    default 1.1 */
    float dir_noise_value;           /* DIR_NOISE_VALUE           --dnv                   default 0.3 */
    float dir_noise_epsi;            /* DIR_NOISE_EPSI            --dne                   default 0.25 */
    int32_t temperature_threshold;   /* TEMPERATURE_TRESHOLD      --temp                  default 43 */
    int32_t concurrent_descents;     /* K descents per tree in flight per leaf batch: the lockstep schedule of K of the reference's search
                                        threads with its active_N ("virtual loss") rule, alphazero_mcts.cpp:91-111.  0 or 1 = one at a
                                        time (THREADS_PER_MCTS = 1 semantics, default); must divide the simulation count; <= 16 */
} az_rules;

typedef struct az_env az_env;

/* counters accumulated on the device by az_env_rollout / az_selfplay_* (GameResults, game/game.h:17-29) */
typedef struct az_counters {
    uint64_t steps;        /* env steps applied                         */
    uint64_t games;        /* games that reached a terminal status      */
    uint64_t wins[2];      /* GameResults::players[i].win               */
    uint64_t draws;        /* GameResults::draw                         */
    uint64_t illegal;      /* rejected actions (always 0 for rollouts)  */
    uint64_t sims;         /* MCTS simulations                          */
    uint64_t evals;        /* network evaluations                       */
    uint64_t path_nodes;   /* sum over the simulations of the tree nodes walked through on the way down (depth of the descent) */
} az_counters;

AZ_API const char* az_last_error(void);
AZ_API int az_version(void);
AZ_API int az_device_count(void);
AZ_API void az_default_rules(az_rules* r);                     /* settings.h:40-62 defaults */

/* ---------------------------------------------------------------- environment (State + UtilityNN) */
/* n_games lockstep games resident in HBM on `device`; first_game_id = global id of game 0
   (games shard over GPUs by contiguous id range; the RNG contract is keyed by global id) */
AZ_API int az_env_create(int n_games, const az_rules* rules, int device, uint32_t first_game_id, az_env** out);
AZ_API int az_env_destroy(az_env* env);
AZ_API int az_env_size(const az_env* env);

/* State::newGame (state/state.cpp:137-167) for every game: Philox(seed, game, ply=0, AZ_STREAM_DEAL) */
AZ_API int az_env_reset(az_env* env, uint64_t seed, void* stream);

/* State::getData() images, n_games x 160 bytes (padding bytes are written as zero / ignored) */
AZ_API int az_env_import_aos(az_env* env, const uint8_t* h_data, void* stream);
AZ_API int az_env_export_aos(az_env* env, uint8_t* h_data, void* stream);

/* UtilityNN::getValidMoves (player/alpha_zero/alphazero_moves.cpp:3-70): 43-bit mask per game */
AZ_API int az_env_valid_moves(az_env* env, uint64_t* h_mask, void* stream);
/* State::gameStatus (state/state.cpp:518-565) */
AZ_API int az_env_status(az_env* env, int8_t* h_status, void* stream);

/* UtilityNN::makeMove (alphazero_moves.cpp:72-233) on every game + gameStatus afterwards.
   h_action[n]: 0..41 land, 42 skip.  h_dice: NULL = dice from the Philox contract
   (seed of the last az_env_reset, game, ply), else n x 5 bytes consumed in the reference's
   order (attacker dice, then defender dice).  h_status[n] receives the status byte. */
AZ_API int az_env_step(az_env* env, const uint8_t* h_action, const uint8_t* h_dice, int8_t* h_status, void* stream);
/* same with every buffer already resident in HBM; d_valid_after may be NULL */
AZ_API int az_env_step_dev(az_env* env, const uint8_t* d_action, const uint8_t* d_dice, int8_t* d_status,
                    uint64_t* d_valid_after, void* stream);

/* ScriptPlayer::takeTurn (player/script/script_player.cpp:162-227) for the side to move of every running game: one WHOLE turn per
   call (in the setup phase: the player's placement and the neutral placement), one ply.  h_script[n][2] carries the ScriptPlayer
   members that survive between calls, one packed word per (game, side); initialise with AZ_SCRIPT_INIT.  Dice / ints come from the
   scripted-opponent streams of the Philox contract (include/az_philox.h).  h_status as az_env_step. */
#define AZ_SCRIPT_INIT 0x00ffffffu
AZ_API int az_env_script_turn(az_env* env, uint32_t* h_script, int8_t* h_status, void* stream);
/* RandomPlayer::takeTurn (player/random/random_player.cpp:22-111), same calling convention (the random player keeps no members) */
AZ_API int az_env_random_turn(az_env* env, int8_t* h_status, void* stream);
/* The same with a player kind per side (AZ_OPPONENT_SCRIPT / AZ_OPPONENT_RANDOM, defined below): the games of
   AlphaZeroTrainer::trainOnGeneratedData (alphazero_trainer.cpp:242-268: Script vs Script, Script vs Random).  h_script may be NULL
   when neither side is scripted. */
AZ_API int az_env_play_turn(az_env* env, int kind_side0, int kind_side1, uint32_t* h_script, int8_t* h_status, void* stream);
/* Player::addTrainingSample (player/base/player.cpp:9-17) for those turns: every call site of script_player.cpp:105-198 and
   random_player.cpp:29-82 stages (state before the move, move) per game; when a turn ends the game, gameFinished ->
   NNTrainDataStorage::updateValues (alphazero_nn_data.cpp:51-65) turns the game's samples into packed AZ_SAMPLE_BYTES records
   (one-hot policy) in an output queue of `capacity_samples`.  A game with more than max_samples_per_game samples, or one that
   does not fit the queue any more, is dropped whole and counted.  az_env_reset discards what is staged.  az_env_turn_samples
   drains the queue (h_records = NULL: size query) — same record format and calling convention as az_selfplay_samples. */
AZ_API int az_env_record_turns(az_env* env, size_t capacity_samples, int max_samples_per_game);
AZ_API int az_env_turn_samples(az_env* env, uint8_t* h_records, size_t max_records, size_t* n_out, uint64_t* h_dropped, void* stream);

/* NNInputData(State) + setInStateTensor (neural_network/alphazero_nn_data.cpp:165-196,
   alphazero_nn.cpp:31-67): fp32 [n][7][6][13] */
AZ_API int az_env_encode(az_env* env, float* h_x, void* stream);
AZ_API int az_env_encode_dev(az_env* env, float* d_x, void* stream);

/* BASELINE config 2: n_steps lockstep steps of uniform-random legal play on every game
   (action = k-th set bit of the mask, k = mulhi(word1, popcount), dice = word0 of the
   real-move Philox block); finished games are re-dealt in place.  Counters accumulate in
   HBM; az_env_counters copies them to the host. */
AZ_API int az_env_rollout(az_env* env, int n_steps, void* stream);
AZ_API int az_env_counters(az_env* env, az_counters* h_out, int reset, void* stream);
/* seconds spent by the last rollout / step launch on the device (CUDA events on `stream`) */
AZ_API int az_env_last_kernel_ms(az_env* env, float* ms);

/* ---------------------------------------------------------------- network (AlphaZeroNN / AlphaZeroNNId forward) */
typedef struct az_nn az_nn;
#define AZ_NN_FP32 0   /* fp32 CUDA-core validation path: agrees with an fp32 restatement of the graph to <= 1e-5 */
#define AZ_NN_BF16 1   /* bf16 tcgen05 tensor-core path, fp32 accumulate / BN / heads */

/* the conv ResNet of /root/reference/python/src/build_graph.py:54-90 with `blocks` residual blocks
   (BLOCKS: 5 = shipped GraphDefs python/model/model_*_5.pb, 20 = CMake default) */
AZ_API int az_nn_create(int blocks, int device, az_nn** out);
/* the same network with value_outputs (1 or 6) value outputs: dense_2/kernel [256][value_outputs], dense_2/bias [value_outputs], each
   output through tanh.  6 = the six-seat value vector of SIXPLAYER.md §2: output k is the value of seat (cur + k) % 6, cur = the seat
   to move in the encoded position.  az_nn_create is value_outputs = 1, the reference graph */
AZ_API int az_nn_create_value(int blocks, int value_outputs, int device, az_nn** out);
/* the same network with input_planes (13 or 16) input planes: conv/kernel [3][3][input_planes][256], everything else unchanged.
   16 = the six-player seat planes of SIXPLAYER.md §2 (AZ_INPUT6_FLOATS per position): plane k (k = 0..5) holds army / 32 on the lands
   of seat (cur + k) % 6, planes 6..15 are planes 3..12 of the 13-plane encoding.  Such a network takes [n][7][6][16] in az_nn_forward,
   az_nn_train_step, az_nn_train6 and the six-player search; the two-player search and az_nn_train reject it.  az_nn_create_value is
   input_planes = 13 */
AZ_API int az_nn_create_planes(int blocks, int value_outputs, int input_planes, int device, az_nn** out);
AZ_API int az_nn_destroy(az_nn* nn);
AZ_API int az_nn_blocks(const az_nn* nn);
AZ_API int az_nn_value_outputs(const az_nn* nn);
AZ_API int az_nn_input_planes(const az_nn* nn);
AZ_API int az_nn_num_vars(const az_nn* nn);
AZ_API size_t az_nn_num_params(const az_nn* nn);
/* i-th variable: TF variable name (e.g. "res0a_branch2a/kernel"), element count, rank, shape (HWIO kernels) */
AZ_API int az_nn_var_info(const az_nn* nn, int i, const char** name, size_t* count, int* rank, int* shape4);
/* weights by TF variable name, fp32, TF layout (replaces save/restore_all, neural_network/alphazero_nn.cpp:189-204) */
AZ_API int az_nn_load_weights(az_nn* nn, const char* name, const float* h_ptr, size_t count);
AZ_API int az_nn_get_weights(const az_nn* nn, const char* name, float* h_ptr, size_t count);
/* all variables as one flat fp32 blob in inventory order (what gets broadcast between GPUs) */
AZ_API int az_nn_export_blob(const az_nn* nn, float* h_out, size_t count);
AZ_API int az_nn_import_blob(az_nn* nn, const float* h_in, size_t count);
/* the graph's "init" op (alphazero_nn.cpp:185): Glorot-uniform kernels, zero biases, BN identity */
AZ_API int az_nn_init_random(az_nn* nn, uint64_t seed);
AZ_API int az_nn_finalize(az_nn* nn);
/* AlphaZeroNN::predict / processBatchPrediction (alphazero_nn.cpp:236-267, 333-349):
   x fp32 [n][7][6][input_planes] -> policy [n][43] (softmax), value [n][value_outputs] (tanh; [n] for the one-output graph) */
AZ_API int az_nn_forward(az_nn* nn, const float* h_x, int n, float* h_policy, float* h_value, int precision, void* stream);
AZ_API int az_nn_forward_dev(az_nn* nn, const float* d_x, int n, float* d_policy, float* d_value, int precision, void* stream);

/* ---------------------------------------------------------------- training step and TensorFlow checkpoints (SURVEY.md §8f N4) */
/* One run of the graph's "optimize" op (AlphaZeroNN::train inner loop, neural_network/alphazero_nn.cpp:389-390;
   python/src/build_graph.py:92-106): training-mode forward (batch statistics, moving averages updated with momentum 0.99), softmax
   cross-entropy + mean squared error + 0.001 * L2 of the kernels, Adam(0.001, 0.9, 0.999, 1e-8).  x [n][7][6][input_planes], target policy
   [n][43], target value [n][value_outputs]; returns the batch's two losses (TF_OUTPUT_LOSS_POLICY / _VALUE; the value loss is the
   mean over all n * value_outputs squared errors).  fp32 on CUDA cores, deterministic. */
AZ_API int az_nn_train_step(az_nn* nn, const float* h_x, const float* h_target_policy, const float* h_target_value, int n,
                            float* loss_policy, float* loss_value, void* stream);
/* AlphaZeroNN::train (alphazero_nn.cpp:351-410) on packed sample records (az_selfplay_samples / the reference's sample files):
   `epochs` shuffled passes, whole batches of batch_size (SETTINGS.BATCH_SIZE = 512) only; per-epoch mean losses (may be NULL).
   Rejects a network with six value outputs (a two-player record holds one value target) or 16 input planes (two-player records
   encode 13) */
AZ_API int az_nn_train(az_nn* nn, const uint8_t* h_records, size_t n_records, int epochs, int batch_size, uint64_t seed,
                       float* h_epoch_loss_policy, float* h_epoch_loss_value, void* stream);
/* AZ_NN_FP32 (default, the parity path) or AZ_NN_BF16: the three convolution-shaped contractions of the step (forward, data gradient,
   weight gradient) as bf16 tcgen05 GEMMs with fp32 accumulation; everything else stays fp32 */
AZ_API int az_nn_train_precision(az_nn* nn, int precision);
/* AlphaZeroNNGroup::train's hand-off to the group's copies on the other GPUs (alphazero_gpu_cluster.cpp:221-231 saves a temporary
   checkpoint and reloads it): every variable, the Adam slots and the beta powers from src to dst, device to device (peer copy over
   NVLink) when the state lives on the device.  Same architecture (blocks, value outputs, input planes) required; synchronises `stream` */
AZ_API int az_nn_copy_state(az_nn* dst, az_nn* src, void* stream);
/* introspection for the parity tests: gradient of the total loss from the last step; Adam slots (which: 0 = m, 1 = v); beta powers */
AZ_API int az_nn_train_get_grad(az_nn* nn, const char* name, float* h_out, size_t count);
AZ_API int az_nn_train_get_layer(az_nn* nn, int layer, int which /* 0 = convolution output, 1 = activation */, float* h_out, size_t count);
/* test introspection of the bf16 tensor-core path.  az_nn_tc_probe: one work buffer of scratch set s as of the last bf16 forward that
   used it — which = 0 the stem operand (bf16 bits, [3 copies][2 chunks][r_alloc][8]), 1..3 the activation buffers (bf16 bits,
   [32 chunks][r_alloc][8], halo and padding rows included), 4 the per-cell head sums (float4 [n][42]); bytes must be the buffer's size
   (h_out = NULL with bytes = 0 reports r_alloc only).  az_tc_conv_test: the training step's contractions through their production
   functions — mode 0 forward conv(a [n*42][256], b = w [9][256][256] HWIO), mode 1 data gradient of dz = a through w = b, mode 2
   weight gradient [9][256][256] of activation a with dz = b [n*42][256] in at most max_splits K splits; n_warm > n first runs the same
   mode at n_warm boards with other data on the same scratch */
AZ_API int az_nn_tc_probe(az_nn* nn, int s, int which, int n, void* h_out, size_t bytes, int* r_alloc);
AZ_API int az_tc_conv_test(int mode, const float* h_a, const float* h_b, int n, int n_warm, int max_splits, float* h_out);
AZ_API int az_nn_optimizer_get(az_nn* nn, const char* name, int which, float* h_out, size_t count);
AZ_API int az_nn_optimizer_powers(az_nn* nn, float* beta1_power, float* beta2_power, uint64_t* steps);
/* AlphaZeroNN::saveCheckpoint / loadCheckpoint (alphazero_nn.cpp:189-214): TensorFlow V2 checkpoint bundle <prefix>.index +
   <prefix>.data-00000-of-00001 holding the tensors of the graph's Saver (variables, moving statistics, "<var>/optimize",
   "<var>/optimize_1", beta1_power, beta2_power) */
AZ_API int az_nn_save_checkpoint(az_nn* nn, const char* prefix);
AZ_API int az_nn_load_checkpoint(az_nn* nn, const char* prefix);

/* the bundle format itself (host only, no device needed): tensorflow/core/util/tensor_bundle */
typedef struct az_ckpt az_ckpt;
AZ_API int az_ckpt_open(const char* prefix, az_ckpt** out);
AZ_API int az_ckpt_close(az_ckpt* ckpt);
AZ_API int az_ckpt_num_tensors(const az_ckpt* ckpt);
/* i-th tensor in table (= ascending name) order; dtype is TensorFlow's DataType (DT_FLOAT = 1); shape8: up to 8 dims */
AZ_API int az_ckpt_tensor_info(const az_ckpt* ckpt, int i, const char** name, int* dtype, int* rank, int64_t* shape8, size_t* bytes);
AZ_API int az_ckpt_find(const az_ckpt* ckpt, const char* name);                 /* index or -1 */
AZ_API int az_ckpt_read(az_ckpt* ckpt, const char* name, void* h_out, size_t bytes);   /* verifies the entry's CRC32C */
AZ_API int az_ckpt_write(const char* prefix, int n, const char* const* names, const int* ranks, const int64_t* const* shapes,
                         const float* const* data);                               /* float32 tensors, one shard */
AZ_API uint32_t az_crc32c(const void* data, size_t n);
/* test / measurement entry of the training step's bf16 tcgen05 GEMM: C[M][256] = A[M][K] * B[256][K]^T for row-major fp32 host
   matrices (rounded to bf16), `splits` K splits; *ms = median device time of the GEMM launch over `reps` runs */
AZ_API int az_tc_gemm_test(const float* h_a, const float* h_b, int M, int K, int splits, int reps, float* h_c, float* ms);

/* ---------------------------------------------------------------- MCTS (AlphaZeroMCTS) and self-play */
typedef struct az_mcts az_mcts;
#define AZ_EVAL_NN 0        /* leaf evaluation by the network (az_nn) */
#define AZ_EVAL_PSEUDO 1    /* include/az_pseudo_net.h: exactly representable outputs, for bit-exact search parity tests */
#define AZ_EVAL_UNIFORM 2   /* uniform prior, value 0 ("null evaluator": tree + env cost only) */
#define AZ_EVAL_PSEUDO6 3   /* six-player search only: AZ_EVAL_PSEUDO's policy with the six-seat value vector az_pn_value6 (SIXPLAYER.md §2) */

/* one search tree (transposition table) per game of `env`; hyper-parameters come from the env's az_rules
   (mcts_simulations, threads_per_mcts -> sims - sims % t, cpuct, dir_noise_*, temperature_threshold).
   Replaces AlphaZeroMCTS (player/alpha_zero/alphazero_mcts.h:75-94) with THREADS_PER_MCTS = 1 semantics.  Evaluators AZ_EVAL_NN,
   _PSEUDO, _UNIFORM; a network with six value outputs or 16 input planes is rejected. */
AZ_API int az_mcts_create(az_env* env, az_nn* nn, int evaluator, int precision, az_mcts** out);
AZ_API int az_mcts_destroy(az_mcts* mcts);
/* node-pool occupancy: the fullest pool any game had at the end of a search since the counters were reset, the capacity of a pool
   (3 x (simulations + 1) + 64 nodes, worst-case sizing; overflows are counted in az_mcts_counters' h_errors) and the table bytes
   held per game (two pools + two hash indices) */
AZ_API int az_mcts_pool_stats(az_mcts* mcts, uint64_t* h_peak_nodes, uint64_t* h_capacity_nodes, uint64_t* h_bytes_per_game, void* stream);
/* Two game cohorts on two CUDA streams inside a search: while one cohort's leaf batch is in the tower the other cohort's tree kernel,
   state packing, stem and head tail run, and the SM pairs a tower layer's last wave leaves idle go to the other cohort's layer.
   Games are independent, so results do not depend on the setting.  0 = automatic (tensor-core evaluator, one descent per tree,
   every game searching, >= 2048 games), 1 = one stream, 2 = two cohorts wherever the conditions other than the game count hold */
AZ_API int az_mcts_set_cohorts(az_mcts* mcts, int cohorts);
AZ_API int az_mcts_simulations(const az_mcts* mcts);
/* StateSimulationsStorage::clearNodes for every game (AlphaZeroPlayer::newGame, alphazero_player.cpp:31-34) */
AZ_API int az_mcts_clear(az_mcts* mcts, void* stream);
/* AlphaZeroMCTS::simulate (alphazero_mcts.cpp:255-287) on the current state of every running game, then
   calculateMoveProbability(1.0) (:121-148) and the move choice: pick_mode 0 = pickHigestWeightedMove (play,
   alphazero_player.cpp:12), 1 = the self-play rule of alphazero_trainer.cpp:98-106 (sample while
   round <= TEMPERATURE_TRESHOLD).  h_extra_trim (NULL or [n]): additional trimNodes before the search —
   1 at the first search of a player's turn in play mode (alphazero_player.cpp:5).  apply_move != 0 also
   plays the chosen move on the env (UtilityNN::makeMove, dice from the Philox contract).
   Outputs (each may be NULL): visit counts N [n][43], pi [n][43], chosen move [n], status after [n]. */
AZ_API int az_mcts_search(az_mcts* mcts, const uint8_t* h_extra_trim, int pick_mode, int apply_move,
                          uint32_t* h_visits, float* h_pi, uint8_t* h_move, int8_t* h_status, void* stream);
/* root statistics of the last search (test introspection): Q [n][43], P [n][43], sumN [n], root value [n],
   number of live nodes in the table [n] */
AZ_API int az_mcts_root_stats(az_mcts* mcts, float* h_q, float* h_p, uint32_t* h_sumn, float* h_value, int32_t* h_table, void* stream);
/* n_moves lockstep self-play moves with no host synchronisation (threadExecuteTrainingGame,
   alphazero_trainer.cpp:80-119): search, temperature-rule move, real move, finished games re-dealt */
AZ_API int az_selfplay_run(az_mcts* mcts, int n_moves, void* stream);
/* ---- self-play training samples (SURVEY.md 8f N3).  threadExecuteTrainingGame pushes NNTrainData(player, NNInputData(rootState),
   policy) before every real move (alphazero_trainer.cpp:108) and NNTrainDataStorage::updateValues fills the values when the game
   ends (neural_network/alphazero_nn_data.cpp:51-65).  One record = what saveTrainingSamples writes per sample (:115-138):
   int8 playerIndex | NNInputData (88 B, alphazero_nn_data.h:73-101; padding bytes 43, 46, 47 written as 0) | float value |
   float policy[43], packed, 265 bytes. */
#define AZ_SAMPLE_BYTES 265
/* enable recording in az_selfplay_run / az_mcts_search(apply_move): device staging of max_moves_per_game samples per running game
   and an output queue of capacity_samples records of FINISHED games (samples that do not fit are counted as dropped) */
AZ_API int az_selfplay_record(az_mcts* mcts, size_t capacity_samples, int max_moves_per_game);
/* copies the queued records to h_records and empties the queue.  h_records = NULL while records are queued = size query
   (*n_out, *h_dropped reported, nothing reset).  Any other call DRAINS: it reports *h_dropped = samples dropped since the last
   draining call and resets that count — also when the queue is empty (h_records may then be NULL).  Every returned record was
   written: a game that does not fit the queue is dropped whole and leaves no hole (the reservation never moves past the capacity) */
AZ_API int az_selfplay_samples(az_mcts* mcts, uint8_t* h_records, size_t max_records, size_t* n_out, uint64_t* h_dropped, void* stream);
/* NNTrainDataStorage::saveTrainingSamples file: size_t count, then the records (readable by the reference's trainer) */
AZ_API int az_samples_write_file(const char* path, const uint8_t* h_records, size_t n);
/* counters since the last reset; *h_errors = node-pool + path-depth overflows (must be 0) */
AZ_API int az_mcts_counters(az_mcts* mcts, az_counters* h_out, uint64_t* h_errors, int reset, void* stream);

/* ---------------------------------------------------------------- arena: `-m play` on the device (SURVEY.md 8f N1 + N2)
   executePlay (src/alphazero_risk.cpp:4-47) -> GameGroup::playGames(pg1, pg2, games) (game/game.cpp:277-312).  Every game slot of
   the MCTS handle's env is one threadPlayGame: player index 0 = AlphaZeroPlayer (player/alpha_zero/alphazero_player.cpp:3-34: search,
   argmax move, table trimmed when its turn starts and cleared at a new game), player index 1 = the opponent; slots claim games in
   pairs like Counter::hasNext(2) (game.cpp:12-24) and play the second game of a pair as the mirror game when mirror_games != 0
   (Game::newGame, game.cpp:170-191); results are GameResults (game/game.h:17-29). */
#define AZ_OPPONENT_SCRIPT 1   /* ScriptPlayer, player/script/script_player.cpp:162-227, on the device */
#define AZ_OPPONENT_RANDOM 2   /* RandomPlayer, player/random/random_player.cpp:22-111, on the device */
#define AZ_OPPONENT_ALPHAZERO 3   /* a second AlphaZeroPlayer with its own network and search tables (az_arena_create_versus) */
typedef struct az_arena az_arena;
typedef struct az_arena_results {
    uint64_t count;               /* GameResults::count */
    uint64_t draw;                /* GameResults::draw */
    uint64_t win[2];              /* GameResults::players[i].win (0 = AlphaZero, 1 = opponent) */
    uint64_t win_and_started[2];  /* GameResults::players[i].winAndStartedGame */
    uint64_t az_moves, az_sims, az_evals, opponent_turns, ticks, errors;
} az_arena_results;
AZ_API int az_arena_create(az_mcts* mcts, int opponent, int mirror_games, az_arena** out);
/* AlphaZero vs AlphaZero: the trainer's comparison match between the new and the old model (AlphaZeroTrainer::updateIfImprovement,
   alphazero_trainer.cpp:147-166: GameGroup::playGames(trainAZPG, generateAZPG, COMPARE_GAMES)).  Player index 0 is searched by
   `mcts`, player index 1 by `opponent_mcts`; both handles must be built over the SAME env (they share the game states) and keep
   separate tables, networks and evaluators.  In the results az_* count player 0's moves, opponent_turns counts player 1's MOVES. */
AZ_API int az_arena_create_versus(az_mcts* mcts, az_mcts* opponent_mcts, int mirror_games, az_arena** out);
AZ_API int az_arena_destroy(az_arena* arena);
/* plays 2 * floor(n_games / 2) games (pairs, like the reference) over the env's slots; seed fixes the Philox contract */
AZ_API int az_arena_play(az_arena* arena, uint64_t n_games, uint64_t seed, az_arena_results* h_out, void* stream);

/* ---------------------------------------------------------------- six-player extension (BASELINE.json configs[3]) — NO reference parity
   The reference is a two-player game (PLAYER_COUNT = 2, state/state.h:13; owner = 2 bits with 2 = neutral, state.h:24-41): there
   is no six-player interface to replace.  az_env6_* is a throughput-only extension whose rules are SIXPLAYER.md (six seats, no
   neutral army, 7 lands + 13 set-up armies each, seats eliminated when they lose their last land, the eliminator takes the cards,
   simple-card trade-ins as in the reference's default STATE_SIMPLE_CARDS mode) and whose only checker is oracle/risk6_oracle.c.
   Same action space (42 lands + skip), status byte (winner seat 0..5, AZ_STATUS_DRAW, AZ_STATUS_RUNNING / _ILLEGAL / _OVER),
   az_rules fields and Philox contract as az_env_*.  State image = AZ_ENV6_IMAGE_BYTES per game: army[42], owner[42], cards[6],
   pool[6], round u16, cur, card_sets, reinf, phase, mob_from, mob_to, allow_draw, attacks, 2 pad bytes. */
typedef struct az_env6 az_env6;
#define AZ_ENV6_IMAGE_BYTES 108
typedef struct az_counters6 { uint64_t steps, games, draws, wins[6]; } az_counters6;
AZ_API int az_env6_create(int n_games, const az_rules* rules, int device, uint32_t first_game_id, az_env6** out);
AZ_API int az_env6_destroy(az_env6* env);
AZ_API int az_env6_reset(az_env6* env, uint64_t seed, void* stream);
AZ_API int az_env6_rollout(az_env6* env, int n_steps, void* stream);          /* uniform-random legal play, finished games re-dealt */
AZ_API int az_env6_last_kernel_ms(az_env6* env, float* ms);
AZ_API int az_env6_step(az_env6* env, const uint8_t* h_action, int8_t* h_status, void* stream);
AZ_API int az_env6_query(az_env6* env, uint64_t* h_valid, int8_t* h_status, void* stream);
AZ_API int az_env6_export(az_env6* env, uint8_t* h_images, void* stream);
AZ_API int az_env6_import(az_env6* env, const uint8_t* h_images, void* stream);
AZ_API int az_env6_counters(az_env6* env, az_counters6* h_out, int reset, void* stream);
/* the six-seat network input: the reference's [n][7][6][13] tensor with "enemy" = the seat that moves next, "neutral" = every other
   seat (SIXPLAYER.md), so the same tower evaluates it */
AZ_API int az_env6_encode(az_env6* env, float* h_x, void* stream);
/* the same with input_planes = 13 (az_env6_encode) or 16: [n][7][6][16], the seat planes of az_nn_create_planes */
AZ_API int az_env6_encode_planes(az_env6* env, int input_planes, float* h_x, void* stream);
/* the six-player SEARCH of SIXPLAYER.md: the reference's MCTS with the table cleared before every search and the six-seat value rule
   (a leaf's value belongs to the seat to move there: +v for that seat's nodes on the path, -v / 5 for the others); K =
   max(1, concurrent_descents) descents per tree per leaf batch under the reference's active_N rule, the two-player lockstep schedule
   (SIXPLAYER.md §2; K = 1 by default = THREADS_PER_MCTS = 1 semantics), hyper-parameters from the env's az_rules, evaluators and
   precisions as az_mcts_create.  az_mcts6_create rejects K > 16 and a simulation count (mcts_simulations - mcts_simulations %
   threads_per_mcts) that K does not divide.  Self-play, both pick modes, sample recording and the arena use the env's K.
   With a six-seat value vector (evaluator AZ_EVAL_NN over a network with six value outputs, or AZ_EVAL_PSEUDO6) a leaf's v[6] is
   relative to its seat to move L and a path node whose mover is s receives v[(s - L + 6) % 6]; a finished game backs up as above,
   and the node's stored value (root statistics) is component 0.  A one-output network keeps the scalar rule bit for bit.  Leaves are
   encoded with the network's input planes (13, or the 16 seat planes). */
typedef struct az_mcts6 az_mcts6;
AZ_API int az_mcts6_create(az_env6* env, az_nn* nn, int evaluator, int precision, az_mcts6** out);
AZ_API int az_mcts6_destroy(az_mcts6* mcts);
AZ_API int az_mcts6_search(az_mcts6* mcts, int pick_mode, int apply_move, uint32_t* h_visits, float* h_pi, uint8_t* h_move, int8_t* h_status, void* stream);
AZ_API int az_mcts6_root_stats(az_mcts6* mcts, float* h_q, float* h_p, uint32_t* h_sumn, int32_t* h_table, void* stream);
AZ_API int az_selfplay6_run(az_mcts6* mcts, int n_moves, void* stream);      /* n_moves moves of every game, finished games re-dealt */
AZ_API int az_mcts6_counters(az_mcts6* mcts, az_counters6* h_out, uint64_t* h_sims, uint64_t* h_evals, uint64_t* h_errors, int reset, void* stream);
/* ---- six-player training samples.  A record format of this project (the reference's 88-byte NNInputData has no room for six owners),
   AZ_SAMPLE6_BYTES per sample, every field 4-byte aligned:
     bytes 0..107    the root position BEFORE the move as its AZ_ENV6_IMAGE_BYTES image (az_env6_export's bytes; seat to move = byte 98)
     bytes 108..111  float value target: 1 when the seat to move won, 0 after a draw, -1/5 (the search's -v / 5 with v = 1) otherwise
                     (the format is the same for both value widths: a six-output network's targets are derived from the status)
     bytes 112..283  float policy target[43]: the search's pi for that move (az_mcts6_search's h_pi), bit for bit
     byte  284       int8 final status of the game (winner seat 0..5 or AZ_STATUS_DRAW); bytes 285..287 zero */
#define AZ_SAMPLE6_BYTES 288
/* enable recording in az_selfplay6_run / az_mcts6_search(apply_move != 0), both pick modes: every real move stages one sample per game
   (max_moves_per_game per game on the device, about 288 bytes each); when a game ends its samples go to an output queue of
   capacity_samples records as one contiguous block with their value targets.  A game that overflows its staging area or does not fit
   the queue is dropped whole and counted.  Staged samples of games abandoned by az_env6_reset / az_env6_import are discarded.
   Recording changes nothing the search computes. */
AZ_API int az_selfplay6_record(az_mcts6* mcts, size_t capacity_samples, int max_moves_per_game);
/* drains the six-player queue: the calling convention of az_selfplay_samples with AZ_SAMPLE6_BYTES records */
AZ_API int az_selfplay6_samples(az_mcts6* mcts, uint8_t* h_records, size_t max_records, size_t* n_out, uint64_t* h_dropped, void* stream);
/* az_nn_train on AZ_SAMPLE6_BYTES records: the same shuffled epochs, whole batches, per-epoch mean losses and training precisions; the
   input planes are the six-seat encoding of az_env6_encode_planes with the network's plane count, built on the device from each
   record's image.  With six value outputs
   target k of a record is the value rule above for seat (cur + k) % 6 (1 for the winner, -1/5 for another seat, 0 after a draw);
   component 0 is the stored float */
AZ_API int az_nn_train6(az_nn* nn, const uint8_t* h_records, size_t n_records, int epochs, int batch_size, uint64_t seed,
                        float* h_epoch_loss_policy, float* h_epoch_loss_value, void* stream);
/* the scripted agent's action (SIXPLAYER.md §5) for the current position of every game, one byte per game: a land 0..41 or 42 =
   skip, always legal; 0xff for a finished game.  A pure function of the position and the env's rules (no randomness, no memory);
   az_env6_step with these actions plays the scripted agent's ply with the real-move dice, as the arena does. */
AZ_API int az_env6_script_actions(az_env6* env, uint8_t* h_action, void* stream);
/* ---- six-player arena (SIXPLAYER.md §4): seat-rotated matches between searchers, the uniform-random player and the scripted agent
   over one env6.  An agent is an az_mcts6 handle over `env` (argmax play, table cleared per search), the uniform-random player
   (az_env6_rollout's rule) or the scripted agent (az_env6_script_actions' rule, SIXPLAYER.md §5).  seat_agent[s] = the agent index that holds seat s; every agent holds at least one seat.  Match game g
   (first_game <= g < first_game + n_games) starts from the deal of game id d (e6_new_game(seed, d, 0)) with ply 0; with rotate_seats
   d = g - g % 6 and seat s is played by seat_agent[(s + g % 6) % 6] (the six games of a group share one deal, every agent sits in
   every seat), without it d = g and seat s by seat_agent[s].  All randomness of a ply is keyed by (seed, g, ply), so a game's
   result depends only on (seed, g, agents), never on the slot that played it or the env's size: a multi-GPU match is disjoint
   first_game ranges plus az_dist_gather_stats over the result struct (all uint64_t). */
typedef struct az_arena6 az_arena6;
typedef struct az_arena6_results {
    uint64_t count, draw;
    uint64_t win[6];        /* by agent index */
    uint64_t win_seat[6];   /* by seat */
    uint64_t moves[6];      /* plies played, by agent index */
    uint64_t sims, evals, ticks, errors;   /* errors = the searchers' overflow counters, must be 0 */
} az_arena6_results;
#define AZ_AGENT6_SEARCHER 0
#define AZ_AGENT6_RANDOM 1
#define AZ_AGENT6_SCRIPT 2
/* kinds[i] = the kind of agent i; agents[i] is an az_mcts6 handle for AZ_AGENT6_SEARCHER and NULL for the other kinds.  Rejects
   unknown kinds, a handle that does not match its kind, handles over another env, the same handle twice, n_agents outside 1..6,
   seat_agent entries >= n_agents and agents without a seat */
AZ_API int az_arena6_create_agents(az_env6* env, az_mcts6* const* agents, const int* kinds /*[n_agents]*/, int n_agents,
                                   const uint8_t* seat_agent /*[6]*/, int rotate_seats, az_arena6** out);
/* az_arena6_create_agents with agents[i] == NULL meaning the uniform-random player and a handle a searcher */
AZ_API int az_arena6_create(az_env6* env, az_mcts6* const* agents, int n_agents, const uint8_t* seat_agent /*[6]*/,
                            int rotate_seats, az_arena6** out);
AZ_API int az_arena6_destroy(az_arena6* arena);
/* resets the env with `seed` and zeroes the searchers' counters, then plays the match over the env's slots.  h_status / h_plies: NULL
   or [n_games], per match game (winner seat 0..5 or AZ_STATUS_DRAW; plies).  Rejects handles with recording enabled, with rotation
   first_game or n_games not a multiple of 6, and first_game + n_games > 2^32.  The handles search stand-alone as before afterwards. */
AZ_API int az_arena6_play(az_arena6* arena, uint64_t first_game, uint64_t n_games, uint64_t seed, az_arena6_results* h_out,
                          int8_t* h_status, uint32_t* h_plies, void* stream);
/* the number of slots that held a game at each tick of the last az_arena6_play (*n_out = its ticks; h_active = NULL: size query) */
AZ_API int az_arena6_active_slots(az_arena6* arena, uint32_t* h_active, size_t max_ticks, size_t* n_out);
/* ---- six-player generated games (SIXPLAYER.md §6): scripted and random play recorded on the device as training records.
   az_env6_play plays n_plies plies of every game with no host synchronisation: the seat to move, cur, plays by seat_kind[cur]
   (AZ_AGENT6_RANDOM = az_env6_rollout's rule, AZ_AGENT6_SCRIPT = az_env6_script_actions' rule), both with the real-move dice of
   (seed, first_game_id + slot, ply).  Finished games are counted and re-dealt in place on az_env6_rollout's schedule and the env
   counters accumulate as there, so six random seats without recording are az_env6_rollout bit for bit.  Bit s of record_seats
   (< 64) records every ply seat s plays, forced plies included: the image before the ply and the played action, staged per slot
   until the game ends.  When a game ends, in any call on a recording env (record_seats = 0 included), its samples become
   AZ_SAMPLE6_BYTES records (value target as above for the final status, policy target 1.0f at the played action and 0 elsewhere)
   in one contiguous block of the queue, within the call in which it ended;
   a game that is still running keeps its staged samples for the next call.  Recording changes no state, dice or counter.  Rejects
   a seat_kind entry that is not RANDOM or SCRIPT, seat_kind == NULL, n_plies < 0, record_seats >= 64 and record_seats != 0 without
   az_env6_record.  Only az_env6_play's own plies are staged: if az_env6_step, az_env6_rollout or a search moves the games in
   between, a game's block holds only the plies az_env6_play played.  az_env6_reset and az_env6_import (so az_arena6_play too)
   discard the staged samples.  Timed by az_env6_last_kernel_ms. */
AZ_API int az_env6_play(az_env6* env, const int* seat_kind /*[6]*/, uint32_t record_seats, int n_plies, void* stream);
/* enable recording in az_env6_play: max_samples_per_game staged samples per slot on the device (112 bytes each), an output queue of
   capacity_samples records.  A game with more samples, or one that does not fit the queue, is dropped whole and counted.  Rejects
   capacity_samples == 0, max_samples_per_game <= 0 and a second call */
AZ_API int az_env6_record(az_env6* env, size_t capacity_samples, int max_samples_per_game);
/* drains the queue of az_env6_play: the calling convention of az_selfplay6_samples (h_records = NULL: size query; a drain resets the
   dropped count).  Rejected before az_env6_record */
AZ_API int az_env6_samples(az_env6* env, uint8_t* h_records, size_t max_records, size_t* n_out, uint64_t* h_dropped, void* stream);

/* ---------------------------------------------------------------- multi-GPU (SURVEY.md 8e): NCCL over NVLink / NVSwitch, never inside a search
   Games shard over GPUs by contiguous global id (first_game_id of az_env_create) and never migrate; every GPU holds a full copy of
   the network.  The only exchanges are the two below.  NCCL is loaded at run time (libnccl.so.2); without it az_dist_init* fail
   with AZ_ERR_NOT_READY and the rest of the library works unchanged.
   Process models: az_dist_init = ONE process drives n GPUs, the reference's model (AlphaZeroCluster::initGpus, neural_network/
   alphazero_gpu_cluster.cpp:147-158; rank i = devices[i], n local members); az_dist_init_rank = one process per GPU (one local
   member; rank 0 creates the id with az_dist_unique_id and ships its AZ_DIST_ID_BYTES bytes to the other ranks by any side
   channel).  Arrays indexed "per local member" have az_dist_local_count() entries, in member order. */
typedef struct az_dist az_dist;
#define AZ_DIST_ID_BYTES 128
AZ_API int az_dist_nccl_version(int* version);
AZ_API int az_dist_init(int n_devices, const int* devices /* NULL = 0 .. n-1 */, az_dist** out);
AZ_API int az_dist_unique_id(uint8_t* id128);
AZ_API int az_dist_init_rank(int world_size, int rank, const uint8_t* id128, int device, az_dist** out);
AZ_API int az_dist_destroy(az_dist* dist);
AZ_API int az_dist_world_size(const az_dist* dist);
AZ_API int az_dist_local_count(const az_dist* dist);
AZ_API int az_dist_rank(const az_dist* dist, int local_index);
/* AlphaZeroNNGroup::train's hand-off of the trained model to the group's copies on the other GPUs (alphazero_gpu_cluster.cpp:221-231
   writes a temporary checkpoint file and reloads it on every other GPU): ncclBroadcast of root_rank's variables (weights and
   BatchNorm moving statistics, fp32, device to device) into nn[i] of every member.  The optimizer slots stay with the trainer
   (az_nn_copy_state moves them too, inside one process).  Collective: every rank must call it. */
AZ_API int az_dist_broadcast_weights(az_dist* dist, az_nn* const* nn, int n_local, int root_rank);
/* GameResults::add over the per-thread results after thread::join (game/game.cpp:298-309): n 64-bit counters per member,
   h_local = [n_local][n]; h_sum = [n] totals over every rank (ncclAllReduce), h_per_rank = [world][n] (ncclAllGather); either
   output may be NULL.  Collective.  The typed forms sum az_counters (az_env_counters / az_mcts_counters) and az_arena_results
   (az_arena_play) field by field. */
AZ_API int az_dist_gather_stats(az_dist* dist, const uint64_t* h_local, int n, uint64_t* h_sum, uint64_t* h_per_rank);
AZ_API int az_dist_gather_counters(az_dist* dist, const az_counters* h_local, az_counters* h_total);
AZ_API int az_dist_gather_results(az_dist* dist, const az_arena_results* h_local, az_arena_results* h_total);
/* every rank has arrived and the earlier device work of its members is complete */
AZ_API int az_dist_barrier(az_dist* dist);

#ifdef __cplusplus
}
#endif
#endif /* AZ_B200_H */
