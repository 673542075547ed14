"""Host-side Python binding of libaz_b200.so (ctypes over the C ABI of include/az_b200.h).

This is plumbing for tests, bench.py and torch.distributed launches; the product is the
CUDA library.  There is NO CPU fallback: importing works anywhere (so the CPU test-suite
can check that the library loads and exports its symbols), but creating any handle without
a CUDA device raises AzError.
"""
import ctypes as C
import os

import numpy as np

PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG, "libaz_b200.so")

LANDS, MOVES, SKIP, NONE = 42, 43, 42, 43
DATA_BYTES, INPUT_FLOATS = 160, 546
INPUT6_FLOATS = 672     # [7][6][16]: the six-player seat planes (AZ_INPUT6_FLOATS, Net(input_planes=16))
STATUS_RUNNING, STATUS_DRAW, STATUS_ILLEGAL, STATUS_OVER = -1, -2, -3, -4


class AzError(RuntimeError):
    pass


class AzRules(C.Structure):
    """mirror of az_rules / SETTINGS.* (reference src/settings.h:40-62)"""
    _fields_ = [("allow_yield", C.c_int32), ("limit_reinforcement", C.c_int32), ("limit_attack", C.c_int32),
                ("max_game_rounds", C.c_int32), ("min_unit_move", C.c_int32), ("mcts_simulations", C.c_int32),
                ("threads_per_mcts", C.c_int32), ("cpuct", C.c_float), ("dir_noise_value", C.c_float),
                ("dir_noise_epsi", C.c_float), ("temperature_threshold", C.c_int32),
                ("concurrent_descents", C.c_int32)]


class AzCounters(C.Structure):
    _fields_ = [("steps", C.c_uint64), ("games", C.c_uint64), ("wins", C.c_uint64 * 2), ("draws", C.c_uint64),
                ("illegal", C.c_uint64), ("sims", C.c_uint64), ("evals", C.c_uint64), ("path_nodes", C.c_uint64)]

    def as_dict(self):
        return dict(steps=int(self.steps), games=int(self.games), wins=[int(self.wins[0]), int(self.wins[1])],
                    draws=int(self.draws), illegal=int(self.illegal), sims=int(self.sims), evals=int(self.evals),
                    path_nodes=int(self.path_nodes))


class AzCounters6(C.Structure):
    _fields_ = [("steps", C.c_uint64), ("games", C.c_uint64), ("draws", C.c_uint64), ("wins", C.c_uint64 * 6)]


_lib = None


def lib():
    """loads libaz_b200.so; raises AzError (never falls back) when it has not been built"""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise AzError("libaz_b200.so is missing: run `python -m alphazero_risk_b200.build` (nvcc, sm_100a)")
        L = C.CDLL(LIB_PATH)
        vp, u8, i8, u64, f32 = C.c_void_p, C.POINTER(C.c_uint8), C.POINTER(C.c_int8), C.POINTER(C.c_uint64), C.POINTER(C.c_float)
        L.az_last_error.restype = C.c_char_p
        L.az_default_rules.argtypes = [C.POINTER(AzRules)]
        L.az_env_create.argtypes = [C.c_int, C.POINTER(AzRules), C.c_int, C.c_uint32, C.POINTER(vp)]
        L.az_env_destroy.argtypes = [vp]
        L.az_env_size.argtypes = [vp]
        L.az_env_reset.argtypes = [vp, C.c_uint64, vp]
        L.az_env_import_aos.argtypes = [vp, vp, vp]
        L.az_env_export_aos.argtypes = [vp, vp, vp]
        L.az_env_valid_moves.argtypes = [vp, vp, vp]
        L.az_env_status.argtypes = [vp, vp, vp]
        L.az_env_step.argtypes = [vp, vp, vp, vp, vp]
        L.az_env_step_dev.argtypes = [vp, vp, vp, vp, vp, vp]
        L.az_env_encode.argtypes = [vp, vp, vp]
        L.az_env_encode_dev.argtypes = [vp, vp, vp]
        L.az_env_rollout.argtypes = [vp, C.c_int, vp]
        L.az_env_counters.argtypes = [vp, C.POINTER(AzCounters), C.c_int, vp]
        L.az_env_last_kernel_ms.argtypes = [vp, C.POINTER(C.c_float)]
        L.az_nn_create.argtypes = [C.c_int, C.c_int, C.POINTER(vp)]
        L.az_nn_create_value.argtypes = [C.c_int, C.c_int, C.c_int, C.POINTER(vp)]
        L.az_nn_value_outputs.argtypes = [vp]
        L.az_nn_value_outputs.restype = C.c_int
        L.az_nn_create_planes.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(vp)]
        L.az_nn_input_planes.argtypes = [vp]
        L.az_nn_input_planes.restype = C.c_int
        L.az_nn_destroy.argtypes = [vp]
        L.az_nn_blocks.argtypes = [vp]
        L.az_nn_num_vars.argtypes = [vp]
        L.az_nn_num_params.argtypes = [vp]
        L.az_nn_num_params.restype = C.c_size_t
        L.az_nn_var_info.argtypes = [vp, C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_size_t), C.POINTER(C.c_int), C.POINTER(C.c_int * 4)]
        L.az_nn_load_weights.argtypes = [vp, C.c_char_p, vp, C.c_size_t]
        L.az_nn_get_weights.argtypes = [vp, C.c_char_p, vp, C.c_size_t]
        L.az_nn_export_blob.argtypes = [vp, vp, C.c_size_t]
        L.az_nn_import_blob.argtypes = [vp, vp, C.c_size_t]
        L.az_nn_init_random.argtypes = [vp, C.c_uint64]
        L.az_nn_finalize.argtypes = [vp]
        L.az_nn_forward.argtypes = [vp, vp, C.c_int, vp, vp, C.c_int, vp]
        L.az_nn_forward_dev.argtypes = [vp, vp, C.c_int, vp, vp, C.c_int, vp]
        L.az_nn_train_step.argtypes = [vp, vp, vp, vp, C.c_int, f32, f32, vp]
        L.az_nn_train.argtypes = [vp, vp, C.c_size_t, C.c_int, C.c_int, C.c_uint64, vp, vp, vp]
        L.az_nn_train_get_grad.argtypes = [vp, C.c_char_p, vp, C.c_size_t]
        L.az_nn_train_precision.argtypes = [vp, C.c_int]
        L.az_nn_copy_state.argtypes = [vp, vp, vp]
        L.az_nn_train_get_layer.argtypes = [vp, C.c_int, C.c_int, vp, C.c_size_t]
        L.az_nn_optimizer_get.argtypes = [vp, C.c_char_p, C.c_int, vp, C.c_size_t]
        L.az_nn_optimizer_powers.argtypes = [vp, f32, f32, u64]
        L.az_nn_save_checkpoint.argtypes = [vp, C.c_char_p]
        L.az_nn_load_checkpoint.argtypes = [vp, C.c_char_p]
        L.az_ckpt_open.argtypes = [C.c_char_p, C.POINTER(vp)]
        L.az_ckpt_close.argtypes = [vp]
        L.az_ckpt_num_tensors.argtypes = [vp]
        L.az_ckpt_tensor_info.argtypes = [vp, C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int64 * 8),
                                          C.POINTER(C.c_size_t)]
        L.az_ckpt_find.argtypes = [vp, C.c_char_p]
        L.az_ckpt_read.argtypes = [vp, C.c_char_p, vp, C.c_size_t]
        L.az_ckpt_write.argtypes = [C.c_char_p, C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_int), C.POINTER(C.POINTER(C.c_int64)),
                                    C.POINTER(vp)]
        L.az_crc32c.argtypes = [vp, C.c_size_t]
        L.az_crc32c.restype = C.c_uint32
        L.az_mcts_create.argtypes = [vp, vp, C.c_int, C.c_int, C.POINTER(vp)]
        L.az_mcts_destroy.argtypes = [vp]
        L.az_mcts_simulations.argtypes = [vp]
        L.az_mcts_set_cohorts.argtypes = [vp, C.c_int]
        L.az_mcts_pool_stats.argtypes = [vp, u64, u64, u64, vp]
        L.az_mcts_clear.argtypes = [vp, vp]
        L.az_mcts_search.argtypes = [vp, vp, C.c_int, C.c_int, vp, vp, vp, vp, vp]
        L.az_mcts_root_stats.argtypes = [vp, vp, vp, vp, vp, vp, vp]
        L.az_selfplay_run.argtypes = [vp, C.c_int, vp]
        L.az_mcts_counters.argtypes = [vp, C.POINTER(AzCounters), C.POINTER(C.c_uint64), C.c_int, vp]
        L.az_selfplay_record.argtypes = [vp, C.c_size_t, C.c_int]
        L.az_env_script_turn.argtypes = [vp, vp, vp, vp]
        L.az_env_random_turn.argtypes = [vp, vp, vp]
        L.az_env_play_turn.argtypes = [vp, C.c_int, C.c_int, vp, vp, vp]
        L.az_env_record_turns.argtypes = [vp, C.c_size_t, C.c_int]
        L.az_env_turn_samples.argtypes = [vp, vp, C.c_size_t, C.POINTER(C.c_size_t), C.POINTER(C.c_uint64), vp]
        L.az_arena_create.argtypes = [vp, C.c_int, C.c_int, C.POINTER(vp)]
        L.az_arena_create_versus.argtypes = [vp, vp, C.c_int, C.POINTER(vp)]
        L.az_arena_destroy.argtypes = [vp]
        L.az_arena_play.argtypes = [vp, C.c_uint64, C.c_uint64, C.POINTER(AzArenaResults), vp]
        L.az_selfplay_samples.argtypes = [vp, vp, C.c_size_t, C.POINTER(C.c_size_t), C.POINTER(C.c_uint64), vp]
        L.az_samples_write_file.argtypes = [C.c_char_p, vp, C.c_size_t]
        L.az_env6_create.argtypes = [C.c_int, C.POINTER(AzRules), C.c_int, C.c_uint32, C.POINTER(vp)]
        L.az_env6_destroy.argtypes = [vp]
        L.az_env6_reset.argtypes = [vp, C.c_uint64, vp]
        L.az_env6_rollout.argtypes = [vp, C.c_int, vp]
        L.az_env6_last_kernel_ms.argtypes = [vp, C.POINTER(C.c_float)]
        L.az_env6_step.argtypes = [vp, vp, vp, vp]
        L.az_env6_query.argtypes = [vp, vp, vp, vp]
        L.az_env6_script_actions.argtypes = [vp, vp, vp]
        L.az_env6_play.argtypes = [vp, vp, C.c_uint32, C.c_int, vp]
        L.az_env6_record.argtypes = [vp, C.c_size_t, C.c_int]
        L.az_env6_samples.argtypes = [vp, vp, C.c_size_t, C.POINTER(C.c_size_t), C.POINTER(C.c_uint64), vp]
        L.az_env6_export.argtypes = [vp, vp, vp]
        L.az_env6_import.argtypes = [vp, vp, vp]
        L.az_env6_counters.argtypes = [vp, C.POINTER(AzCounters6), C.c_int, vp]
        L.az_env6_encode.argtypes = [vp, vp, vp]
        L.az_env6_encode_planes.argtypes = [vp, C.c_int, vp, vp]
        L.az_mcts6_create.argtypes = [vp, vp, C.c_int, C.c_int, C.POINTER(vp)]
        L.az_mcts6_destroy.argtypes = [vp]
        L.az_mcts6_search.argtypes = [vp, C.c_int, C.c_int, vp, vp, vp, vp, vp]
        L.az_mcts6_root_stats.argtypes = [vp, vp, vp, vp, vp, vp]
        L.az_selfplay6_run.argtypes = [vp, C.c_int, vp]
        L.az_mcts6_counters.argtypes = [vp, C.POINTER(AzCounters6), u64, u64, u64, C.c_int, vp]
        L.az_selfplay6_record.argtypes = [vp, C.c_size_t, C.c_int]
        L.az_selfplay6_samples.argtypes = [vp, vp, C.c_size_t, C.POINTER(C.c_size_t), C.POINTER(C.c_uint64), vp]
        L.az_nn_train6.argtypes = [vp, vp, C.c_size_t, C.c_int, C.c_int, C.c_uint64, vp, vp, vp]
        L.az_arena6_create.argtypes = [vp, C.POINTER(vp), C.c_int, vp, C.c_int, C.POINTER(vp)]
        L.az_arena6_create_agents.argtypes = [vp, C.POINTER(vp), vp, C.c_int, vp, C.c_int, C.POINTER(vp)]
        L.az_arena6_destroy.argtypes = [vp]
        L.az_arena6_play.argtypes = [vp, C.c_uint64, C.c_uint64, C.c_uint64, C.POINTER(AzArena6Results), vp, vp, vp]
        L.az_arena6_active_slots.argtypes = [vp, vp, C.c_size_t, C.POINTER(C.c_size_t)]
        L.az_dist_nccl_version.argtypes = [C.POINTER(C.c_int)]
        L.az_dist_init.argtypes = [C.c_int, C.POINTER(C.c_int), C.POINTER(vp)]
        L.az_dist_unique_id.argtypes = [vp]
        L.az_dist_init_rank.argtypes = [C.c_int, C.c_int, vp, C.c_int, C.POINTER(vp)]
        L.az_dist_destroy.argtypes = [vp]
        L.az_dist_world_size.argtypes = [vp]
        L.az_dist_local_count.argtypes = [vp]
        L.az_dist_rank.argtypes = [vp, C.c_int]
        L.az_dist_broadcast_weights.argtypes = [vp, C.POINTER(vp), C.c_int, C.c_int]
        L.az_dist_gather_stats.argtypes = [vp, vp, C.c_int, vp, vp]
        L.az_dist_gather_counters.argtypes = [vp, C.POINTER(AzCounters), C.POINTER(AzCounters)]
        L.az_dist_gather_results.argtypes = [vp, C.POINTER(AzArenaResults), C.POINTER(AzArenaResults)]
        L.az_dist_barrier.argtypes = [vp]
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise AzError("libaz_b200 error %d: %s" % (rc, lib().az_last_error().decode()))


def default_rules(**kw):
    r = AzRules()
    lib().az_default_rules(C.byref(r))
    for k, v in kw.items():
        setattr(r, k, v)
    return r


def _ptr(a):
    return C.c_void_p(a.ctypes.data)


class Env:
    """n lockstep Risk games resident in HBM (az_env_*)."""

    def __init__(self, n_games, rules=None, device=0, first_game_id=0):
        self.L = lib()
        self.n = int(n_games)
        self.rules = rules if rules is not None else default_rules()
        self.device = device
        h = C.c_void_p()
        check(self.L.az_env_create(self.n, C.byref(self.rules), device, first_game_id, C.byref(h)))
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.L.az_env_destroy(self.h)
            self.h = None

    __del__ = close

    def reset(self, seed, stream=None):
        check(self.L.az_env_reset(self.h, int(seed), stream))

    def import_aos(self, data, stream=None):
        a = np.ascontiguousarray(data, np.uint8)
        assert a.shape == (self.n, DATA_BYTES)
        check(self.L.az_env_import_aos(self.h, _ptr(a), stream))

    def export_aos(self, out=None, stream=None):
        a = out if out is not None else np.empty((self.n, DATA_BYTES), np.uint8)
        check(self.L.az_env_export_aos(self.h, _ptr(a), stream))
        return a

    def valid_moves(self, stream=None):
        a = np.empty(self.n, np.uint64)
        check(self.L.az_env_valid_moves(self.h, _ptr(a), stream))
        return a

    def status(self, stream=None):
        a = np.empty(self.n, np.int8)
        check(self.L.az_env_status(self.h, _ptr(a), stream))
        return a

    def step(self, action, dice=None, out=None, stream=None):
        act = np.ascontiguousarray(action, np.uint8)
        assert act.shape == (self.n,)
        st = out if out is not None else np.empty(self.n, np.int8)
        d = None
        if dice is not None:
            d = np.ascontiguousarray(dice, np.uint8)
            assert d.shape == (self.n, 5)
        check(self.L.az_env_step(self.h, _ptr(act), _ptr(d) if d is not None else None, _ptr(st), stream))
        return st

    def step_dev(self, d_action, d_dice, d_status, d_valid_after=None, stream=None):
        """raw device pointers (ints), e.g. torch tensors' data_ptr()"""
        check(self.L.az_env_step_dev(self.h, d_action, d_dice, d_status, d_valid_after, stream))

    def script_turn(self, script, stream=None):
        """ScriptPlayer::takeTurn for the side to move of every running game; `script` = uint32 [n, 2] (in/out), SCRIPT_INIT at first"""
        st = np.empty(self.n, np.int8)
        check(self.L.az_env_script_turn(self.h, _ptr(script), _ptr(st), stream))
        return st

    def random_turn(self, stream=None):
        """RandomPlayer::takeTurn for the side to move of every running game"""
        st = np.empty(self.n, np.int8)
        check(self.L.az_env_random_turn(self.h, _ptr(st), stream))
        return st

    def play_turn(self, kind_side0, kind_side1, script=None, stream=None):
        """one turn of every running game, side 0 / side 1 played by OPPONENT_SCRIPT or OPPONENT_RANDOM (az_env_play_turn)"""
        st = np.empty(self.n, np.int8)
        check(self.L.az_env_play_turn(self.h, int(kind_side0), int(kind_side1), _ptr(script) if script is not None else None, _ptr(st), stream))
        return st

    def record_turns(self, capacity_samples, max_samples_per_game=4096):
        """record what Player::addTrainingSample receives inside scripted / random turns (az_env_record_turns)"""
        check(self.L.az_env_record_turns(self.h, C.c_size_t(int(capacity_samples)), int(max_samples_per_game)))

    def turn_samples(self, stream=None):
        """finished games' samples as a [k, 265] uint8 array (reference file layout per record) and the dropped count"""
        n, dropped = C.c_size_t(0), C.c_uint64(0)
        check(self.L.az_env_turn_samples(self.h, None, C.c_size_t(0), C.byref(n), C.byref(dropped), stream))
        out = np.empty((n.value, SAMPLE_BYTES), np.uint8)
        if n.value:          # an empty queue was drained (and its dropped count reset) by the query itself
            check(self.L.az_env_turn_samples(self.h, _ptr(out), C.c_size_t(n.value), C.byref(n), C.byref(dropped), stream))
        return out[:n.value], int(dropped.value)

    def encode(self, stream=None):
        a = np.empty((self.n, 7, 6, 13), np.float32)
        check(self.L.az_env_encode(self.h, _ptr(a), stream))
        return a

    def encode_dev(self, d_x, stream=None):
        check(self.L.az_env_encode_dev(self.h, d_x, stream))

    def rollout(self, n_steps, stream=None):
        check(self.L.az_env_rollout(self.h, int(n_steps), stream))

    def counters(self, reset=False, stream=None):
        c = AzCounters()
        check(self.L.az_env_counters(self.h, C.byref(c), int(reset), stream))
        return c.as_dict()

    def last_kernel_ms(self):
        ms = C.c_float(0)
        check(self.L.az_env_last_kernel_ms(self.h, C.byref(ms)))
        return float(ms.value)


FP32, BF16 = 0, 1


class Net:
    """the policy/value conv ResNet (az_nn_*); weights keyed by the reference graph's TF variable names.  value_outputs = 6: the
    six-seat value vector of SIXPLAYER.md §2 (output k = the value of seat (cur + k) % 6); 1 = the reference graph.  input_planes = 16:
    the six-player seat planes of SIXPLAYER.md §2 (inputs [n, 42 * 16], Env6.encode(planes=16)); 13 = the reference graph"""

    def __init__(self, blocks=5, device=0, seed=None, value_outputs=1, input_planes=13):
        self.L = lib()
        h = C.c_void_p()
        check(self.L.az_nn_create_planes(int(blocks), int(value_outputs), int(input_planes), device, C.byref(h)))
        self.h, self.blocks, self.device = h, int(blocks), device
        self.value_outputs = int(self.L.az_nn_value_outputs(h))
        self.input_planes = int(self.L.az_nn_input_planes(h))
        if seed is not None:
            self.init_random(seed)

    def close(self):
        if getattr(self, "h", None):
            self.L.az_nn_destroy(self.h)
            self.h = None

    __del__ = close

    def variables(self):
        out = []
        for i in range(self.L.az_nn_num_vars(self.h)):
            name, cnt, rank, shp = C.c_char_p(), C.c_size_t(), C.c_int(), (C.c_int * 4)()
            check(self.L.az_nn_var_info(self.h, i, C.byref(name), C.byref(cnt), C.byref(rank), C.byref(shp)))
            out.append((name.value.decode(), tuple(shp[k] for k in range(rank.value))))
        return out

    def num_params(self):
        return int(self.L.az_nn_num_params(self.h))

    def init_random(self, seed):
        check(self.L.az_nn_init_random(self.h, int(seed)))

    def load(self, name, array):
        a = np.ascontiguousarray(array, np.float32)
        check(self.L.az_nn_load_weights(self.h, name.encode(), _ptr(a), a.size))

    def get(self, name, shape):
        a = np.empty(shape, np.float32)
        check(self.L.az_nn_get_weights(self.h, name.encode(), _ptr(a), a.size))
        return a

    def weights(self):
        return {n: self.get(n, s) for n, s in self.variables()}

    def export_blob(self):
        a = np.empty(self.num_params(), np.float32)
        check(self.L.az_nn_export_blob(self.h, _ptr(a), a.size))
        return a

    def import_blob(self, blob):
        a = np.ascontiguousarray(blob, np.float32)
        check(self.L.az_nn_import_blob(self.h, _ptr(a), a.size))

    def finalize(self):
        check(self.L.az_nn_finalize(self.h))

    def forward(self, x, precision=FP32, stream=None):
        """x [n, 42 * input_planes] (any shape of that size) -> (policy [n, 43], value [n] with one value output, [n, 6] with six)"""
        a = np.ascontiguousarray(x, np.float32).reshape(-1, 42 * self.input_planes)
        n = a.shape[0]
        pol = np.empty((n, MOVES), np.float32)
        val = np.empty(n, np.float32) if self.value_outputs == 1 else np.empty((n, self.value_outputs), np.float32)
        check(self.L.az_nn_forward(self.h, _ptr(a), n, _ptr(pol), _ptr(val), precision, stream))
        return pol, val

    def forward_dev(self, d_x, n, d_policy, d_value, precision=FP32, stream=None):
        check(self.L.az_nn_forward_dev(self.h, d_x, int(n), d_policy, d_value, precision, stream))

    # ---- training step and checkpoints (AlphaZeroNN::train / saveCheckpoint / loadCheckpoint)
    def train_step(self, x, target_policy, target_value, stream=None):
        """one optimizer step on a batch x [n, 42 * input_planes]; target_value [n] (one value output) or [n, 6] (six); returns (policy
        loss, value loss)"""
        a = np.ascontiguousarray(x, np.float32).reshape(-1, 42 * self.input_planes)
        tp = np.ascontiguousarray(target_policy, np.float32).reshape(-1, MOVES)
        tv = np.ascontiguousarray(target_value, np.float32)
        assert tv.shape == ((a.shape[0],) if self.value_outputs == 1 else (a.shape[0], self.value_outputs)), tv.shape
        assert tp.shape[0] == a.shape[0]
        lp, lv = C.c_float(), C.c_float()
        check(self.L.az_nn_train_step(self.h, _ptr(a), _ptr(tp), _ptr(tv), a.shape[0], C.byref(lp), C.byref(lv), stream))
        return float(lp.value), float(lv.value)

    def train(self, records, epochs, batch_size=512, seed=0, stream=None):
        """AlphaZeroNN::train on packed 265-byte sample records; returns per-epoch (policy loss, value loss) means"""
        r = np.ascontiguousarray(records, np.uint8).reshape(-1, SAMPLE_BYTES)
        lp, lv = np.zeros(epochs, np.float32), np.zeros(epochs, np.float32)
        check(self.L.az_nn_train(self.h, _ptr(r), r.shape[0], int(epochs), int(batch_size), int(seed), _ptr(lp), _ptr(lv), stream))
        return lp, lv

    def train6(self, records, epochs, batch_size=512, seed=0, stream=None):
        """train() on six-player SAMPLE6_BYTES records (Mcts6.samples), with the six-seat input encoding; returns per-epoch
        (policy loss, value loss) means.  With six value outputs target k of a record is the value of seat (cur + k) % 6 under the
        record's final status"""
        r = np.ascontiguousarray(records, np.uint8).reshape(-1, SAMPLE6_BYTES)
        lp, lv = np.zeros(epochs, np.float32), np.zeros(epochs, np.float32)
        check(self.L.az_nn_train6(self.h, _ptr(r), r.shape[0], int(epochs), int(batch_size), int(seed), _ptr(lp), _ptr(lv), stream))
        return lp, lv

    def copy_state_from(self, other, stream=None):
        """variables + Adam slots + beta powers of `other` (same architecture, any device) into this network"""
        check(self.L.az_nn_copy_state(self.h, other.h, stream))

    def train_precision(self, precision):
        """FP32 (default, parity path) or BF16 (contractions as tcgen05 GEMMs)"""
        check(self.L.az_nn_train_precision(self.h, int(precision)))

    def layer(self, layer, which, n):
        """convolution output (which = 0) / activation (1) of tower layer `layer` from the last training step, [n, 7, 6, 256]"""
        a = np.empty((n, 7, 6, 256), np.float32)
        check(self.L.az_nn_train_get_layer(self.h, int(layer), int(which), _ptr(a), a.size))
        return a

    def grad(self, name, shape):
        a = np.empty(shape, np.float32)
        check(self.L.az_nn_train_get_grad(self.h, name.encode(), _ptr(a), a.size))
        return a

    def optimizer_slot(self, name, which, shape):
        a = np.empty(shape, np.float32)
        check(self.L.az_nn_optimizer_get(self.h, name.encode(), int(which), _ptr(a), a.size))
        return a

    def optimizer_powers(self):
        b1, b2, st = C.c_float(), C.c_float(), C.c_uint64()
        check(self.L.az_nn_optimizer_powers(self.h, C.byref(b1), C.byref(b2), C.byref(st)))
        return float(b1.value), float(b2.value), int(st.value)

    def save_checkpoint(self, prefix):
        check(self.L.az_nn_save_checkpoint(self.h, str(prefix).encode()))

    def load_checkpoint(self, prefix):
        check(self.L.az_nn_load_checkpoint(self.h, str(prefix).encode()))


class Checkpoint:
    """a TensorFlow V2 checkpoint bundle on the host (az_ckpt_*): <prefix>.index + <prefix>.data-00000-of-00001"""

    def __init__(self, prefix):
        self.L = lib()
        h = C.c_void_p()
        check(self.L.az_ckpt_open(str(prefix).encode(), C.byref(h)))
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.L.az_ckpt_close(self.h)
            self.h = None

    __del__ = close

    def tensors(self):
        """[(name, dtype, shape, bytes)] in table order"""
        out = []
        for i in range(self.L.az_ckpt_num_tensors(self.h)):
            name, dt, rank, shp, nb = C.c_char_p(), C.c_int(), C.c_int(), (C.c_int64 * 8)(), C.c_size_t()
            check(self.L.az_ckpt_tensor_info(self.h, i, C.byref(name), C.byref(dt), C.byref(rank), C.byref(shp), C.byref(nb)))
            out.append((name.value.decode(), int(dt.value), tuple(int(shp[k]) for k in range(rank.value)), int(nb.value)))
        return out

    def read(self, name):
        i = self.L.az_ckpt_find(self.h, name.encode())
        if i < 0:
            raise KeyError(name)
        _, dt, shape, nb = self.tensors()[i]
        a = np.empty(nb // 4, np.float32)
        check(self.L.az_ckpt_read(self.h, name.encode(), _ptr(a), nb))
        return a.reshape(shape)

    @staticmethod
    def write(prefix, tensors):
        """tensors: {name: float32 array}"""
        L = lib()
        names = list(tensors)
        arrs = [np.asarray(tensors[n], dtype=np.float32, order="C") for n in names]     # keeps scalars 0-d
        shapes = [(C.c_int64 * max(1, a.ndim))(*a.shape) for a in arrs]
        c_names = (C.c_char_p * len(names))(*[n.encode() for n in names])
        c_ranks = (C.c_int * len(names))(*[a.ndim for a in arrs])
        c_shapes = (C.POINTER(C.c_int64) * len(names))(*[C.cast(s, C.POINTER(C.c_int64)) for s in shapes])
        c_data = (C.c_void_p * len(names))(*[a.ctypes.data for a in arrs])
        check(L.az_ckpt_write(str(prefix).encode(), len(names), c_names, c_ranks, c_shapes, c_data))


EVAL_NN, EVAL_PSEUDO, EVAL_UNIFORM = 0, 1, 2
EVAL_PSEUDO6 = 3    # six-player search only: the pseudo evaluator with the six-seat value vector (include/az_pseudo_net.h)
OPPONENT_SCRIPT, OPPONENT_RANDOM, OPPONENT_ALPHAZERO = 1, 2, 3
SCRIPT_INIT = 0x00ffffff


class AzArenaResults(C.Structure):
    _fields_ = [("count", C.c_uint64), ("draw", C.c_uint64), ("win", C.c_uint64 * 2), ("win_and_started", C.c_uint64 * 2),
                ("az_moves", C.c_uint64), ("az_sims", C.c_uint64), ("az_evals", C.c_uint64), ("opponent_turns", C.c_uint64),
                ("ticks", C.c_uint64), ("errors", C.c_uint64)]

    def as_dict(self):
        return dict(count=int(self.count), draw=int(self.draw), win=[int(self.win[0]), int(self.win[1])],
                    win_and_started=[int(self.win_and_started[0]), int(self.win_and_started[1])], az_moves=int(self.az_moves),
                    az_sims=int(self.az_sims), az_evals=int(self.az_evals), opponent_turns=int(self.opponent_turns),
                    ticks=int(self.ticks), errors=int(self.errors))


class Arena:
    """`-m play` on the device: the Mcts handle's games as AlphaZero (player 0) vs a device-side opponent (player 1)"""

    def __init__(self, mcts, opponent=OPPONENT_SCRIPT, mirror_games=True, opponent_mcts=None):
        """opponent_mcts: a second Mcts over the same Env = AlphaZero vs AlphaZero (the trainer's comparison match, az_arena_create_versus)"""
        self.L, self.mcts, self.opponent_mcts = lib(), mcts, opponent_mcts
        h = C.c_void_p()
        if opponent_mcts is not None:
            check(self.L.az_arena_create_versus(mcts.h, opponent_mcts.h, int(mirror_games), C.byref(h)))
        else:
            check(self.L.az_arena_create(mcts.h, opponent, int(mirror_games), C.byref(h)))
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.L.az_arena_destroy(self.h)
            self.h = None

    __del__ = close

    def play(self, n_games, seed, stream=None):
        r = AzArenaResults()
        check(self.L.az_arena_play(self.h, int(n_games), int(seed), C.byref(r), stream))
        return r.as_dict()

SAMPLE_BYTES = 265


def write_samples_file(path, records):
    """NNTrainDataStorage::saveTrainingSamples file (az_samples_write_file)"""
    a = np.ascontiguousarray(records, np.uint8).reshape(-1, SAMPLE_BYTES)
    check(lib().az_samples_write_file(path.encode(), _ptr(a) if len(a) else None, C.c_size_t(len(a))))

PICK_ARGMAX, PICK_SELFPLAY = 0, 1


class Mcts:
    """one search tree per game of `env` (az_mcts_*); hyper-parameters come from env.rules"""

    def __init__(self, env, net=None, evaluator=EVAL_NN, precision=FP32):
        self.L = lib()
        self.env, self.net = env, net
        h = C.c_void_p()
        check(self.L.az_mcts_create(env.h, net.h if net is not None else None, evaluator, precision, C.byref(h)))
        self.h, self.n = h, env.n

    def close(self):
        if getattr(self, "h", None):
            self.L.az_mcts_destroy(self.h)
            self.h = None

    __del__ = close

    def simulations(self):
        return int(self.L.az_mcts_simulations(self.h))

    def clear(self, stream=None):
        check(self.L.az_mcts_clear(self.h, stream))

    def pool_stats(self, stream=None):
        """(peak nodes in any game's pool, nodes per pool, table bytes per game)"""
        a, b, c = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
        check(self.L.az_mcts_pool_stats(self.h, C.byref(a), C.byref(b), C.byref(c), stream))
        return int(a.value), int(b.value), int(c.value)

    def set_cohorts(self, cohorts):
        """0 = automatic, 1 = one stream, 2 = two game cohorts on two streams wherever possible (az_mcts_set_cohorts)"""
        check(self.L.az_mcts_set_cohorts(self.h, int(cohorts)))

    def search(self, pick_mode=PICK_ARGMAX, apply_move=False, extra_trim=None, stream=None):
        n = self.n
        N, pi = np.empty((n, MOVES), np.uint32), np.empty((n, MOVES), np.float32)
        mv, st = np.empty(n, np.uint8), np.empty(n, np.int8)
        et = None if extra_trim is None else np.ascontiguousarray(extra_trim, np.uint8)
        check(self.L.az_mcts_search(self.h, _ptr(et) if et is not None else None, pick_mode, int(apply_move),
                                    _ptr(N), _ptr(pi), _ptr(mv), _ptr(st), stream))
        return dict(N=N, pi=pi, move=mv, status=st)

    def root_stats(self, stream=None):
        n = self.n
        q, p = np.empty((n, MOVES), np.float32), np.empty((n, MOVES), np.float32)
        sumn, val, tab = np.empty(n, np.uint32), np.empty(n, np.float32), np.empty(n, np.int32)
        check(self.L.az_mcts_root_stats(self.h, _ptr(q), _ptr(p), _ptr(sumn), _ptr(val), _ptr(tab), stream))
        return dict(Q=q, P=p, sumN=sumn, value=val, table=tab)

    def selfplay(self, n_moves, stream=None):
        check(self.L.az_selfplay_run(self.h, int(n_moves), stream))

    def record(self, capacity_samples, max_moves_per_game=1024):
        """enable training-sample recording (az_selfplay_record)"""
        check(self.L.az_selfplay_record(self.h, C.c_size_t(int(capacity_samples)), int(max_moves_per_game)))

    def samples(self, stream=None):
        """finished-game samples as a [k, 265] uint8 array (reference file layout per record) and the dropped count"""
        n, dropped = C.c_size_t(0), C.c_uint64(0)
        check(self.L.az_selfplay_samples(self.h, None, C.c_size_t(0), C.byref(n), C.byref(dropped), stream))
        out = np.empty((n.value, SAMPLE_BYTES), np.uint8)
        if n.value:          # an empty queue was drained (and its dropped count reset) by the query itself
            check(self.L.az_selfplay_samples(self.h, _ptr(out), C.c_size_t(n.value), C.byref(n), C.byref(dropped), stream))
        return out[:n.value], int(dropped.value)

    def counters(self, reset=False, stream=None):
        c, err = AzCounters(), C.c_uint64(0)
        check(self.L.az_mcts_counters(self.h, C.byref(c), C.byref(err), int(reset), stream))
        d = c.as_dict()
        d["errors"] = int(err.value)
        return d


DIST_ID_BYTES = 128


class Dist:
    """the two cross-GPU exchanges over NCCL (az_dist_*): weight broadcast and statistics gather.

    Dist(devices=[0, 1, ...])                      one process drives several GPUs (the reference's model)
    Dist(world_size=N, rank=r, unique_id=b, device=d)   one process per GPU; rank 0 makes the id with Dist.unique_id()
    """

    def __init__(self, devices=None, world_size=None, rank=None, unique_id=None, device=0):
        self.L = lib()
        h = C.c_void_p()
        if world_size is None:
            devs = list(devices) if devices is not None else [0]
            arr = (C.c_int * len(devs))(*devs)
            check(self.L.az_dist_init(len(devs), arr, C.byref(h)))
        else:
            idb = np.frombuffer(bytes(unique_id), np.uint8).copy()
            assert idb.size == DIST_ID_BYTES
            check(self.L.az_dist_init_rank(int(world_size), int(rank), _ptr(idb), int(device), C.byref(h)))
        self.h = h

    @staticmethod
    def unique_id():
        out = np.zeros(DIST_ID_BYTES, np.uint8)
        check(lib().az_dist_unique_id(_ptr(out)))
        return out.tobytes()

    @staticmethod
    def nccl_version():
        v = C.c_int(0)
        check(lib().az_dist_nccl_version(C.byref(v)))
        return int(v.value)

    def close(self):
        if getattr(self, "h", None):
            self.L.az_dist_destroy(self.h)
            self.h = None

    __del__ = close

    def world_size(self):
        return int(self.L.az_dist_world_size(self.h))

    def local_count(self):
        return int(self.L.az_dist_local_count(self.h))

    def rank(self, local_index=0):
        return int(self.L.az_dist_rank(self.h, int(local_index)))

    def broadcast_weights(self, nets, root_rank=0):
        """nets: one Net per local member, in member order"""
        nets = list(nets)
        arr = (C.c_void_p * len(nets))(*[n.h for n in nets])
        check(self.L.az_dist_broadcast_weights(self.h, arr, len(nets), int(root_rank)))

    def gather_stats(self, local, per_rank=False):
        """local: uint64 [local_count, n] -> (sum [n], per-rank [world, n] or None)"""
        a = np.ascontiguousarray(local, np.uint64).reshape(self.local_count(), -1)
        n = a.shape[1]
        total = np.zeros(n, np.uint64)
        ranks = np.zeros((self.world_size(), n), np.uint64) if per_rank else None
        check(self.L.az_dist_gather_stats(self.h, _ptr(a), n, _ptr(total), _ptr(ranks) if per_rank else None))
        return total, ranks

    def gather_counters(self, counters):
        """counters: list of dicts as returned by Env.counters() / Mcts.counters(), one per local member -> summed dict"""
        loc = (AzCounters * len(counters))()
        for i, c in enumerate(counters):
            loc[i].steps, loc[i].games, loc[i].draws = c["steps"], c["games"], c["draws"]
            loc[i].wins[0], loc[i].wins[1] = c["wins"]
            loc[i].illegal, loc[i].sims, loc[i].evals, loc[i].path_nodes = c["illegal"], c["sims"], c["evals"], c.get("path_nodes", 0)
        tot = AzCounters()
        check(self.L.az_dist_gather_counters(self.h, loc, C.byref(tot)))
        return tot.as_dict()

    def gather_results(self, results):
        """results: list of Arena.play() dicts, one per local member -> GameResults::add over every rank"""
        loc = (AzArenaResults * len(results))()
        for i, r in enumerate(results):
            loc[i].count, loc[i].draw = r["count"], r["draw"]
            loc[i].win[0], loc[i].win[1] = r["win"]
            loc[i].win_and_started[0], loc[i].win_and_started[1] = r["win_and_started"]
            loc[i].az_moves, loc[i].az_sims, loc[i].az_evals = r["az_moves"], r["az_sims"], r["az_evals"]
            loc[i].opponent_turns, loc[i].ticks, loc[i].errors = r["opponent_turns"], r["ticks"], r["errors"]
        tot = AzArenaResults()
        check(self.L.az_dist_gather_results(self.h, loc, C.byref(tot)))
        return tot.as_dict()

    def barrier(self):
        check(self.L.az_dist_barrier(self.h))


ENV6_IMAGE_BYTES = 108
# six-player training record: image[108] | float value | float pi[43] | int8 final status | 3 zero bytes (include/az_b200.h)
SAMPLE6_BYTES = 288


class Env6:
    """n lockstep SIX-PLAYER games (az_env6_*): the configs[3] extension, rules = SIXPLAYER.md, no reference parity"""

    def __init__(self, n_games, rules=None, device=0, first_game_id=0):
        self.L = lib()
        self.n = int(n_games)
        self.rules = rules if rules is not None else default_rules()
        h = C.c_void_p()
        check(self.L.az_env6_create(self.n, C.byref(self.rules), device, first_game_id, C.byref(h)))
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.L.az_env6_destroy(self.h)
            self.h = None

    __del__ = close

    def reset(self, seed, stream=None):
        check(self.L.az_env6_reset(self.h, int(seed), stream))

    def rollout(self, n_steps, stream=None):
        check(self.L.az_env6_rollout(self.h, int(n_steps), stream))

    def last_kernel_ms(self):
        ms = C.c_float(0)
        check(self.L.az_env6_last_kernel_ms(self.h, C.byref(ms)))
        return float(ms.value)

    def step(self, action, stream=None):
        act = np.ascontiguousarray(action, np.uint8)
        assert act.shape == (self.n,)
        st = np.empty(self.n, np.int8)
        check(self.L.az_env6_step(self.h, _ptr(act), _ptr(st), stream))
        return st

    def query(self, stream=None):
        v, st = np.empty(self.n, np.uint64), np.empty(self.n, np.int8)
        check(self.L.az_env6_query(self.h, _ptr(v), _ptr(st), stream))
        return v, st

    def script_actions(self, stream=None):
        """the scripted agent's action (SIXPLAYER.md §5) for every game's position, uint8 [n]; 0xff for a finished game"""
        a = np.empty(self.n, np.uint8)
        check(self.L.az_env6_script_actions(self.h, _ptr(a), stream))
        return a

    def play(self, seat_kinds, n_plies, record_seats=0, stream=None):
        """n_plies plies of every game by scripted and uniform-random seats (az_env6_play, SIXPLAYER.md §6): seat_kinds[s] is None
        (the uniform-random player) or SCRIPT6; bit s of record_seats records the plies of seat s (record() first)"""
        kinds = list(seat_kinds)
        assert len(kinds) == 6, "seat_kinds needs six entries"
        for k in kinds:
            if k is not None and k is not SCRIPT6:
                raise AzError("a seat of Env6.play is None (the random player) or SCRIPT6, not %r" % (k,))
        ks = np.ascontiguousarray([AGENT6_SCRIPT if k is SCRIPT6 else AGENT6_RANDOM for k in kinds], np.int32)
        seats = int(record_seats)
        if not 0 <= seats < 64:                  # c_uint32 would wrap a larger value into range
            raise AzError("record_seats must be in 0..63, not %d" % seats)
        check(self.L.az_env6_play(self.h, _ptr(ks), C.c_uint32(seats), int(n_plies), stream))

    def record(self, capacity_samples, max_samples_per_game=4096):
        """enable recording in play() (az_env6_record).  Staging costs 112 bytes x max_samples_per_game per game on the device:
        about 7.5 GB for 16384 games at the default 4096; a game with more recorded plies is dropped whole and counted"""
        check(self.L.az_env6_record(self.h, C.c_size_t(int(capacity_samples)), int(max_samples_per_game)))

    def samples(self, stream=None):
        """records of the finished games of play() as a [k, SAMPLE6_BYTES] uint8 array and the dropped count (az_env6_samples)"""
        n, dropped = C.c_size_t(0), C.c_uint64(0)
        check(self.L.az_env6_samples(self.h, None, C.c_size_t(0), C.byref(n), C.byref(dropped), stream))
        out = np.empty((n.value, SAMPLE6_BYTES), np.uint8)
        if n.value:          # an empty queue was drained (and its dropped count reset) by the query itself
            check(self.L.az_env6_samples(self.h, _ptr(out), C.c_size_t(n.value), C.byref(n), C.byref(dropped), stream))
        return out[:n.value], int(dropped.value)

    def export(self, stream=None):
        a = np.empty((self.n, ENV6_IMAGE_BYTES), np.uint8)
        check(self.L.az_env6_export(self.h, _ptr(a), stream))
        return a

    def import_images(self, images, stream=None):
        a = np.ascontiguousarray(images, np.uint8)
        assert a.shape == (self.n, ENV6_IMAGE_BYTES)
        check(self.L.az_env6_import(self.h, _ptr(a), stream))

    def counters(self, reset=False, stream=None):
        c = AzCounters6()
        check(self.L.az_env6_counters(self.h, C.byref(c), int(reset), stream))
        return dict(steps=int(c.steps), games=int(c.games), draws=int(c.draws), wins=[int(c.wins[i]) for i in range(6)])

    def encode(self, planes=13, stream=None):
        """the network input of every game, [n, 7, 6, planes]: 13 = the two-player planes read for six seats, 16 = the seat planes"""
        a = np.empty((self.n, 7, 6, int(planes)), np.float32)
        check(self.L.az_env6_encode_planes(self.h, int(planes), _ptr(a), stream))
        return a


class Mcts6:
    """one search tree per six-player game of `env` (az_mcts6_*, SIXPLAYER.md); hyper-parameters come from env.rules"""

    def __init__(self, env, net=None, evaluator=0, precision=0):
        self.L, self.env, self.net, self.n = lib(), env, net, env.n
        h = C.c_void_p()
        check(self.L.az_mcts6_create(env.h, net.h if net is not None else None, evaluator, precision, C.byref(h)))
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.L.az_mcts6_destroy(self.h)
            self.h = None

    __del__ = close

    def search(self, pick_mode=0, apply_move=False, stream=None):
        n = self.n
        N, pi = np.empty((n, MOVES), np.uint32), np.empty((n, MOVES), np.float32)
        mv, st = np.empty(n, np.uint8), np.empty(n, np.int8)
        check(self.L.az_mcts6_search(self.h, pick_mode, int(apply_move), _ptr(N), _ptr(pi), _ptr(mv), _ptr(st), stream))
        return dict(N=N, pi=pi, move=mv, status=st)

    def root_stats(self, stream=None):
        n = self.n
        q, p = np.empty((n, MOVES), np.float32), np.empty((n, MOVES), np.float32)
        sumn, tab = np.empty(n, np.uint32), np.empty(n, np.int32)
        check(self.L.az_mcts6_root_stats(self.h, _ptr(q), _ptr(p), _ptr(sumn), _ptr(tab), stream))
        return dict(Q=q, P=p, sumN=sumn, table=tab)

    def selfplay(self, n_moves, stream=None):
        check(self.L.az_selfplay6_run(self.h, int(n_moves), stream))

    def record(self, capacity_samples, max_moves_per_game=4096):
        """enable training-sample recording (az_selfplay6_record) in selfplay() and search(apply_move=True).  Staging costs about
        288 bytes x max_moves_per_game per game on the device: roughly 19 GB for 16384 games at the default 4096.  Under
        uniform-random play a game with the default rules lasts 598 / 2690 / 3349 plies (min / median / max over 60 games), about
        415 with max_game_rounds = 20; a game longer than max_moves_per_game is dropped whole and counted."""
        check(self.L.az_selfplay6_record(self.h, C.c_size_t(int(capacity_samples)), int(max_moves_per_game)))

    def samples(self, stream=None):
        """finished-game samples as a [k, SAMPLE6_BYTES] uint8 array and the dropped count (az_selfplay6_samples)"""
        n, dropped = C.c_size_t(0), C.c_uint64(0)
        check(self.L.az_selfplay6_samples(self.h, None, C.c_size_t(0), C.byref(n), C.byref(dropped), stream))
        out = np.empty((n.value, SAMPLE6_BYTES), np.uint8)
        if n.value:          # an empty queue was drained (and its dropped count reset) by the query itself
            check(self.L.az_selfplay6_samples(self.h, _ptr(out), C.c_size_t(n.value), C.byref(n), C.byref(dropped), stream))
        return out[:n.value], int(dropped.value)

    def counters(self, reset=False, stream=None):
        c, sims, evals, errs = AzCounters6(), C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
        check(self.L.az_mcts6_counters(self.h, C.byref(c), C.byref(sims), C.byref(evals), C.byref(errs), int(reset), stream))
        return dict(steps=int(c.steps), games=int(c.games), draws=int(c.draws), wins=[int(c.wins[i]) for i in range(6)], sims=int(sims.value),
                    evals=int(evals.value), errors=int(errs.value))


class AzArena6Results(C.Structure):
    """mirror of az_arena6_results"""
    _fields_ = [("count", C.c_uint64), ("draw", C.c_uint64), ("win", C.c_uint64 * 6), ("win_seat", C.c_uint64 * 6),
                ("moves", C.c_uint64 * 6), ("sims", C.c_uint64), ("evals", C.c_uint64), ("ticks", C.c_uint64), ("errors", C.c_uint64)]

    def as_dict(self):
        return dict(count=int(self.count), draw=int(self.draw), win=[int(v) for v in self.win], win_seat=[int(v) for v in self.win_seat],
                    moves=[int(v) for v in self.moves], sims=int(self.sims), evals=int(self.evals), ticks=int(self.ticks),
                    errors=int(self.errors))


# agent kinds of az_arena6_create_agents (include/az_b200.h)
AGENT6_SEARCHER, AGENT6_RANDOM, AGENT6_SCRIPT = 0, 1, 2


class _Script6:
    def __repr__(self):
        return "SCRIPT6"


# the scripted six-player agent (SIXPLAYER.md §5) as an Arena6 agent, next to Mcts6 handles and None (the uniform-random player)
SCRIPT6 = _Script6()


class Arena6:
    """six-player matches on the device (az_arena6_*, SIXPLAYER.md §4): `agents` are Mcts6 handles over `env`, None (the
    uniform-random player) or SCRIPT6 (the scripted agent, SIXPLAYER.md §5), seat_agent[s] = the agent index that holds seat s;
    with rotate_seats the six games of a group share one deal and rotate the seats"""

    def __init__(self, env, agents, seat_agent, rotate_seats=True):
        self.L, self.env, self.agents = lib(), env, list(agents)
        kinds = [AGENT6_RANDOM if a is None else AGENT6_SCRIPT if a is SCRIPT6 else AGENT6_SEARCHER for a in self.agents]
        hs = (C.c_void_p * max(1, len(self.agents)))(*[a.h if k == AGENT6_SEARCHER else None for a, k in zip(self.agents, kinds)])
        ks = np.ascontiguousarray(kinds if kinds else [0], np.int32)
        seats = np.ascontiguousarray(seat_agent, np.uint8)
        assert seats.shape == (6,)
        h = C.c_void_p()
        check(self.L.az_arena6_create_agents(env.h, hs, _ptr(ks), len(self.agents), _ptr(seats), int(rotate_seats), C.byref(h)))
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.L.az_arena6_destroy(self.h)
            self.h = None

    __del__ = close

    def play(self, n_games, seed, first_game=0, stream=None):
        """match games first_game .. first_game + n_games - 1: the result tallies plus per-game `status` (winner seat or STATUS_DRAW)
        and `plies`"""
        r = AzArena6Results()
        st, pl = np.empty(int(n_games), np.int8), np.empty(int(n_games), np.uint32)
        check(self.L.az_arena6_play(self.h, int(first_game), int(n_games), int(seed), C.byref(r), _ptr(st), _ptr(pl), stream))
        out = r.as_dict()
        out.update(status=st, plies=pl)
        return out

    def active_slots(self):
        """slots that held a game at each tick of the last play()"""
        n = C.c_size_t(0)
        check(self.L.az_arena6_active_slots(self.h, None, C.c_size_t(0), C.byref(n)))
        out = np.empty(n.value, np.uint32)
        if n.value:
            check(self.L.az_arena6_active_slots(self.h, _ptr(out), C.c_size_t(n.value), C.byref(n)))
        return out
