"""ctypes binding of libmzb200.so (the C ABI in include/mzb200.h).

Fails loudly: if the shared library is missing or a CUDA device is not present the import /
``mz_create`` raises - there is NO CPU fallback anywhere in the product path.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmzb200.so")

MZ_MAX_LAYERS = 8
MZ_MAX_ACTIONS = 128
MZ_MEM_HOST, MZ_MEM_DEVICE = 0, 1
MZ_FLAG_KEEP_TREE, MZ_FLAG_STEPWISE, MZ_FLAG_CONTINUE = 1, 2, 4
MZ_EINVAL, MZ_EUNSUPPORTED, MZ_ESTATE = -1, -3, -4

_L = C.c_int32 * MZ_MAX_LAYERS


class MzNetDesc(C.Structure):
    _fields_ = [
        ("kind", C.c_int32), ("obs_c", C.c_int32), ("obs_h", C.c_int32), ("obs_w", C.c_int32),
        ("action_space", C.c_int32), ("support_size", C.c_int32), ("encoding", C.c_int32),
        ("n_fc_representation", C.c_int32), ("fc_representation", _L),
        ("n_fc_dynamics", C.c_int32), ("fc_dynamics", _L),
        ("n_fc_reward", C.c_int32), ("fc_reward", _L),
        ("n_fc_value", C.c_int32), ("fc_value", _L),
        ("n_fc_policy", C.c_int32), ("fc_policy", _L),
        ("blocks", C.c_int32), ("channels", C.c_int32),
        ("reduced_reward", C.c_int32), ("reduced_value", C.c_int32), ("reduced_policy", C.c_int32),
        ("n_res_fc_reward", C.c_int32), ("res_fc_reward", _L),
        ("n_res_fc_value", C.c_int32), ("res_fc_value", _L),
        ("n_res_fc_policy", C.c_int32), ("res_fc_policy", _L),
        ("downsample", C.c_int32),
    ]


class MzSearchDesc(C.Structure):
    _fields_ = [
        ("max_games", C.c_int32), ("num_simulations", C.c_int32), ("num_players", C.c_int32), ("extra_expansions", C.c_int32),
        ("discount", C.c_double), ("pb_c_base", C.c_double), ("pb_c_init", C.c_double),
        ("root_dirichlet_alpha", C.c_double), ("root_exploration_fraction", C.c_double),
        ("seed", C.c_uint64), ("pb_c_table", C.POINTER(C.c_double)), ("sqrt_table", C.POINTER(C.c_double)),
        ("ucb_table", C.POINTER(C.c_double)),
    ]


class MzTensor(C.Structure):
    _fields_ = [("name", C.c_char_p), ("data", C.c_void_p), ("numel", C.c_int64)]


class MzTrace(C.Structure):
    _fields_ = [("max_depth", C.c_int32), ("reserved", C.c_int32), ("depth", C.c_void_p), ("actions", C.c_void_p),
                ("value", C.c_void_p), ("reward", C.c_void_p), ("priors", C.c_void_p),
                ("root_priors_raw", C.c_void_p), ("root_reward", C.c_void_p), ("noise", C.c_void_p)]


class MzTeacher(C.Structure):
    _fields_ = [("root_value", C.c_void_p), ("root_reward", C.c_void_p), ("root_priors", C.c_void_p),
                ("value", C.c_void_p), ("reward", C.c_void_p), ("priors", C.c_void_p)]


class MzSearchIO(C.Structure):
    _fields_ = [
        ("n_games", C.c_int32), ("mem", C.c_int32),
        ("obs", C.c_void_p), ("legal_mask", C.c_void_p), ("to_play", C.c_void_p),
        ("add_exploration_noise", C.c_int32), ("flags", C.c_int32),
        ("noise", C.c_void_p), ("first_index", C.c_void_p), ("game_id", C.c_void_p), ("move_index", C.c_void_p),
        ("visit_counts", C.c_void_p), ("root_value", C.c_void_p), ("root_predicted_value", C.c_void_p),
        ("max_tree_depth", C.c_void_p), ("tie_count", C.c_void_p), ("root_priors", C.c_void_p),
        ("value_range", C.c_void_p),
        ("teacher", C.POINTER(MzTeacher)), ("trace", C.POINTER(MzTrace)),
    ]


class MzTreeExport(C.Structure):
    _fields_ = [("n_expansions", C.c_int32), ("child_visit", C.c_void_p), ("child_value_sum", C.c_void_p),
                ("child_reward", C.c_void_p), ("child_prior", C.c_void_p), ("child_expansion", C.c_void_p),
                ("hidden", C.c_void_p), ("root_visit", C.c_int32), ("root_value_sum", C.c_double),
                ("root_reward", C.c_float), ("reserved", C.c_int32)]


class MzInferenceOut(C.Structure):
    _fields_ = [("value_logits", C.c_void_p), ("reward_logits", C.c_void_p), ("policy_logits", C.c_void_p),
                ("hidden", C.c_void_p), ("value", C.c_void_p), ("reward", C.c_void_p)]


class MzSelfPlayDesc(C.Structure):
    _fields_ = [("env", C.c_int32), ("max_moves", C.c_int32), ("temperature_threshold", C.c_int32),
                ("reward_scale", C.c_int32), ("first_game_id", C.c_int64), ("game_id_stride", C.c_int64),
                ("td_steps", C.c_int32), ("reserved", C.c_int32), ("per_alpha", C.c_double), ("discount_pow", C.c_void_p),
                ("staging_bytes", C.c_uint64)]


class MzSelfPlayInject(C.Structure):
    _fields_ = [("forced_action", C.c_void_p), ("uniform", C.c_void_p), ("noise", C.c_void_p), ("first_index", C.c_void_p)]


class MzSelfPlayStats(C.Structure):
    _fields_ = [("env_steps", C.c_int64), ("games_finished", C.c_int64), ("staged_bytes", C.c_int64),
                ("staged_games", C.c_int32), ("parked_slots", C.c_int32), ("device_ms", C.c_double),
                ("staging_capacity", C.c_int64)]


class MzSelfPlayPeek(C.Structure):
    _fields_ = [("obs", C.c_void_p), ("legal_mask", C.c_void_p), ("to_play", C.c_void_p), ("game_id", C.c_void_p),
                ("move_index", C.c_void_p), ("last_action", C.c_void_p)]


MZ_ENV_CARTPOLE, MZ_ENV_TICTACTOE, MZ_ENV_CONNECT4 = 0, 1, 2
MZ_OPPONENT_SELF, MZ_OPPONENT_EXPERT, MZ_OPPONENT_RANDOM = 0, 1, 2
MZ_STAGED_HEADER_BYTES = 32

# every symbol include/mzb200.h declares: (name, restype, argtypes)
SYMBOLS = [
    ("mz_create", C.c_int, [C.POINTER(MzNetDesc), C.POINTER(MzSearchDesc), C.c_int, C.POINTER(C.c_void_p)]),
    ("mz_destroy", C.c_int, [C.c_void_p]),
    ("mz_last_error", C.c_char_p, [C.c_void_p]),
    ("mz_abi_version", C.c_int, []),
    ("mz_load_weights", C.c_int, [C.c_void_p, C.POINTER(MzTensor), C.c_int32]),
    ("mz_search", C.c_int, [C.c_void_p, C.POINTER(MzSearchIO)]),
    ("mz_initial_inference", C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.POINTER(MzInferenceOut)]),
    ("mz_recurrent_inference", C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.POINTER(MzInferenceOut)]),
    ("mz_export_tree", C.c_int, [C.c_void_p, C.c_int32, C.POINTER(MzTreeExport)]),
    ("mz_import_tree", C.c_int, [C.c_void_p, C.c_int32, C.POINTER(MzTreeExport)]),
    ("mz_hidden_elems", C.c_int64, [C.c_void_p]),
    ("mz_obs_elems", C.c_int64, [C.c_void_p]),
    ("mz_launch_count", C.c_int64, [C.c_void_p]),
    ("mz_graph_partitions", C.c_int32, [C.c_void_p]),
    ("mz_last_search_ms", C.c_double, [C.c_void_p]),
    ("mz_kernel_timing", C.c_int, [C.c_void_p, C.c_int32]),
    ("mz_kernel_times", C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    ("mz_numerics", C.c_char_p, [C.c_void_p]),
    ("mz_selfplay_begin", C.c_int, [C.c_void_p, C.POINTER(MzSelfPlayDesc)]),
    ("mz_selfplay_moves", C.c_int, [C.c_void_p, C.c_int32, C.c_double, C.POINTER(MzSelfPlayInject), C.POINTER(MzSelfPlayStats)]),
    ("mz_selfplay_enqueue", C.c_int, [C.c_void_p, C.c_int32, C.c_double]),
    ("mz_selfplay_wait", C.c_int, [C.c_void_p, C.POINTER(MzSelfPlayStats)]),
    ("mz_selfplay_drain", C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64), C.POINTER(C.c_int32),
                                    C.POINTER(C.c_void_p)]),
    ("mz_selfplay_peek", C.c_int, [C.c_void_p, C.POINTER(MzSelfPlayPeek)]),
    ("mz_selfplay_set_opponent", C.c_int, [C.c_void_p, C.c_int32, C.c_int32]),
    ("mz_debug_opponent_action", C.c_int, [C.c_int, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_void_p]),
    ("mz_debug_small_search_plan", C.c_int, [C.c_int32] * 10 + [C.POINTER(C.c_int64)]),
    ("mz_debug_conv3x3", C.c_int, [C.c_int, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
]

_lib = None


def load_library():
    """dlopen the in-tree library; raises with build instructions if it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing. Build it with `python -m muzero_general_b200.build` "
            "(nvcc, sm_100a). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, restype, argtypes in SYMBOLS:
        fn = getattr(lib, name)          # AttributeError if the ABI and the binary disagree
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


class MzError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"[mzb200 {code}] {message}")
        self.code = code
