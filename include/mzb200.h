/*
 * mzb200 - C ABI of the B200-native self-play search library (libmzb200.so).
 *
 * The reference (werner-duvaud/muzero-general) is pure Python and has no FFI; the drop-in
 * boundary is therefore the set of Python call sites listed next to each entry point below
 * (file:line in the reference).  A maintainer binds these symbols with ctypes
 * (see INTEGRATION.md and muzero_general_b200/_lib.py); nothing here mentions torch.
 *
 * Conventions
 *   - every function returns 0 on success, a negative MZ_E* code on failure; the message is
 *     available from mz_last_error(handle) (or mz_last_error(NULL) for mz_create failures);
 *     the library never aborts the process;
 *   - the caller owns every buffer passed in; the library borrows it for the duration of the
 *     call.  `mem` says whether the IO pointers of that call are HOST or DEVICE pointers
 *     (device = the handle's device).  Host buffers are staged through library-owned pinned
 *     memory, copies included in the call;
 *   - a handle is NOT thread-safe: one host thread per handle, one handle per GPU process
 *     (mirrors the reference's one-thread-per-actor model, self_play.py:11-29);
 *   - all library-owned scratch (node pool, hidden-state pool, staging) is allocated in
 *     mz_create, sized from max_games, num_simulations, action_space and the net shape.
 */
#ifndef MZB200_H
#define MZB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MZ_ABI_VERSION 2
#define MZ_MAX_LAYERS 8          /* hidden layers per MLP head */
#define MZ_MAX_ACTIONS 128       /* |action_space| supported by the tree kernels (one lane per action up to 32,
                                    four actions per lane above: csrc/tree_wide.cu) */

enum { MZ_OK = 0, MZ_EINVAL = -1, MZ_ECUDA = -2, MZ_EUNSUPPORTED = -3, MZ_ESTATE = -4, MZ_ENOMEM = -5 };
enum { MZ_NET_FC = 0, MZ_NET_RESNET = 1 };
enum { MZ_MEM_HOST = 0, MZ_MEM_DEVICE = 1 };

/* Shape of the networks built by models.MuZeroNetwork(config)  (models.py:7-41). */
typedef struct MzNetDesc {
    int32_t kind;                 /* MZ_NET_FC (models.py:80-195) or MZ_NET_RESNET (models.py:436-623) */
    int32_t obs_c, obs_h, obs_w;  /* stacked input: C*(s+1)+s channels, H, W (self_play.py:513-550) */
    int32_t action_space;         /* len(config.action_space); actions are 0..A-1 */
    int32_t support_size;         /* config.support_size; heads emit 2S+1 logits */
    /* fully connected */
    int32_t encoding;
    int32_t n_fc_representation, fc_representation[MZ_MAX_LAYERS];
    int32_t n_fc_dynamics, fc_dynamics[MZ_MAX_LAYERS];
    int32_t n_fc_reward, fc_reward[MZ_MAX_LAYERS];
    int32_t n_fc_value, fc_value[MZ_MAX_LAYERS];
    int32_t n_fc_policy, fc_policy[MZ_MAX_LAYERS];
    /* residual */
    int32_t blocks, channels;
    int32_t reduced_reward, reduced_value, reduced_policy;
    int32_t n_res_fc_reward, res_fc_reward[MZ_MAX_LAYERS];
    int32_t n_res_fc_value, res_fc_value[MZ_MAX_LAYERS];
    int32_t n_res_fc_policy, res_fc_policy[MZ_MAX_LAYERS];
    int32_t downsample;           /* 0 = none, 1 = "resnet" (models.py:233-275) */
} MzNetDesc;

/* The MuZeroConfig attributes MCTS reads (self_play.py:249-430). */
typedef struct MzSearchDesc {
    int32_t max_games;            /* capacity B: games searched in lockstep by one call */
    int32_t num_simulations;      /* config.num_simulations */
    int32_t num_players;          /* len(config.players); 1 or 2 (self_play.py:411-430) */
    int32_t extra_expansions;     /* node-pool room beyond num_simulations + 1 expansions per game, for searches that
                                     continue from an imported tree (override_root_with, self_play.py:275-277); the
                                     three tables below then have num_simulations + extra_expansions + 2 entries (per side) */
    double discount;              /* config.discount */
    double pb_c_base, pb_c_init;  /* self_play.py:384-390 */
    double root_dirichlet_alpha;  /* used only when noise is generated on the device */
    double root_exploration_fraction; /* self_play.py:476 */
    uint64_t seed;                /* key of the counter-based tie-break / noise stream */
    /* log((n+base+1)/base)+init and sqrt(n) for n = 0..num_simulations+1, computed by the
     * caller with the host language's libm so the device reproduces math.log / math.sqrt
     * (self_play.py:385-390) exactly.  NULL: the library computes them with C log()/sqrt(). */
    const double* pb_c_table;
    const double* sqrt_table;
    /* optional [(N+2) x (N+2)]: ucb_table[n_p*(N+2) + n_c] = pb_c_table[n_p] * (sqrt_table[n_p] / (n_c + 1)), i.e. the
     * exploration factor of self_play.py:384-390 with its two roundings, evaluated by the caller; saves two fp64
     * operations (one division) per child per tree level on the device.  NULL: computed on the device. */
    const double* ucb_table;
} MzSearchDesc;

/* One named tensor of the reference state_dict (models.py:69-73), fp32 host memory. */
typedef struct MzTensor {
    const char* name;             /* e.g. "dynamics_encoded_state_network.module.0.weight" */
    const float* data;
    int64_t numel;
} MzTensor;

/* Optional per-simulation record of what the device did (student forcing, SURVEY.md 8c). */
typedef struct MzTrace {
    int32_t max_depth;            /* D: entries kept per path */
    int32_t reserved;
    int32_t* depth;               /* [n, N]      number of select_child calls of simulation i */
    uint8_t* actions;             /* [n, N, D]   actions chosen root->leaf */
    float* value;                 /* [n, N]      scalarised value of the expanded leaf */
    float* reward;                /* [n, N]      scalarised reward of the expanded leaf */
    float* priors;                /* [n, N, A]   fp32 softmax priors of the expanded leaf */
    float* root_priors_raw;       /* [n, A]      root priors before noise (0 for illegal) */
    float* root_reward;           /* [n] */
    double* noise;                /* [n, A]      Dirichlet noise mixed into the root priors (given or device-drawn) */
} MzTrace;

/* Teacher forcing: bypass the networks, feed the tree these per-simulation outputs instead. */
typedef struct MzTeacher {
    const float* root_value;      /* [n] */
    const float* root_reward;     /* [n] */
    const float* root_priors;     /* [n, A] by action id (illegal entries ignored) */
    const float* value;           /* [n, N] */
    const float* reward;          /* [n, N] */
    const float* priors;          /* [n, N, A] */
} MzTeacher;

/* Arguments of one batched MCTS.run (self_play.py:260-361) over n games. */
typedef struct MzSearchIO {
    int32_t n_games;              /* <= max_games */
    int32_t mem;                  /* MZ_MEM_HOST or MZ_MEM_DEVICE for every pointer below */
    /* inputs */
    const float* obs;             /* [n, obs_c*obs_h*obs_w] fp32 (torch.tensor(obs).float(), self_play.py:281-282) */
    const uint8_t* legal_mask;    /* [n, A] non-zero = legal (self_play.py:296-308); NULL = all legal */
    const int32_t* to_play;       /* [n] game.to_play(); NULL = 0 */
    int32_t add_exploration_noise;/* self_play.py:310-314 */
    int32_t flags;                /* MZ_FLAG_* */
    const double* noise;          /* [n, A] Dirichlet draw by action id (host draws); NULL = drawn on the device
                                     (Philox + Marsaglia-Tsang gamma, root_dirichlet_alpha) */
    const int32_t* first_index;   /* [n] index into the legal list picked at the first simulation's
                                     all-way tie (self_play.py:371); NULL = device Philox */
    const int64_t* game_id;       /* [n] global game ids keying the Philox stream; NULL = 0..n-1 */
    const int32_t* move_index;    /* [n] move number keying the Philox stream; NULL = 0 */
    /* outputs (any may be NULL) */
    int32_t* visit_counts;        /* [n, A] child.visit_count by action id, 0 if illegal */
    double* root_value;           /* [n] root.value() (self_play.py:509) */
    float* root_predicted_value;  /* [n] mcts_info["root_predicted_value"] */
    int32_t* max_tree_depth;      /* [n] mcts_info["max_tree_depth"] */
    int32_t* tie_count;           /* [n] exact UCB ties met after the first simulation */
    double* root_priors;          /* [n, A] root priors after noise */
    double* value_range;          /* [n, 2] MinMaxStats minimum, maximum */
    const MzTeacher* teacher;     /* NULL = use the networks */
    const MzTrace* trace;         /* NULL = no trace */
} MzSearchIO;

#define MZ_FLAG_KEEP_TREE 1       /* leave the full tree in the HBM node pool for mz_export_tree */
#define MZ_FLAG_STEPWISE  2       /* force the generic select/infer/expand+backup pipeline */
#define MZ_FLAG_CONTINUE  4       /* MCTS.run(..., override_root_with=node), self_play.py:275-277: no root inference; the
                                     search runs num_simulations more simulations on the tree mz_import_tree put into the
                                     pool (n_games must be 1; fresh MinMaxStats; the root noise is mixed into the
                                     imported root priors).  obs is ignored. */

/* Full tree of one game after a search with MZ_FLAG_KEEP_TREE (host pointers). Slot layout:
 * expansion e (0 = root, e = i+1 for simulation i) owns child slots [e*A, e*A+A). */
typedef struct MzTreeExport {
    int32_t n_expansions;         /* out */
    int32_t* child_visit;         /* [(N+1)*A] */
    double* child_value_sum;      /* [(N+1)*A] */
    float* child_reward;          /* [(N+1)*A] */
    double* child_prior;          /* [(N+1)*A] */
    int32_t* child_expansion;     /* [(N+1)*A] expansion id of the child, -1 if not expanded */
    float* hidden;                /* [(N+1), hidden_elems] or NULL */
    int32_t root_visit;           /* out */
    double root_value_sum;        /* out */
    float root_reward;            /* out: reward of the root node (-0.0 for a fresh root; the child's reward after an import) */
    int32_t reserved;
} MzTreeExport;

/* Results of a batched network call, all DEVICE or all HOST per `mem`; any pointer may be NULL. */
typedef struct MzInferenceOut {
    float* value_logits;          /* [n, 2S+1] */
    float* reward_logits;         /* [n, 2S+1] */
    float* policy_logits;         /* [n, A] */
    float* hidden;                /* [n, hidden_elems] (rescaled state) */
    float* value;                 /* [n] support_to_scalar(value_logits)  (models.py:645-666) */
    float* reward;                /* [n] support_to_scalar(reward_logits) */
} MzInferenceOut;

typedef struct MzHandle MzHandle;

/* replaces SelfPlay.__init__ model construction (self_play.py:25-29) + MCTS(config) (self_play.py:257-258) */
int mz_create(const MzNetDesc* net, const MzSearchDesc* search, int device, MzHandle** out);
int mz_destroy(MzHandle* h);
const char* mz_last_error(const MzHandle* h);
int mz_abi_version(void);

/* replaces model.set_weights(state_dict) (models.py:72-73, self_play.py:27,37) */
int mz_load_weights(MzHandle* h, const MzTensor* tensors, int32_t n_tensors);

/* replaces MCTS.run for a batch of games (self_play.py:260-361; called from self_play.py:144-150) */
int mz_search(MzHandle* h, const MzSearchIO* io);

/* replaces model.initial_inference / recurrent_inference (models.py:172-195, 601-623) */
int mz_initial_inference(MzHandle* h, int32_t n, int32_t mem, const float* obs, const MzInferenceOut* out);
int mz_recurrent_inference(MzHandle* h, int32_t n, int32_t mem, const float* hidden, const int32_t* action,
                           const MzInferenceOut* out);

/* Node graph access for callers that walk the tree (self_play.py:229-232,499-509; diagnose_model.py:164,222-255) */
int mz_export_tree(MzHandle* h, int32_t game, MzTreeExport* out);
/* The inverse: seed game `game`'s tree in the pool from host arrays in the same layout (n_expansions, root_visit,
 * root_value_sum, root_reward are inputs; hidden = [n_expansions, hidden_elems] dense states, required unless the
 * search is teacher-forced).  Used by MCTS.run(override_root_with=...) followed by mz_search(MZ_FLAG_CONTINUE). */
int mz_import_tree(MzHandle* h, int32_t game, const MzTreeExport* tree);

/* sizes derived from the descriptors */
int64_t mz_hidden_elems(const MzHandle* h);
int64_t mz_obs_elems(const MzHandle* h);
/* number of kernels this handle has launched so far (bench.py's gpu_launches) */
int64_t mz_launch_count(const MzHandle* h);
/* parallel branches of the CUDA graph the step-wise search is replayed from: the simulations of disjoint game ranges
 * overlap (towers of one range with the heads / tree steps of the others); 1 = a single chain.  MZ_PARTS=1..4 overrides. */
int32_t mz_graph_partitions(const MzHandle* h);
/* device time of the search kernels of the last mz_search call, ms (CUDA events on the library stream) */
double mz_last_search_ms(const MzHandle* h);

/* Per-kernel-class device timing for the roofline line of bench.py.  While enabled (process-wide), the step-wise
 * pipeline runs launch by launch with a CUDA event pair around every kernel instead of replaying its CUDA graph.
 * mz_kernel_times synchronises and returns the accumulated milliseconds / launch counts since the last call:
 * [0] tree_step_kernel, [1] conv_tower_tc_kernel (tcgen05 towers, resident or streaming), [2] heads_kernel,
 * [3] conv3x3_kernel (CUDA cores, one conv per launch), [4] other, [5] small_tower_kernel (fused CUDA-core towers),
 * [6] small_search_kernel (small residual networks: all simulations of a search in one launch). */
#define MZ_KERNEL_CLASSES 7
int mz_kernel_timing(MzHandle* h, int32_t enable);
int mz_kernel_times(MzHandle* h, double* ms, int64_t* count);

/* Debug / tests (host only, no device needed): launch plan of the fused small-network search (csrc/small_search.cu) for a
 * hidden board H x W x C, |A| actions, n games on sm_count SMs, with tower_floats + heads_floats of weights and scratch_floats
 * of per-warp scratch in shared memory and cap_channels channels per activation buffer.  Returns 1 and fills
 * plan[8] = {P, CO, G, games per CTA, threads per CTA, shared-memory bytes, row stride, board stride}, or 0 when the shape
 * is not handled (the step-wise pipeline is used then). */
int mz_debug_small_search_plan(int32_t H, int32_t W, int32_t C, int32_t A, int32_t n, int32_t sm_count, int32_t tower_floats,
                               int32_t heads_floats, int32_t scratch_floats, int32_t cap_channels, int64_t* plan);

/* Debug / parity: one conv3x3 (C -> C, stride 1, pad 1; models.py:206-209) with optional bias, residual and
 * ReLU on host NCHW fp32 data, through the CUDA-core kernel (use_tensor_cores = 0) or the tcgen05 implicit
 * GEMM (C = 64, H <= 6, W <= 7): 1 = fp16 operands, 2 = split fp16+bf16 operands with three partial products
 * (fp32-grade, the default of the search path).  w is [C][C][3][3] as in the reference state_dict. */
int mz_debug_conv3x3(int device, int32_t n, int32_t C, int32_t H, int32_t W, const float* x, const float* w,
                     const float* bias, const float* residual, int32_t relu, int32_t use_tensor_cores, float* out);

/* Arithmetic the handle's search path computes in, e.g. "f32 nets + f64 tree statistics" (bench.py's dtype). */
const char* mz_numerics(const MzHandle* h);

/* ------------------------------------------------------------------------------------------------------------------
 * Device-resident self-play (SURVEY.md 8f-1): the per-move loop of SelfPlay.play_game (self_play.py:110-183) for
 * max_games environments whose state lives on the GPU.  One move = [batched MCTS.run on the device-side observations]
 * -> [visit-count sampling, self_play.py:222-245] -> [environment step] -> [one struct-of-arrays record per game].
 * A finished game (done, or max_moves reached, self_play.py:129-131) is packed into a pinned host staging area by the
 * kernel that detects it and its slot starts a new game with a fresh global id (old id + game_id_stride); the host reads
 * finished games only.  Root noise, the first simulation's tie and the action sample come from Philox4x32-10 streams
 * keyed (seed, game id, move), so a game's history does not depend on the batch or on the number of ranks.
 * Requires config.stacked_observations == 0 (the observation is the environment's own). */
enum { MZ_ENV_CARTPOLE = 0, MZ_ENV_TICTACTOE = 1, MZ_ENV_CONNECT4 = 2 };

typedef struct MzSelfPlayDesc {
    int32_t env;                  /* MZ_ENV_*: games/cartpole.py:131-174 (restated cart-pole physics),
                                     games/tictactoe.py:243-306, games/connect4.py:220-305 */
    int32_t max_moves;            /* config.max_moves */
    int32_t temperature_threshold;/* config.temperature_threshold, 0 = None (self_play.py:153-156) */
    int32_t reward_scale;         /* board games: reward of the winning move (tictactoe.py:144: 20, connect4.py:144: 10) */
    int64_t first_game_id;        /* slot g plays the global games first_game_id + g + k * game_id_stride, k = 0, 1, ... */
    int64_t game_id_stride;       /* 0 = max_games; world_size * max_games keeps ids unique across ranks */
    /* Initial prioritised-replay priorities |root_value - n-step target| ** PER_alpha of every position of a finished
     * game (ReplayBuffer.save_game + compute_target_value, replay_buffer.py:33-51,230-262), evaluated by the warp that packs
     * the game.  td_steps = 0: not computed.  discount_pow[k] = config.discount ** k for k = 0..td_steps, computed by the
     * caller (Python's own pow, so the products are the reference's); per_alpha must be 0.5 or 1 (an exact sqrt / identity). */
    int32_t td_steps;
    int32_t reserved;
    double per_alpha;
    const double* discount_pow;
    uint64_t staging_bytes;       /* capacity of the finished-game staging area, 0 = library default (4x the bytes of
                                     every slot finishing a maximum-length game at once, within [16 MiB, 64 MiB];
                                     the library keeps two such areas) */
} MzSelfPlayDesc;

/* Optional per-move overrides (HOST pointers, n = max_games; only with n_moves == 1).  Parity tests drive the
 * environments with recorded actions and replay the host loop's draws through them. */
typedef struct MzSelfPlayInject {
    const int32_t* forced_action; /* [n] play this action instead of sampling (entries < 0: sample) */
    const double* uniform;        /* [n] the uniform of the action sample instead of the Philox draw */
    const double* noise;          /* [n, A] root Dirichlet noise by action id instead of the device draw */
    const int32_t* first_index;   /* [n] first-simulation pick instead of the device draw */
} MzSelfPlayInject;

typedef struct MzSelfPlayStats {
    int64_t env_steps;            /* moves played since mz_selfplay_begin (all slots) */
    int64_t games_finished;       /* games packed into the staging area since mz_selfplay_begin */
    int64_t staged_bytes;         /* bytes waiting in the staging area */
    int32_t staged_games;         /* games waiting in the staging area */
    int32_t parked_slots;         /* times a finished game did not fit into the staging area during the last call
                                     (it waits in its slot and is staged after the next drain) */
    double device_ms;             /* device time of the last mz_selfplay_moves call */
    int64_t staging_capacity;     /* bytes the staging area holds (callers size their moves-per-call from it) */
} MzSelfPlayStats;

/* Current device-side view of the environments (HOST output pointers, any may be NULL). */
typedef struct MzSelfPlayPeek {
    float* obs;                   /* [n, obs_elems] observation the next search will see */
    uint8_t* legal_mask;          /* [n, A] */
    int32_t* to_play;             /* [n] */
    int64_t* game_id;             /* [n] */
    int32_t* move_index;          /* [n] moves played in the slot's current game */
    int32_t* last_action;         /* [n] action played by the last move (-1 before the first) */
} MzSelfPlayPeek;

/* Staged games are self-describing blocks laid out back to back (all little endian, 8-byte aligned):
 *   int64 game_id; int32 slot; int32 length T; int32 first_to_play; int32 obs_elems O; int32 actions A; int32 bytes;
 *   double root_value[T]; int32 visit_counts[T][A]; int32 action[T]; float reward[T]; int32 to_play[T] (after the move);
 *   float priority[T] (zeros unless td_steps > 0); float observation[T+1][O] (index 0 = reset observation); padding to 8.
 * = the fields of GameHistory (self_play.py:479-511) minus the dummy first entries.
 * A move of the hard-coded opponent (mz_selfplay_set_opponent) is recorded like any other move, with root_value NaN and
 * all visit counts 0 (a searched move always sums to num_simulations): the reference stores no search statistics for it
 * (store_search_statistics(None, ...), self_play.py:175,496-511). */
#define MZ_STAGED_HEADER_BYTES 32

/* replaces the per-move body of SelfPlay.play_game / continuous_self_play for a whole batch (self_play.py:31-183) */
int mz_selfplay_begin(MzHandle* h, const MzSelfPlayDesc* desc);
int mz_selfplay_moves(MzHandle* h, int32_t n_moves, double temperature, const MzSelfPlayInject* inject, MzSelfPlayStats* stats);
/* the same in two halves, so the host can work while the device plays: enqueue returns at once, wait synchronises */
int mz_selfplay_enqueue(MzHandle* h, int32_t n_moves, double temperature);
int mz_selfplay_wait(MzHandle* h, MzSelfPlayStats* stats);
/* pointer to the staged games (pinned host memory owned by the library) and marks them consumed.  The library keeps
 * two staging areas and swaps them here: the games returned stay intact during the NEXT mz_selfplay_moves / enqueue and
 * are overwritten by the one after the next drain.  `index` (may be NULL) receives a table of n_games pairs of uint64:
 * {byte offset of the game's block, (slot << 32) | length}, so a consumer can address any game without walking. */
int mz_selfplay_drain(MzHandle* h, const void** data, uint64_t* bytes, int32_t* n_games, const uint64_t** index);
int mz_selfplay_peek(MzHandle* h, const MzSelfPlayPeek* out);

/* Evaluation games (self_play.py:54-90, muzero.py:369-424): MuZero plays the side muzero_player, a hard-coded opponent the
 * other one.  MZ_OPPONENT_EXPERT = the reference's expert scan (games/tictactoe.py:310-349, games/connect4.py:307-348): a
 * move that completes a line of the side to move, else one that blocks the other side, else a uniformly random legal
 * move; MZ_OPPONENT_RANDOM = a uniformly random legal move.  The random move is floor(u * n_legal) over the legal
 * actions in ascending order with u a Philox uniform keyed (seed, game id, move) - numpy.random.choice's distribution,
 * not its stream.  Only MuZero's moves are searched: the opponent replies in the same move, so every search sees
 * MuZero to move; env_steps counts the moves of both sides.  Board games only (not CartPole), td_steps == 0,
 * max_moves >= 2.  MZ_OPPONENT_SELF (the default) is ordinary self-play. */
enum { MZ_OPPONENT_SELF = 0, MZ_OPPONENT_EXPERT = 1, MZ_OPPONENT_RANDOM = 2 };
/* after mz_selfplay_begin, before the first move; plays the opponent's opening move where it moves first */
int mz_selfplay_set_opponent(MzHandle* h, int32_t opponent, int32_t muzero_player);
/* the device expert / random policy on n given positions (board [n][H*W] int8 with values +1/-1/0, row 0 = the bottom
 * row, player [n] = +1/-1, uniform [n] = the default-move draw); one warp per position, same device function as the step
 * kernel.  action [n] receives the move (-1 for a position without a legal action). */
int mz_debug_opponent_action(int device, int32_t env, int32_t opponent, int32_t n, const int8_t* board,
                             const int8_t* player, const double* uniform, int32_t* action);

#ifdef __cplusplus
}
#endif
#endif /* MZB200_H */
