// Device-resident self-play: the per-move loop of SelfPlay.play_game (self_play.py:110-183) for a whole batch.
//
//   move t:   [batched MCTS.run on the device-side observations]            mz_dispatch_search (fc_search.cu / pipeline.cu)
//             [select_action (self_play.py:222-245) + Game.step + record]   selfplay_step_kernel, lane 0 of the slot's warp
//             [finished games -> pinned host staging, slot restarts]        the same kernel, the whole warp
//
// Environments restated for the device (rules and observation planes of the reference):
//   CartPole   games/cartpole.py:131-174 wraps gym's CartPole-v1 (not vendored): Euler-integrated cart-pole, 20 ms step,
//              +1 reward per step, done at |x| > 2.4, |theta| > 12 deg or 500 steps; observation (1,1,4) fp32
//   TicTacToe  games/tictactoe.py:243-306; Connect4  games/connect4.py:220-305: planes [own stones of player +1,
//              stones of player -1, side to move (+1/-1)], player +1 = to_play 0 moves first, reward_scale for the mover
//              on completing a line, done on a line or a full board; Connect4 actions are columns (gravity)
// State per slot lives in HBM (a few dozen bytes); per-move records go to per-slot struct-of-arrays buffers
// [B][max_moves] and leave the device only when the game ends, as one packed block written by a warp straight into
// mapped pinned host memory (no per-move D2H, no host-side bookkeeping per move).
//
// Evaluation games (mz_selfplay_set_opponent): MuZero plays muzero_player's side, a hard-coded opponent (the expert
// scan of games/tictactoe.py:310-349 / games/connect4.py:307-348, or a uniformly random legal move) the other one.  Only
// MuZero's moves are searched: the opponent replies inside the same step-kernel pass, so every slot reaches the next
// batched search with MuZero to move.
//
// Random draws: Philox4x32-10 keyed by (seed, global game id, move): root noise and first-simulation ties inside the
// search (tree.cuh), the action sample here (tag kTagAction), CartPole's reset state (tag kTagReset), the opponent's
// default move (tag kTagOpponent).
#include <math.h>
#include <stdio.h>
#include <string.h>

#include "handle.h"
#include "common.cuh"

namespace mz {

constexpr uint32_t kTagReset = 0x7169E004u;
constexpr uint32_t kTagOpponent = 0x7169E005u;
constexpr int kMaxCells = 48;              // board cells per slot (Connect4: 42)

struct SpDev {
    int env, B, A, O, H, W, K, max_moves, threshold, reward_scale;
    int opponent, muzero_player;           // MZ_OPPONENT_*; the side MuZero plays when the opponent is not "self"
    uint64_t seed;
    int64_t id_stride;         // a slot's next game id = current + id_stride
    int td_steps;              // > 0: PER priorities are computed while packing (replay_buffer.py:33-51)
    double per_alpha;
    const double* discount_pow;   // [td_steps + 1] discount ** k as the caller's language evaluates it
    // environment state
    double* cart;              // [B][4]
    int* cart_steps;           // [B]
    int8_t* board;             // [B][kMaxCells], +1 / -1 / 0
    int8_t* player;            // [B] side to move, +1 / -1
    // search inputs / outputs (device)
    float* obs;                // [B][O]
    uint8_t* legal;            // [B][A]
    int32_t* to_play;          // [B]
    int64_t* game_id;          // [B]
    int32_t* move;             // [B] moves played in the current game
    int32_t* visits;           // [B][A]
    double* root_value;        // [B]
    // per-slot records of the game in flight
    double* rec_root;          // [B][T]
    int32_t* rec_visits;       // [B][T][A]
    int32_t* rec_action;       // [B][T]
    float* rec_reward;         // [B][T]
    int32_t* rec_to_play;      // [B][T]   (after the move)
    float* rec_obs;            // [B][T+1][O]
    int32_t* first_to_play;    // [B]
    int32_t* fin;              // [B] 0 = playing, T > 0 = finished after T moves, waiting to be packed
    int32_t* last_action;      // [B]
    // counters: [0] env_steps, [1] games_finished, [2] staging cursor (may run past the capacity), [3] staged games,
    //           [4] park events of this call, [5] end of the valid staged bytes
    unsigned long long* counters;
    unsigned char* staging;    // mapped pinned host memory
    unsigned long long staging_cap;
    unsigned long long* index; // mapped pinned host memory: per staged game {byte offset, (slot << 32) | length}
    // per-move overrides (device copies) or nullptr
    const int32_t* forced_action;
    const double* uniform;
    double temperature;
};

MZ_DEVINL double philox_uniform53(uint64_t seed, int64_t game, int move, uint32_t c2, uint32_t tag) {
    const Philox4 r = philox4x32_10((uint32_t)game, (uint32_t)move, c2, (uint32_t)((uint64_t)game >> 32),
                                    (uint32_t)seed, (uint32_t)(seed >> 32) ^ tag);
    // 53 random bits like numpy's random_sample: (a >> 5) * 2^26 + (b >> 6)
    return ((double)(r.x >> 5) * 67108864.0 + (double)(r.y >> 6)) * (1.0 / 9007199254740992.0);
}

// ------------------------------------------------------------------------------------------
// environments
// ------------------------------------------------------------------------------------------
constexpr double kGravity = 9.8, kMassCart = 1.0, kMassPole = 0.1, kHalfLen = 0.5, kForce = 10.0, kDt = 0.02;
constexpr double kXLimit = 2.4;
constexpr int kEpisodeCap = 500;

MZ_DEVINL void cartpole_reset(const SpDev& s, int g, int64_t gid) {
    double* st = s.cart + (size_t)g * 4;
    for (int k = 0; k < 4; ++k) {
        const double u = philox_uniform53(s.seed, gid, 0, (uint32_t)k, kTagReset);
        st[k] = -0.05 + 0.1 * u;                                   // uniform(-0.05, 0.05) like gym's reset
    }
    s.cart_steps[g] = 0;
}

MZ_DEVINL void cartpole_observe(const SpDev& s, int g, float* out) {
    const double* st = s.cart + (size_t)g * 4;
    for (int k = 0; k < 4; ++k) out[k] = (float)st[k];
}

// returns done; reward is always 1
MZ_DEVINL bool cartpole_step(const SpDev& s, int g, int action) {
    double* st = s.cart + (size_t)g * 4;
    const double x = st[0], xd = st[1], th = st[2], thd = st[3];
    const double force = action == 1 ? kForce : -kForce;
    const double c = cos(th), sn = sin(th);
    const double total = kMassCart + kMassPole, pml = kMassPole * kHalfLen;
    const double tmp = (force + pml * thd * thd * sn) / total;
    const double thacc = (kGravity * sn - c * tmp) / (kHalfLen * (4.0 / 3.0 - kMassPole * c * c / total));
    const double xacc = tmp - pml * thacc * c / total;
    st[0] = x + kDt * xd; st[1] = xd + kDt * xacc; st[2] = th + kDt * thd; st[3] = thd + kDt * thacc;
    const int steps = ++s.cart_steps[g];
    const double theta_limit = 12.0 * 2.0 * 3.141592653589793 / 360.0;
    return fabs(st[0]) > kXLimit || fabs(st[2]) > theta_limit || steps >= kEpisodeCap;
}

MZ_DEVINL void board_reset(const SpDev& s, int g) {
    int8_t* b = s.board + (size_t)g * kMaxCells;
    for (int i = 0; i < kMaxCells; ++i) b[i] = 0;
    s.player[g] = 1;
}

MZ_DEVINL void board_observe(const SpDev& s, int g, float* out) {
    const int8_t* b = s.board + (size_t)g * kMaxCells;
    const int cells = s.H * s.W;
    const float side = (float)s.player[g];
    for (int i = 0; i < cells; ++i) {
        out[i] = b[i] == 1 ? 1.0f : 0.0f;
        out[cells + i] = b[i] == -1 ? 1.0f : 0.0f;
        out[2 * cells + i] = side;
    }
}

MZ_DEVINL void board_legal(const SpDev& s, int g, uint8_t* legal) {
    const int8_t* b = s.board + (size_t)g * kMaxCells;
    if (s.env == MZ_ENV_CONNECT4) {
        for (int x = 0; x < s.W; ++x) legal[x] = b[(s.H - 1) * s.W + x] == 0;
    } else {
        for (int i = 0; i < s.H * s.W; ++i) legal[i] = b[i] == 0;
    }
}

// places the mover's stone, returns (won, done); the side to move flips
MZ_DEVINL void board_step(const SpDev& s, int g, int action, bool* won, bool* done) {
    int8_t* b = s.board + (size_t)g * kMaxCells;
    const int me = s.player[g];
    int y = -1, x = -1;
    if (s.env == MZ_ENV_CONNECT4) {
        x = action;
        for (int r = 0; r < s.H; ++r) if (b[r * s.W + x] == 0) { y = r; break; }   // lowest empty row; a full column changes nothing
    } else {
        y = action / s.W; x = action % s.W;
    }
    bool w = false;
    if (y >= 0) {
        b[y * s.W + x] = (int8_t)me;
        // a new line must pass through the new stone
        const int dirs[4][2] = {{0, 1}, {1, 0}, {1, 1}, {-1, 1}};
        for (int d = 0; d < 4 && !w; ++d) {
            int run = 1;
            for (int sgn = -1; sgn <= 1; sgn += 2)
                for (int i = 1; i < s.K; ++i) {
                    const int yy = y + sgn * i * dirs[d][0], xx = x + sgn * i * dirs[d][1];
                    if (yy < 0 || yy >= s.H || xx < 0 || xx >= s.W || b[yy * s.W + xx] != me) break;
                    ++run;
                }
            w = run >= s.K;
        }
    }
    bool any = false;
    if (s.env == MZ_ENV_CONNECT4) { for (int c = 0; c < s.W; ++c) any |= b[(s.H - 1) * s.W + c] == 0; }
    else { for (int i = 0; i < s.H * s.W; ++i) any |= b[i] == 0; }
    s.player[g] = (int8_t)(-me);
    *won = w;
    *done = w || !any;
}

// writes the search inputs of slot g from its environment state
MZ_DEVINL void publish(const SpDev& s, int g) {
    float* o = s.obs + (size_t)g * s.O;
    uint8_t* lg = s.legal + (size_t)g * s.A;
    if (s.env == MZ_ENV_CARTPOLE) {
        cartpole_observe(s, g, o);
        for (int k = 0; k < s.A; ++k) lg[k] = 1;
        s.to_play[g] = 0;
    } else {
        board_observe(s, g, o);
        board_legal(s, g, lg);
        s.to_play[g] = s.player[g] == 1 ? 0 : 1;
    }
}

MZ_DEVINL void start_game(const SpDev& s, int g, int64_t gid) {
    s.game_id[g] = gid;
    s.move[g] = 0;
    s.fin[g] = 0;
    s.last_action[g] = -1;
    if (s.env == MZ_ENV_CARTPOLE) cartpole_reset(s, g, gid); else board_reset(s, g);
    publish(s, g);
    s.first_to_play[g] = s.to_play[g];
    const float* o = s.obs + (size_t)g * s.O;
    float* r0 = s.rec_obs + (size_t)g * (s.max_moves + 1) * s.O;
    for (int i = 0; i < s.O; ++i) r0[i] = o[i];
}

__global__ void selfplay_reset_kernel(const SpDev s, int64_t first_game_id) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= s.B) return;
    start_game(s, g, first_game_id + g);
}

// ------------------------------------------------------------------------------------------
// select_action (self_play.py:222-245) on the visit counts of the search that just finished, then Game.step
// ------------------------------------------------------------------------------------------
MZ_DEVINL int sample_action(const SpDev& s, int g, double temperature, double u) {
    const int32_t* v = s.visits + (size_t)g * s.A;
    const uint8_t* lg = s.legal + (size_t)g * s.A;
    const int A = s.A;
    if (temperature == 0.0) {                                  // numpy.argmax: the first maximum in action order
        int best = -1, arg = 0;
        for (int k = 0; k < A; ++k) if (lg[k] && v[k] > best) { best = v[k]; arg = k; }
        return arg;
    }
    int n_legal = 0, last = 0;
    for (int k = 0; k < A; ++k) if (lg[k]) { ++n_legal; last = k; }
    if (isinf(temperature)) {                                  // numpy.random.choice(actions)
        int idx = (int)(u * n_legal);
        if (idx >= n_legal) idx = n_legal - 1;
        for (int k = 0; k < A; ++k) if (lg[k] && idx-- == 0) return k;
        return last;
    }
    // p = visit_counts ** (1 / T) / sum, then the first action whose cumulative probability exceeds u.
    // 1/T is 1, 2 or 4 for every reference schedule (games/*.py visit_softmax_temperature_fn): integer powers are exact
    const double inv = 1.0 / temperature;
    double total = 0.0;
    double p[MZ_MAX_ACTIONS];
    for (int k = 0; k < A; ++k) {
        double x = lg[k] ? (double)v[k] : 0.0;
        if (inv == 2.0) x = x * x;
        else if (inv == 4.0) { x = x * x; x = x * x; }
        else if (inv != 1.0) x = pow(x, inv);
        p[k] = x;
        total += x;
    }
    double cdf = 0.0;
    int pick = 0;
    for (int k = 0; k < A; ++k) {
        cdf = __dadd_rn(cdf, __ddiv_rn(p[k], total));
        if (u >= cdf) pick = k + 1;
    }
    return pick > last ? last : pick;                          // rounding can leave u >= cdf[-1]
}

// Game.step + record of the slot's next move (one thread).  searched: the move was chosen by the search that just
// finished (its root value and visit counts are recorded); otherwise it is an opponent's move: root value NaN, no visits
MZ_DEVINL void slot_play(const SpDev& s, int g, int action, bool searched) {
    const int t = s.move[g];
    float reward;
    bool done;
    if (s.env == MZ_ENV_CARTPOLE) {
        done = cartpole_step(s, g, action);
        reward = 1.0f;
    } else {
        bool won;
        board_step(s, g, action, &won, &done);
        reward = won ? (float)s.reward_scale : 0.0f;
    }
    // record of move t (store_search_statistics uses the pre-step root, self_play.py:169-175)
    const size_t r = (size_t)g * s.max_moves + t;
    s.rec_root[r] = searched ? s.root_value[g] : __longlong_as_double(0x7FF8000000000000ll);
    for (int k = 0; k < s.A; ++k) s.rec_visits[r * s.A + k] = searched ? s.visits[(size_t)g * s.A + k] : 0;
    s.rec_action[r] = action;
    s.rec_reward[r] = reward;
    publish(s, g);
    s.rec_to_play[r] = s.to_play[g];
    const float* o = s.obs + (size_t)g * s.O;
    float* ro = s.rec_obs + ((size_t)g * (s.max_moves + 1) + t + 1) * s.O;
    for (int i = 0; i < s.O; ++i) ro[i] = o[i];
    s.move[g] = t + 1;
    s.last_action[g] = action;
    if (done || t + 1 >= s.max_moves) s.fin[g] = t + 1;
}

// select_action + Game.step + record for slot g (one thread)
MZ_DEVINL void slot_act(const SpDev& s, int g) {
    const int t = s.move[g];
    const int64_t gid = s.game_id[g];
    int action = s.forced_action ? s.forced_action[g] : -1;
    if (action < 0) {
        const double T = (s.threshold == 0 || t + 1 < s.threshold) ? s.temperature : 0.0;
        const double u = s.uniform ? s.uniform[g] : philox_uniform53(s.seed, gid, t, 0u, kTagAction);
        action = sample_action(s, g, T, u);
    }
    slot_play(s, g, action, true);
}

// ------------------------------------------------------------------------------------------
// hard-coded opponents of evaluation games (SelfPlay.select_opponent_action, self_play.py:188-220), one warp per position
// board: H*W stones (+1 / -1 / 0, row 0 = the bottom row), player: side to move (+1 / -1); every lane returns the move
// ------------------------------------------------------------------------------------------
// numpy.random.choice(legal_actions()) with the uniform u: floor(u * n_legal) over the legal actions in ascending order
// (sample_action's T = inf rule); -1 when nothing is legal
MZ_DEVINL int random_action(const int8_t* board, int env, double u, int lane) {
    const bool c4 = env == MZ_ENV_CONNECT4;
    const int A = c4 ? 7 : 9;
    unsigned legal = __ballot_sync(0xffffffffu, lane < A && board[c4 ? 5 * 7 + lane : lane] == 0);
    const int n = __popc(legal);
    int idx = (int)(u * n);
    if (idx >= n) idx = n - 1;
    for (int i = 0; i < idx; ++i) legal &= legal - 1;
    return __ffs(legal) - 1;
}

// The expert (games/_boards.py::_threat_scan with tictactoe.py / connect4.py::_expert_windows): the reference walks its
// windows in order; a window whose stones sum to +-need has one gap, which becomes the candidate move if it is playable,
// and is played at once if the window belongs to the side to move (a win); a later qualifying window overwrites the
// candidate (a block); without one the random move is played.  Here lane L takes window 32c + L of chunk c: the first
// chunk with a win plays its lowest such lane, otherwise the highest qualifying lane of the last chunk that has one.
//   TicTacToe: 8 windows of 3 cells, need 2: row i then column i for i = 0..2, the diagonal, the anti-diagonal.
//   Connect4: 120 windows of 4 cells, need 3: for every 4x4 sub-board (k = 0..2 rows up, l = 0..3 columns right) row i
//   then column i for i = 0..3, the diagonal, the anti-diagonal.  A gap is playable only as the next free cell of its
//   column; a vertical window names its column without looking at the gap.
// The windows are index arithmetic rather than a table: a lookup per lane at 32 different addresses would serialise
// on the constant cache.
MZ_DEVINL int expert_action(const int8_t* board, int player, int env, double u, int lane) {
    const bool c4 = env == MZ_ENV_CONNECT4;
    const int H = c4 ? 6 : 3, W = c4 ? 7 : 3, len = c4 ? 4 : 3, need = c4 ? 3 : 2, n_windows = c4 ? 120 : 8;
    int height = 0;                                   // Connect4: stones in column `lane` = row of its next free cell
    if (c4 && lane < W)
        for (int y = 0; y < H; ++y) height += board[y * W + lane] != 0;
    int candidate = -1;
    for (int base = 0; base < n_windows; base += 32) {
        const int w = base + lane;
        int y0, x0, dy = 0, dx = 0, fixed = -1;        // cells (y0 + j * dy, x0 + j * dx), j < len
        if (c4) {
            const int k = w / 40, l = (w / 10) % 4, r = w % 10, i = r >> 1;
            if (r == 8) { y0 = k; x0 = l; dy = 1; dx = 1; }
            else if (r == 9) { y0 = k; x0 = l + 3; dy = 1; dx = -1; }
            else if (r & 1) { y0 = k; x0 = l + i; dy = 1; fixed = l + i; }
            else { y0 = k + i; x0 = l; dx = 1; }
        } else {
            const int i = w >> 1;
            if (w == 6) { y0 = 0; x0 = 0; dy = 1; dx = 1; }
            else if (w == 7) { y0 = 0; x0 = 2; dy = 1; dx = -1; }
            else if (w & 1) { y0 = 0; x0 = i; dy = 1; }
            else { y0 = i; x0 = 0; dx = 1; }
        }
        int sum = 0, gy = 0, gx = 0;
        if (w < n_windows)
            for (int j = 0; j < len; ++j) {
                const int y = y0 + j * dy, x = x0 + j * dx, v = board[y * W + x];
                sum += v;
                if (v == 0) { gy = y; gx = x; }
            }
        const int gap_height = c4 ? __shfl_sync(0xffffffffu, height, gx) : 0;
        const bool qualifies = w < n_windows && (sum == need || sum == -need) && (!c4 || fixed >= 0 || gap_height == gy);
        const int action = fixed >= 0 ? fixed : c4 ? gx : gy * W + gx;
        const unsigned wins = __ballot_sync(0xffffffffu, qualifies && player * sum > 0);
        if (wins) return __shfl_sync(0xffffffffu, action, __ffs(wins) - 1);
        const unsigned blocks = __ballot_sync(0xffffffffu, qualifies);
        if (blocks) candidate = __shfl_sync(0xffffffffu, action, 31 - __clz(blocks));
    }
    return candidate >= 0 ? candidate : random_action(board, env, u, lane);
}

MZ_DEVINL int opponent_action(const int8_t* board, int player, int env, int opponent, double u, int lane) {
    return opponent == MZ_OPPONENT_EXPERT ? expert_action(board, player, env, u, lane) : random_action(board, env, u, lane);
}

// the opponent's move in slot g: the whole warp chooses it, lane 0 steps and records it; returns fin[g] after the move.
// The caller has synchronised the warp after the slot's last write.
MZ_DEVINL int opponent_move(const SpDev& s, int g, int lane) {
    const double u = philox_uniform53(s.seed, s.game_id[g], s.move[g], 0u, kTagOpponent);
    const int action = opponent_action(s.board + (size_t)g * kMaxCells, s.player[g], s.env, s.opponent, u, lane);
    int T = 0;
    if (lane == 0) {
        slot_play(s, g, action, false);
        T = s.fin[g];
    }
    T = __shfl_sync(0xffffffffu, T, 0);
    __syncwarp();
    return T;
}

__host__ __device__ inline unsigned long long staged_block_bytes(int T, int A, int O) {
    unsigned long long b = MZ_STAGED_HEADER_BYTES;
    b += (unsigned long long)T * 8;                 // root_value
    b += (unsigned long long)T * A * 4;             // visit counts
    b += (unsigned long long)T * 4 * 4;             // action, reward, to_play, priority
    b += (unsigned long long)(T + 1) * O * 4;       // observations
    return (b + 7) & ~7ull;
}

// ReplayBuffer.save_game's initial priority of position i of the finished game in slot g (replay_buffer.py:39-51 with
// compute_target_value, :230-262), in the reference's operation order on fp64:
//   value = (+/-)root_value[i + td] * discount**td           if i + td < T, else 0
//   value += (+/-)reward_history[i + 1 + k] * discount**k    for k = 0 .. td - 1 while i + 1 + k <= T
//   priority = |root_value[i] - value| ** alpha
// reward_history[j + 1] = the reward of move j; to_play_history[0] = first_to_play, [j + 1] = to_play after move j.
MZ_DEVINL float initial_priority(const SpDev& s, int g, int T, int i) {
    const size_t r = (size_t)g * s.max_moves;
    auto to_play_hist = [&](int j) { return j == 0 ? s.first_to_play[g] : s.rec_to_play[r + j - 1]; };
    const int td = s.td_steps;
    const int me = to_play_hist(i);
    double value = 0.0;
    if (i + td < T) {
        const double last = to_play_hist(i + td) == me ? s.rec_root[r + i + td] : -s.rec_root[r + i + td];
        value = __dmul_rn(last, s.discount_pow[td]);
    }
    for (int k = 0; k < td && i + k < T; ++k) {
        const double rew = (double)s.rec_reward[r + i + k];
        const double signed_rew = to_play_hist(i + k) == me ? rew : -rew;
        value = __dadd_rn(value, __dmul_rn(signed_rew, s.discount_pow[k]));
    }
    const double d = fabs(__dsub_rn(s.rec_root[r + i], value));
    return (float)(s.per_alpha == 1.0 ? d : __dsqrt_rn(d));
}

// One warp per slot, 32 slots per CTA.  act != 0: lane 0 plays the slot's move (sampling, environment step, record)
// unless the slot is parked; then, whatever `act`, a finished game is copied into the staging area by the whole warp and
// the slot starts its next game (act == 0 is the drain-only pass that re-packs games parked by an earlier call).
// Staging space is reserved with ONE atomicAdd per finished game (a compare-and-swap loop serialises hundreds of
// finishing warps per move: 89 us per launch at 4096 CartPole games, profiles/r02_selfplay_loop.md): the cursor may run
// past the capacity, reservations that end beyond it are void (the game stays parked), and since the cursor only grows
// the valid reservations are a contiguous prefix whose end is tracked in counters[5].
// kOpponent (evaluation games): after MuZero's move the opponent replies in a game that goes on, and after a restart it
// opens the next game when MuZero plays second, so the next search sees MuZero to move in every slot.  Self-play runs
// the kOpponent = false instance, which has no opponent code.
constexpr int kStepThreads = 1024;

template <bool kOpponent>
__global__ void __launch_bounds__(kStepThreads) selfplay_step_kernel(const SpDev s, int act) {
    __shared__ int s_active;                         // moves played by this CTA
    if (threadIdx.x == 0) s_active = 0;
    __syncthreads();
    const int g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    int T = 0;
    if (g < s.B) {
        if (lane == 0) {
            T = s.fin[g];
            if (act && T == 0) {
                slot_act(s, g);
                atomicAdd(&s_active, 1);
                T = s.fin[g];
            }
        }
        T = __shfl_sync(0xffffffffu, T, 0);
        __syncwarp();
        if (kOpponent && act && T == 0) {            // MuZero moved and the game goes on (move + 1 < max_moves)
            T = opponent_move(s, g, lane);
            if (lane == 0) atomicAdd(&s_active, 1);
        }
    }
    if (T != 0) {
        const unsigned long long bytes = staged_block_bytes(T, s.A, s.O);
        unsigned long long off = 0;
        int ok = 0;
        if (lane == 0) {
            off = atomicAdd(&s.counters[2], bytes);
            ok = off + bytes <= s.staging_cap;
            if (ok) {
                atomicMax(&s.counters[5], off + bytes);
                atomicAdd(&s.counters[1], 1ull);
                const unsigned long long i = atomicAdd(&s.counters[3], 1ull);
                s.index[2 * i] = off;
                s.index[2 * i + 1] = ((unsigned long long)(unsigned)g << 32) | (unsigned)T;
            } else {
                atomicAdd(&s.counters[4], 1ull);
            }
        }
        ok = __shfl_sync(0xffffffffu, ok, 0);
        if (ok) {                                     // else parked: packed by a later call, after the host has drained
            off = ((unsigned long long)__shfl_sync(0xffffffffu, (unsigned)(off >> 32), 0) << 32) | __shfl_sync(0xffffffffu, (unsigned)off, 0);
            unsigned char* dst = s.staging + off;
            if (lane == 0) {
                *reinterpret_cast<int64_t*>(dst) = s.game_id[g];
                int32_t* hd = reinterpret_cast<int32_t*>(dst + 8);
                hd[0] = g; hd[1] = T; hd[2] = s.first_to_play[g]; hd[3] = s.O; hd[4] = s.A; hd[5] = (int32_t)bytes;
            }
            unsigned char* p = dst + MZ_STAGED_HEADER_BYTES;
            const size_t r = (size_t)g * s.max_moves;
            {
                double* d = reinterpret_cast<double*>(p);
                for (int i = lane; i < T; i += 32) d[i] = s.rec_root[r + i];
                p += (size_t)T * 8;
            }
            {
                int32_t* d = reinterpret_cast<int32_t*>(p);
                for (int i = lane; i < T * s.A; i += 32) d[i] = s.rec_visits[r * s.A + i];
                p += (size_t)T * s.A * 4;
                d = reinterpret_cast<int32_t*>(p);
                for (int i = lane; i < T; i += 32) d[i] = s.rec_action[r + i];
                p += (size_t)T * 4;
                float* f = reinterpret_cast<float*>(p);
                for (int i = lane; i < T; i += 32) f[i] = s.rec_reward[r + i];
                p += (size_t)T * 4;
                d = reinterpret_cast<int32_t*>(p);
                for (int i = lane; i < T; i += 32) d[i] = s.rec_to_play[r + i];
                p += (size_t)T * 4;
                f = reinterpret_cast<float*>(p);
                for (int i = lane; i < T; i += 32) f[i] = s.td_steps > 0 ? initial_priority(s, g, T, i) : 0.0f;
                p += (size_t)T * 4;
                f = reinterpret_cast<float*>(p);
                const float* src = s.rec_obs + (size_t)g * (s.max_moves + 1) * s.O;
                for (int i = lane; i < (T + 1) * s.O; i += 32) f[i] = src[i];
            }
            __syncwarp();
            if (lane == 0) start_game(s, g, s.game_id[g] + s.id_stride);
            if (kOpponent && s.muzero_player == 1) {  // the opponent plays move 0 of the slot's next game
                __syncwarp();
                opponent_move(s, g, lane);
                if (lane == 0) atomicAdd(&s_active, 1);
            }
        }
    }
    __syncthreads();
    if (threadIdx.x == 0 && s_active) atomicAdd(&s.counters[0], (unsigned long long)s_active);
}

static void launch_step(MzHandle* h, const SpDev& s, int act) {
    const int blocks = (s.B * 32 + kStepThreads - 1) / kStepThreads;
    if (s.opponent == MZ_OPPONENT_SELF) selfplay_step_kernel<false><<<blocks, kStepThreads, 0, h->stream>>>(s, act);
    else selfplay_step_kernel<true><<<blocks, kStepThreads, 0, h->stream>>>(s, act);
    h->launches += 1;
}

// move 0 of the games mz_selfplay_begin started, played by the opponent (one warp per slot)
__global__ void selfplay_open_kernel(const SpDev s) {
    const int g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (g >= s.B) return;
    opponent_move(s, g, lane);
    if (lane == 0) atomicAdd(&s.counters[0], 1ull);
}

__global__ void opponent_debug_kernel(int env, int opponent, int n, const int8_t* board, const int8_t* player,
                                      const double* uniform, int32_t* action) {
    const int p = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (p >= n) return;
    const int cells = env == MZ_ENV_CONNECT4 ? 42 : 9;
    const int a = opponent_action(board + (size_t)p * cells, player[p], env, opponent, uniform[p], lane);
    if (lane == 0) action[p] = a;
}

}  // namespace mz

using namespace mz;

struct MzSelfPlay {
    MzSelfPlayDesc desc{};
    SpDev dev{};
    std::vector<void*> allocs;
    // two staging areas (pinned + mapped) used alternately: while the host reads the games of call i, call i+1 writes the
    // other one, so the copy on the host overlaps the next moves on the device
    unsigned char* staging[2] = {nullptr, nullptr};
    unsigned long long* index[2] = {nullptr, nullptr};
    unsigned char* d_staging[2] = {nullptr, nullptr};       // device views of the same memory
    unsigned long long* d_index[2] = {nullptr, nullptr};
    int cur = 0;                               // area the next mz_selfplay_moves / enqueue writes
    bool in_flight = false;                    // moves enqueued, not waited for yet
    bool moves_played = false;                 // moves enqueued or opening moves played since mz_selfplay_begin
    unsigned long long* h_counters = nullptr;  // pinned copy of the counters
    int32_t* d_forced = nullptr;
    double* d_uniform = nullptr;
    double* d_noise = nullptr;
    int32_t* d_first = nullptr;
    uint64_t drained_bytes = 0;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
};

void mz_selfplay_destroy(MzHandle* h) {
    if (!h || !h->sp) return;
    MzSelfPlay* sp = h->sp;
    for (void* p : sp->allocs) cudaFree(p);
    for (int i = 0; i < 2; ++i) {
        if (sp->staging[i]) cudaFreeHost(sp->staging[i]);
        if (sp->index[i]) cudaFreeHost(sp->index[i]);
    }
    if (sp->h_counters) cudaFreeHost(sp->h_counters);
    if (sp->e0) cudaEventDestroy(sp->e0);
    if (sp->e1) cudaEventDestroy(sp->e1);
    delete sp;
    h->sp = nullptr;
}

template <typename T>
static bool sp_alloc(MzSelfPlay* sp, T** p, size_t count) {
    void* q = nullptr;
    if (cudaMalloc(&q, count * sizeof(T) + 16) != cudaSuccess) return false;
    cudaMemset(q, 0, count * sizeof(T) + 16);
    sp->allocs.push_back(q);
    *p = reinterpret_cast<T*>(q);
    return true;
}

extern "C" int mz_selfplay_begin(MzHandle* h, const MzSelfPlayDesc* d) {
    if (!h || !d) return fail(h, MZ_EINVAL, "mz_selfplay_begin: null argument");
    MZ_CUDA(h, cudaSetDevice(h->device));
    MZ_CUDA(h, cudaStreamSynchronize(h->stream));
    mz_selfplay_destroy(h);
    const int B = h->search.max_games, A = h->net.action_space, O = (int)h->obs_elems;
    int H = 1, W = 1, K = 0;
    switch (d->env) {
        case MZ_ENV_CARTPOLE: if (A != 2 || O != 4) return fail(h, MZ_EINVAL, "mz_selfplay_begin: CartPole needs 2 actions and a 4-value observation (stacked_observations must be 0)"); break;
        case MZ_ENV_TICTACTOE: H = 3; W = 3; K = 3; if (A != 9 || O != 27) return fail(h, MZ_EINVAL, "mz_selfplay_begin: TicTacToe needs 9 actions and a 3x3x3 observation (stacked_observations must be 0)"); break;
        case MZ_ENV_CONNECT4: H = 6; W = 7; K = 4; if (A != 7 || O != 126) return fail(h, MZ_EINVAL, "mz_selfplay_begin: Connect4 needs 7 actions and a 3x6x7 observation (stacked_observations must be 0)"); break;
        default: return fail(h, MZ_EUNSUPPORTED, "mz_selfplay_begin: unknown environment");
    }
    if (d->max_moves < 1) return fail(h, MZ_EINVAL, "mz_selfplay_begin: max_moves < 1");
    MzSelfPlay* sp = new (std::nothrow) MzSelfPlay();
    if (!sp) return fail(h, MZ_ENOMEM, "mz_selfplay_begin: out of host memory");
    h->sp = sp;
    sp->desc = *d;
    SpDev& s = sp->dev;
    s.env = d->env; s.B = B; s.A = A; s.O = O; s.H = H; s.W = W; s.K = K; s.max_moves = d->max_moves;
    s.threshold = d->temperature_threshold; s.reward_scale = d->reward_scale; s.seed = h->search.seed;
    s.id_stride = d->game_id_stride > 0 ? d->game_id_stride : B;
    s.td_steps = 0; s.per_alpha = 1.0; s.discount_pow = nullptr;
    if (d->td_steps > 0) {
        if (!d->discount_pow || !(d->per_alpha == 0.5 || d->per_alpha == 1.0)) {
            mz_selfplay_destroy(h);
            return fail(h, MZ_EUNSUPPORTED, "mz_selfplay_begin: device priorities need discount_pow and per_alpha of 0.5 or 1");
        }
        double* dp = nullptr;
        if (!sp_alloc(sp, &dp, (size_t)d->td_steps + 1)) { mz_selfplay_destroy(h); return fail(h, MZ_ENOMEM, "mz_selfplay_begin: out of device memory"); }
        MZ_CUDA(h, cudaMemcpy(dp, d->discount_pow, ((size_t)d->td_steps + 1) * 8, cudaMemcpyHostToDevice));
        s.td_steps = d->td_steps; s.per_alpha = d->per_alpha; s.discount_pow = dp;
    }
    const size_t T = (size_t)d->max_moves;
    bool ok = sp_alloc(sp, &s.cart, (size_t)B * 4) && sp_alloc(sp, &s.cart_steps, B) && sp_alloc(sp, &s.board, (size_t)B * kMaxCells) &&
              sp_alloc(sp, &s.player, B) && sp_alloc(sp, &s.obs, (size_t)B * O) && sp_alloc(sp, &s.legal, (size_t)B * A) &&
              sp_alloc(sp, &s.to_play, B) && sp_alloc(sp, &s.game_id, B) && sp_alloc(sp, &s.move, B) &&
              sp_alloc(sp, &s.visits, (size_t)B * A) && sp_alloc(sp, &s.root_value, B) && sp_alloc(sp, &s.rec_root, B * T) &&
              sp_alloc(sp, &s.rec_visits, B * T * A) && sp_alloc(sp, &s.rec_action, B * T) && sp_alloc(sp, &s.rec_reward, B * T) &&
              sp_alloc(sp, &s.rec_to_play, B * T) && sp_alloc(sp, &s.rec_obs, B * (T + 1) * O) && sp_alloc(sp, &s.first_to_play, B) &&
              sp_alloc(sp, &s.fin, B) && sp_alloc(sp, &s.last_action, B) && sp_alloc(sp, &s.counters, 8) &&
              sp_alloc(sp, &sp->d_forced, B) && sp_alloc(sp, &sp->d_uniform, B) && sp_alloc(sp, &sp->d_noise, (size_t)B * A) &&
              sp_alloc(sp, &sp->d_first, B);
    if (!ok) { mz_selfplay_destroy(h); return fail(h, MZ_ENOMEM, "mz_selfplay_begin: out of device memory"); }
    // staging (two areas of this size): by default 4x the room for every slot finishing a maximum-length game at once,
    // within [16, 64] MiB;
    // whatever the size, games that do not fit wait in their slots (parked) - nothing is dropped
    unsigned long long cap = d->staging_bytes;
    const unsigned long long worst = staged_block_bytes(d->max_moves, A, O) * (unsigned long long)B;
    if (cap == 0) {
        cap = 4 * worst;
        if (cap < (16ull << 20)) cap = 16ull << 20;
        if (cap > (64ull << 20)) cap = 64ull << 20;
        if (cap < staged_block_bytes(d->max_moves, A, O)) cap = staged_block_bytes(d->max_moves, A, O);
    }
    if (cap < staged_block_bytes(d->max_moves, A, O)) { mz_selfplay_destroy(h); return fail(h, MZ_EINVAL, "mz_selfplay_begin: staging_bytes smaller than one game"); }
    const unsigned long long index_entries = cap / staged_block_bytes(1, A, O) + 1;
    bool pinned = cudaHostAlloc(reinterpret_cast<void**>(&sp->h_counters), 64, cudaHostAllocDefault) == cudaSuccess;
    for (int i = 0; i < 2 && pinned; ++i)
        pinned = cudaHostAlloc(reinterpret_cast<void**>(&sp->staging[i]), cap, cudaHostAllocMapped) == cudaSuccess &&
                 cudaHostAlloc(reinterpret_cast<void**>(&sp->index[i]), index_entries * 16, cudaHostAllocMapped) == cudaSuccess;
    if (!pinned) {
        (void)cudaGetLastError();
        mz_selfplay_destroy(h);
        return fail(h, MZ_ENOMEM, "mz_selfplay_begin: pinned staging allocation failed");
    }
    memset(sp->h_counters, 0, 64);
    for (int i = 0; i < 2; ++i) {
        void* dptr = nullptr;
        if (cudaHostGetDevicePointer(&dptr, sp->staging[i], 0) != cudaSuccess) { mz_selfplay_destroy(h); return fail(h, MZ_ECUDA, "mz_selfplay_begin: staging is not device-mappable"); }
        sp->d_staging[i] = reinterpret_cast<unsigned char*>(dptr);
        if (cudaHostGetDevicePointer(&dptr, sp->index[i], 0) != cudaSuccess) { mz_selfplay_destroy(h); return fail(h, MZ_ECUDA, "mz_selfplay_begin: index is not device-mappable"); }
        sp->d_index[i] = reinterpret_cast<unsigned long long*>(dptr);
    }
    s.staging = sp->d_staging[0];
    s.index = sp->d_index[0];
    s.staging_cap = cap;
    cudaEventCreate(&sp->e0); cudaEventCreate(&sp->e1);
    selfplay_reset_kernel<<<(B + 127) / 128, 128, 0, h->stream>>>(s, d->first_game_id);
    h->launches += 1;
    MZ_CUDA(h, cudaGetLastError());
    MZ_CUDA(h, cudaStreamSynchronize(h->stream));
    return MZ_OK;
}

static int sp_read_counters(MzHandle* h, MzSelfPlayStats* stats, float ms) {
    MzSelfPlay* sp = h->sp;
    MZ_CUDA(h, cudaMemcpyAsync(sp->h_counters, sp->dev.counters, 48, cudaMemcpyDeviceToHost, h->stream));
    MZ_CUDA(h, cudaStreamSynchronize(h->stream));
    if (stats) {
        stats->env_steps = (int64_t)sp->h_counters[0];
        stats->games_finished = (int64_t)sp->h_counters[1];
        stats->staged_bytes = (int64_t)sp->h_counters[5];
        stats->staged_games = (int32_t)sp->h_counters[3];
        stats->parked_slots = (int32_t)sp->h_counters[4];
        stats->device_ms = ms;
        stats->staging_capacity = (int64_t)sp->dev.staging_cap;
    }
    return MZ_OK;
}

static int sp_enqueue(MzHandle* h, int32_t n_moves, double temperature, const MzSelfPlayInject* inj, const char* who) {
    if (!h || !h->sp) return fail(h, MZ_ESTATE, std::string(who) + ": call mz_selfplay_begin first");
    if (!h->weights_loaded) return fail(h, MZ_ESTATE, std::string(who) + ": weights not loaded");
    if (n_moves < 0) return fail(h, MZ_EINVAL, std::string(who) + ": n_moves < 0");
    if (inj && n_moves > 1 && (inj->forced_action || inj->uniform || inj->noise || inj->first_index))
        return fail(h, MZ_EINVAL, std::string(who) + ": per-move overrides need n_moves == 1");
    if (!(temperature >= 0.0)) return fail(h, MZ_EINVAL, std::string(who) + ": temperature must be >= 0");
    MzSelfPlay* sp = h->sp;
    if (sp->in_flight) return fail(h, MZ_ESTATE, std::string(who) + ": moves already enqueued, call mz_selfplay_wait first");
    MZ_CUDA(h, cudaSetDevice(h->device));
    SpDev s = sp->dev;
    s.staging = sp->d_staging[sp->cur];
    s.index = sp->d_index[sp->cur];
    const int B = s.B, A = s.A;
    s.temperature = temperature;
    s.forced_action = nullptr; s.uniform = nullptr;
    const double* noise = nullptr;
    const int32_t* first = nullptr;
    if (inj) {
        if (inj->forced_action) { MZ_CUDA(h, cudaMemcpyAsync(sp->d_forced, inj->forced_action, (size_t)B * 4, cudaMemcpyHostToDevice, h->stream)); s.forced_action = sp->d_forced; }
        if (inj->uniform) { MZ_CUDA(h, cudaMemcpyAsync(sp->d_uniform, inj->uniform, (size_t)B * 8, cudaMemcpyHostToDevice, h->stream)); s.uniform = sp->d_uniform; }
        if (inj->noise) { MZ_CUDA(h, cudaMemcpyAsync(sp->d_noise, inj->noise, (size_t)B * A * 8, cudaMemcpyHostToDevice, h->stream)); noise = sp->d_noise; }
        if (inj->first_index) { MZ_CUDA(h, cudaMemcpyAsync(sp->d_first, inj->first_index, (size_t)B * 4, cudaMemcpyHostToDevice, h->stream)); first = sp->d_first; }
    }
    if (sp->drained_bytes) {
        // the host has taken the staged games (and the areas were swapped): rewind the cursor; parked games are packed
        // by the first pass below
        MZ_CUDA(h, cudaMemsetAsync(s.counters + 2, 0, 16, h->stream));
        MZ_CUDA(h, cudaMemsetAsync(s.counters + 5, 0, 8, h->stream));
        sp->drained_bytes = 0;
    }
    SearchCall call{};
    call.n = B;
    call.obs = s.obs; call.legal_mask = s.legal; call.to_play = s.to_play;
    call.add_noise = 1; call.noise = noise; call.first_index = first;
    call.game_id = s.game_id; call.move_index = s.move;
    call.visit_counts = s.visits; call.root_value = s.root_value;
    sp->moves_played = true;
    MZ_CUDA(h, cudaEventRecord(sp->e0, h->stream));
    if (sp->h_counters[4]) launch_step(h, s, 0);      // games parked by the previous call first, so their slots play again
    MZ_CUDA(h, cudaMemsetAsync(s.counters + 4, 0, 8, h->stream));      // [4] = park events of THIS call
    for (int m = 0; m < n_moves; ++m) {
        int rc = mz_dispatch_search(h, call, false, false, 0);
        if (rc) return rc;
        launch_step(h, s, 1);
    }
    MZ_CUDA(h, cudaGetLastError());
    MZ_CUDA(h, cudaEventRecord(sp->e1, h->stream));
    sp->in_flight = true;
    return MZ_OK;
}

static int sp_wait(MzHandle* h, MzSelfPlayStats* stats) {
    MzSelfPlay* sp = h->sp;
    int rc = sp_read_counters(h, stats, 0.0f);
    if (rc) return rc;
    sp->in_flight = false;
    if (h->res && resnet_take_saturations(h->res, h->stream) > 0) {
        // the moves above searched with towers outside their accuracy contract (activations beyond the fp16 range are
        // carried with a saturated high part, not dropped); later calls use the fp32 towers
        mz_switch_to_strict(h);
    }
    float ms = 0.0f;
    if (cudaEventElapsedTime(&ms, sp->e0, sp->e1) == cudaSuccess && stats) stats->device_ms = ms;
    return MZ_OK;
}

extern "C" int mz_selfplay_moves(MzHandle* h, int32_t n_moves, double temperature, const MzSelfPlayInject* inj, MzSelfPlayStats* stats) {
    int rc = sp_enqueue(h, n_moves, temperature, inj, "mz_selfplay_moves");
    if (rc) return rc;
    return sp_wait(h, stats);
}

extern "C" int mz_selfplay_enqueue(MzHandle* h, int32_t n_moves, double temperature) {
    return sp_enqueue(h, n_moves, temperature, nullptr, "mz_selfplay_enqueue");
}

extern "C" int mz_selfplay_wait(MzHandle* h, MzSelfPlayStats* stats) {
    if (!h || !h->sp) return fail(h, MZ_ESTATE, "mz_selfplay_wait: call mz_selfplay_begin first");
    if (!h->sp->in_flight) return fail(h, MZ_ESTATE, "mz_selfplay_wait: nothing enqueued");
    MZ_CUDA(h, cudaSetDevice(h->device));
    return sp_wait(h, stats);
}

extern "C" int mz_selfplay_drain(MzHandle* h, const void** data, uint64_t* bytes, int32_t* n_games, const uint64_t** index) {
    if (!h || !h->sp || !data || !bytes || !n_games) return fail(h, MZ_EINVAL, "mz_selfplay_drain: bad argument");
    MzSelfPlay* sp = h->sp;
    if (sp->in_flight) return fail(h, MZ_ESTATE, "mz_selfplay_drain: moves in flight, call mz_selfplay_wait first");
    MZ_CUDA(h, cudaSetDevice(h->device));
    int rc = sp_read_counters(h, nullptr, 0.0f);
    if (rc) return rc;
    *data = sp->staging[sp->cur];
    if (index) *index = reinterpret_cast<const uint64_t*>(sp->index[sp->cur]);
    *bytes = sp->h_counters[5];
    *n_games = (int32_t)sp->h_counters[3];
    if (sp->h_counters[2]) {
        // the cursor moved (valid or void reservations): the next call rewinds it and writes the OTHER area, so what is
        // returned here stays intact while those moves run
        sp->drained_bytes = sp->h_counters[2];
        sp->cur ^= 1;
        sp->h_counters[2] = sp->h_counters[3] = sp->h_counters[5] = 0;     // a second drain before new moves returns nothing
    }
    return MZ_OK;
}

extern "C" int mz_selfplay_peek(MzHandle* h, const MzSelfPlayPeek* out) {
    if (!h || !h->sp || !out) return fail(h, MZ_EINVAL, "mz_selfplay_peek: bad argument");
    MZ_CUDA(h, cudaSetDevice(h->device));
    MZ_CUDA(h, cudaStreamSynchronize(h->stream));
    const SpDev& s = h->sp->dev;
    const size_t B = s.B;
    if (out->obs) MZ_CUDA(h, cudaMemcpy(out->obs, s.obs, B * s.O * 4, cudaMemcpyDeviceToHost));
    if (out->legal_mask) MZ_CUDA(h, cudaMemcpy(out->legal_mask, s.legal, B * s.A, cudaMemcpyDeviceToHost));
    if (out->to_play) MZ_CUDA(h, cudaMemcpy(out->to_play, s.to_play, B * 4, cudaMemcpyDeviceToHost));
    if (out->game_id) MZ_CUDA(h, cudaMemcpy(out->game_id, s.game_id, B * 8, cudaMemcpyDeviceToHost));
    if (out->move_index) MZ_CUDA(h, cudaMemcpy(out->move_index, s.move, B * 4, cudaMemcpyDeviceToHost));
    if (out->last_action) MZ_CUDA(h, cudaMemcpy(out->last_action, s.last_action, B * 4, cudaMemcpyDeviceToHost));
    return MZ_OK;
}

extern "C" int mz_selfplay_set_opponent(MzHandle* h, int32_t opponent, int32_t muzero_player) {
    if (!h || !h->sp) return fail(h, MZ_ESTATE, "mz_selfplay_set_opponent: call mz_selfplay_begin first");
    MzSelfPlay* sp = h->sp;
    SpDev& s = sp->dev;
    if (sp->moves_played) return fail(h, MZ_ESTATE, "mz_selfplay_set_opponent: moves already played, call mz_selfplay_begin first");
    if (opponent != MZ_OPPONENT_SELF && opponent != MZ_OPPONENT_EXPERT && opponent != MZ_OPPONENT_RANDOM)
        return fail(h, MZ_EINVAL, "mz_selfplay_set_opponent: unknown opponent");
    if (muzero_player != 0 && muzero_player != 1) return fail(h, MZ_EINVAL, "mz_selfplay_set_opponent: muzero_player must be 0 or 1");
    if (opponent != MZ_OPPONENT_SELF) {
        if (s.env == MZ_ENV_CARTPOLE) return fail(h, MZ_EINVAL, "mz_selfplay_set_opponent: CartPole has one player, its opponent is \"self\"");
        if (s.td_steps > 0)
            return fail(h, MZ_EINVAL, "mz_selfplay_set_opponent: evaluation games are not for the replay buffer, td_steps must be 0");
        if (s.max_moves < 2) return fail(h, MZ_EINVAL, "mz_selfplay_set_opponent: max_moves < 2 leaves no move to MuZero");
    }
    MZ_CUDA(h, cudaSetDevice(h->device));
    s.opponent = opponent;
    s.muzero_player = opponent == MZ_OPPONENT_SELF ? 0 : muzero_player;
    if (s.opponent != MZ_OPPONENT_SELF && s.muzero_player == 1) {
        selfplay_open_kernel<<<(s.B * 32 + 255) / 256, 256, 0, h->stream>>>(s);
        h->launches += 1;
        MZ_CUDA(h, cudaGetLastError());
        MZ_CUDA(h, cudaStreamSynchronize(h->stream));
        sp->moves_played = true;
    }
    return MZ_OK;
}

extern "C" int mz_debug_opponent_action(int device, int32_t env, int32_t opponent, int32_t n, const int8_t* board,
                                        const int8_t* player, const double* uniform, int32_t* action) {
    if (!board || !player || !uniform || !action || n < 0) return fail(nullptr, MZ_EINVAL, "mz_debug_opponent_action: bad argument");
    if (env != MZ_ENV_TICTACTOE && env != MZ_ENV_CONNECT4)
        return fail(nullptr, MZ_EINVAL, "mz_debug_opponent_action: env must be MZ_ENV_TICTACTOE or MZ_ENV_CONNECT4");
    if (opponent != MZ_OPPONENT_EXPERT && opponent != MZ_OPPONENT_RANDOM)
        return fail(nullptr, MZ_EINVAL, "mz_debug_opponent_action: opponent must be MZ_OPPONENT_EXPERT or MZ_OPPONENT_RANDOM");
    if (n == 0) return MZ_OK;
    if (cudaSetDevice(device) != cudaSuccess) return fail(nullptr, MZ_ECUDA, "mz_debug_opponent_action: no such device");
    const size_t cells = env == MZ_ENV_CONNECT4 ? 42 : 9;
    const size_t o_player = (size_t)n * cells, o_uniform = (o_player + n + 7) & ~(size_t)7, o_action = o_uniform + 8 * (size_t)n;
    unsigned char* d = nullptr;
    if (cudaMalloc(&d, o_action + 4 * (size_t)n) != cudaSuccess) return fail(nullptr, MZ_ENOMEM, "mz_debug_opponent_action: out of device memory");
    cudaError_t e = cudaMemcpy(d, board, o_player, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(d + o_player, player, n, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(d + o_uniform, uniform, 8 * (size_t)n, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        opponent_debug_kernel<<<(int)(((size_t)n * 32 + 255) / 256), 256>>>(
            env, opponent, n, reinterpret_cast<const int8_t*>(d), reinterpret_cast<const int8_t*>(d + o_player),
            reinterpret_cast<const double*>(d + o_uniform), reinterpret_cast<int32_t*>(d + o_action));
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpy(action, d + o_action, 4 * (size_t)n, cudaMemcpyDeviceToHost);
    cudaFree(d);
    if (e != cudaSuccess) return fail(nullptr, MZ_ECUDA, std::string("mz_debug_opponent_action: ") + cudaGetErrorString(e));
    return MZ_OK;
}
