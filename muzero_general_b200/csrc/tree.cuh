// Tree arithmetic of one game, executed by a group of G lanes.
//
// Restates, for the device, the reference's per-simulation tree work:
//   select_child / ucb_score   self_play.py:363-404
//   Node.expand                self_play.py:451-465
//   add_exploration_noise      self_play.py:467-476
//   backpropagate              self_play.py:406-430
//   MinMaxStats                self_play.py:553-570
// All statistics are IEEE fp64 evaluated in the reference's operation order with explicit
// round-to-nearest intrinsics (never contracted into FMAs), so that visit counts, paths and
// root values are bit-identical to the Python implementation when the network outputs are
// the same (teacher / student forcing, tests/test_tree_parity_gpu.py).
//
// Storage (same layout in shared memory for the fused FC kernel and in the HBM node pool):
// expansion e (0 = root, e = i+1 for simulation i) owns the child slots [e*A, e*A+A);
// child k of a non-root expansion is action k; root children are indexed by action id and
// masked by the legal bitmask.  Per slot: visit i32, value_sum f64, reward f32, prior f32,
// expansion id i32 (-1 = leaf).  Root priors after noise are kept in fp64 separately
// (they are not fp32-representable, self_play.py:476).
#pragma once
#include "common.cuh"

namespace mz {

struct TreeConst {
    int A;                 // |action_space|
    int N;                 // num_simulations
    int P;                 // number of players (1 or 2)
    double discount;
    double noise_frac;     // root_exploration_fraction
    double noise_alpha;    // root_dirichlet_alpha (device-generated noise only)
    uint64_t seed;
    const double* pbc;     // [N+2]  log((n+base+1)/base)+init
    const double* sqrtn;   // [N+2]  sqrt(n)
    const double* ucb;     // [(N+2)^2] pbc[n_p] * (sqrtn[n_p] / (n_c + 1)) precomputed by the host, or nullptr
};

// Pointers to ONE game's tree (shared or global memory).
struct GameTree {
    int* visit;            // [(N+1)*A]
    double* vsum;          // [(N+1)*A]
    double* mval;          // [(N+1)*A] reward + discount * (+/-)(value_sum / visits), refreshed by every backup (see tree_backup)
    float* reward;         // [(N+1)*A]
    float* prior;          // [(N+1)*A]
    int* expansion;        // [(N+1)*A]
    double* root_prior;    // [A]
    int* path;             // [N+2] slots of the current simulation, path[0] = -1 (root)
    float* path_reward;    // [N+2] reward of every node on that path (the leaf's entry is filled at expansion)
    // scalars of the game
    int root_visit;
    double root_vsum;
    float root_reward;
    double lo, hi;         // MinMaxStats
    unsigned legal;        // bitmask of legal root actions
    int n_expanded;        // expansions so far (>= 1 after the root expansion)
    int ties;              // exact ties after the first simulation
};

struct Leaf {
    int depth;             // number of select_child calls
    int parent_exp;        // expansion id of the leaf's parent (its hidden state feeds dynamics)
    int action;            // action leading to the leaf
    int slot;              // child slot of the leaf
};

MZ_DEVINL double value_range_normalize(double v, double lo, double hi) {
    // MinMaxStats.normalize, self_play.py:566-570
    if (hi > lo) {
        // the node that set the lower bound has v == lo: a zero numerator would send the division down its out-of-line
        // slow path (and the whole warp with it); 0 / (hi - lo) is +0, so divide a harmless 1.0 and select
        const double d = __dsub_rn(v, lo);
        const double q = __ddiv_rn(d == 0.0 ? 1.0 : d, __dsub_rn(hi, lo));
        return d == 0.0 ? 0.0 : q;
    }
    return v;
}

// n-th (0-based) set bit of m
MZ_DEVINL int nth_set_bit(unsigned m, int n) { return (int)__fns(m, 0, n + 1); }

// ------------------------------------------------------------------------------------------
// Root: fp32 softmax over the legal logits, optional Dirichlet mixing.  (self_play.py:460-476)
// `logit` is this lane's policy logit (lane k <-> action k); returns this lane's fp32 prior.
// ------------------------------------------------------------------------------------------
template <int G>
MZ_DEVINL float group_softmax_masked(float logit, bool valid) {
    const float m = group_max_f32<G>(valid ? logit : -INFINITY);
    const float e = valid ? expf(logit - m) : 0.0f;
    const float s = group_sum_f32<G>(e);
    return div_pos_or_zero(e, s);          // masked lanes (e = 0) must not drag the warp through the division slow path
}

// the same over the first W lanes only (W = pow2 >= |A|, compile time): valid in lanes < W, same bits
template <int G, int W>
MZ_DEVINL float group_softmax_masked_w(float logit, bool valid) {
    const float m = group_max_f32_w<G, W>(valid ? logit : -INFINITY);
    const float e = valid ? expf(logit - m) : 0.0f;
    const float s = group_sum_f32_w<G, W>(e);
    return div_pos_or_zero(e, s);
}

template <int G>
MZ_DEVINL void tree_init_root(const TreeConst& c, GameTree& t, float prior_f32, float root_reward,
                              const double* noise /* [A] by action or nullptr */, bool generate_noise = false,
                              int64_t game_id = 0, int move = 0, double* noise_out = nullptr) {
    const int k = LaneGroup<G>::lane();
    const bool legal = (k < c.A) && ((t.legal >> k) & 1u);
    double nz = 0.0;
    bool have_noise = false;
    if (noise != nullptr) {
        nz = legal ? noise[k] : 0.0;
        have_noise = true;
    } else if (generate_noise) {
        // Dirichlet(alpha) over the legal actions = normalised Gamma(alpha) draws (numpy.random.dirichlet)
        const double gm = legal ? philox_gamma(c.seed, game_id, move, k, c.noise_alpha) : 0.0;
        double sum = gm;
        const unsigned m = LaneGroup<G>::mask();
        for (int off = G >> 1; off > 0; off >>= 1) sum += shfl_xor_f64(m, sum, off, G);
        nz = gm / sum;
        have_noise = true;
    }
    if (noise_out && k < c.A) noise_out[k] = nz;
    if (k < c.A) {
        double p = (double)prior_f32;
        if (legal && have_noise) {
            // prior * (1 - frac) + n * frac       (self_play.py:476)
            p = __dadd_rn(__dmul_rn(p, __dsub_rn(1.0, c.noise_frac)), __dmul_rn(nz, c.noise_frac));
        }
        t.root_prior[k] = legal ? p : 0.0;
        t.visit[k] = 0;
        t.vsum[k] = 0.0;
        t.reward[k] = 0.0f;
        t.prior[k] = legal ? prior_f32 : 0.0f;
        t.expansion[k] = -1;
    }
    t.root_visit = 0;
    t.root_vsum = 0.0;
    t.root_reward = root_reward;
    t.lo = INFINITY;
    t.hi = -INFINITY;
    t.n_expanded = 1;
    t.ties = 0;
    LaneGroup<G>::sync();
}

// ------------------------------------------------------------------------------------------
// Selection: descend from the root until an unexpanded child is reached.
// first_index >= 0: host-supplied pick (index into the tied list) for the all-way tie of the
// first simulation (self_play.py:371-377 with sqrt(0) = 0, see SURVEY.md appendix A.4).
// ------------------------------------------------------------------------------------------
// kPool: the tree lives in the HBM node pool (step-wise pipeline).  Every level is then exactly ONE round trip to
// L2: all fields of this lane's child (and the two table entries of the parent) are requested together, nothing
// is loaded conditionally on a value that has just arrived, and as soon as the child's expansion id is known the
// lines holding ITS children are prefetched into L1, overlapping the score arithmetic of the current level.
template <int G, bool kPool = false>
MZ_DEVINL Leaf tree_select(const TreeConst& c, GameTree& t, int sim, int64_t game_id, int move, int first_index) {
    const int k = LaneGroup<G>::lane();
    const int width = pow2_ceil(c.A);
    int e = 0;
    int n_parent = t.root_visit;
    int depth = 0;
    Leaf leaf;
    if (k == 0) { t.path[0] = -1; t.path_reward[0] = t.root_reward; }
    while (true) {
        const int base = e * c.A;
        const bool valid = (k < c.A) && (e != 0 || ((t.legal >> k) & 1u));
        double score = -INFINITY;
        int nc = 0, child_exp_k = -1;
        float reward_k = 0.0f;
        if (valid) {
            // one round of independent loads per level: everything this lane's child may need
            nc = t.visit[base + k];
            child_exp_k = t.expansion[base + k];
            const double pr = (e == 0) ? t.root_prior[k] : (double)t.prior[base + k];
            double mv = 0.0, tab_pbc = 0.0, tab_sqrt = 0.0;
            if (kPool) {
                reward_k = t.reward[base + k];
                mv = t.mval[base + k];
                tab_pbc = __ldg(c.pbc + n_parent);
                tab_sqrt = __ldg(c.sqrtn + n_parent);
                if (child_exp_k >= 0) {
                    const int nb = child_exp_k * c.A;
                    prefetch_l1(t.visit + nb); prefetch_l1(t.expansion + nb); prefetch_l1(t.prior + nb);
                    prefetch_l1(t.reward + nb); prefetch_l1(t.mval + nb);
                    prefetch_l1(t.mval + nb + c.A - 1);             // A doubles may straddle a line
                }
            }
            // pb_c = (log(...) + init) * (sqrt(n_p) / (n_c + 1))     self_play.py:384-390
            double pbc;
            if (kPool) {
                pbc = __dmul_rn(tab_pbc, __ddiv_rn(tab_sqrt, (double)(nc + 1)));
            } else if (c.ucb) {
                pbc = __ldg(c.ucb + n_parent * (c.N + 2) + nc);
            } else {
                const double q = __ddiv_rn(c.sqrtn[n_parent], (double)(nc + 1));
                pbc = __dmul_rn(c.pbc[n_parent], q);
            }
            score = __dmul_rn(pbc, pr);
            if (nc > 0) {
                // value_score = normalize(reward + discount * (+/-)mean)  (self_play.py:392-402).  The argument only changes
                // when a backup passes through the child, and the backup evaluates exactly this expression for the
                // min-max statistics: it is stored there (mval) and read back here, which takes an fp64 division and a
                // multiply-add off the per-level critical path without changing a bit.
                if (!kPool) reward_k = t.reward[base + k];
                const double v = value_range_normalize(kPool ? mv : t.mval[base + k], t.lo, t.hi);
                score = __dadd_rn(score, v);
            } else {
                reward_k = 0.0f;                   // (an unvisited child's stored reward is 0 anyway)
                score = __dadd_rn(score, 0.0);     // prior_score + 0
            }
        }
        const double best = group_max_f64<G>(score, width > G ? G : width);
        const unsigned tied = LaneGroup<G>::ballot(valid && score == best);
        const int n_tied = __popc(tied);
        int pick;
        if (n_tied <= 1) {
            pick = max(__ffs(tied) - 1, 0);        // n_tied == 0 only for a root without legal actions (rejected by the
                                                   // host; the clamp keeps the slot inside the game's pool regardless)
        } else {
            int idx;
            if (sim == 0 && depth == 0 && first_index >= 0) {
                idx = first_index < n_tied ? first_index : n_tied - 1;
            } else {
                idx = philox_tie_index(c.seed, game_id, move, sim, depth, n_tied);
                if (!(sim == 0 && depth == 0)) t.ties += 1;
            }
            pick = nth_set_bit(tied, idx);
        }
        const int slot = base + pick;
        depth += 1;
        // the picked child's fields come from the lane that scored it (no second round of loads)
        const int child_exp = LaneGroup<G>::bcast(child_exp_k, pick);
        const int child_visits = LaneGroup<G>::bcast(nc, pick);
        if (k == pick) { t.path[depth] = slot; t.path_reward[depth] = reward_k; }
        if (child_exp < 0) {
            leaf.depth = depth;
            leaf.parent_exp = e;
            leaf.action = pick;
            leaf.slot = slot;
            break;
        }
        n_parent = child_visits;
        e = child_exp;
    }
    LaneGroup<G>::sync();
    return leaf;
}

// ------------------------------------------------------------------------------------------
// Lookahead selection for |A| <= 2 (shared-memory trees): the same descent as tree_select, K levels per round.
// With sibling width W = 2 only 2 lanes of the group score a level; here level l of a round (l = 0..K-1) is scored by
// the 2^(l+1) lanes starting at lane 2^(l+1) - 2, one lane per grandchild path: lane local index j = 2*p + a scores child
// a of the node reached by the action bits of p (most significant = level 0).  K = 2 (G = 8), 3 (G = 16: lanes 0-1,
// 2-5, 6-13) or 4 (G = 32).  Every lane reaches its node by chasing at most K-1 expansion ids from the round's start
// and gives up (score -inf) below an unexpanded one.  Each score is the one tree_select would compute at that node
// (same loads, same operations, same order; the tree does not change during selection), so one xor-butterfly and one
// ballot serve all levels, and the path is resolved level by level as uniform integer work on the ballot: tie count,
// Philox tie draw with the true depth, tie counter on the resolved path only, and stop at the first unexpanded pick.
// The next round starts from the last pick.  Bit-identical to tree_select<G, false>; only unread scores are added.
// ------------------------------------------------------------------------------------------
template <int G>
constexpr int lookahead_levels() { return G >= 32 ? 4 : G >= 16 ? 3 : G >= 8 ? 2 : 1; }

template <int G>
MZ_DEVINL Leaf tree_select_lookahead(const TreeConst& c, GameTree& t, int sim, int64_t game_id, int move, int first_index) {
    constexpr int K = lookahead_levels<G>();
    static_assert(K >= 2, "lookahead needs at least two levels per round");
    const int k = LaneGroup<G>::lane();
    const int A = c.A;                                  // 1 or 2
    int e = 0;
    int n_parent = t.root_visit;
    int depth = 0;
    Leaf leaf;
    if (k == 0) { t.path[0] = -1; t.path_reward[0] = t.root_reward; }
    while (true) {
        // this lane's level l and local index j inside it: lanes [2^(l+1) - 2, 2^(l+2) - 2); unused lanes get l = K.
        // Recomputed every round from an opaque copy of the lane id: hoisted out of the simulation loop they would stay
        // live through the network evaluation, where the fixed-shape kernel has no register to spare.
        int kr = k;
        asm volatile("" : "+r"(kr));
        const int j = kr + 2 - (2 << (30 - __clz(kr + 2)));
        const int lvl = (kr < (2 << K) - 2 && (A == 2 || j == 0)) ? 30 - __clz(kr + 2) : K;   // |A| = 1: only action 0
        // 1. reach this lane's node (-1 if an ancestor is unexpanded): the ancestors' actions are the higher bits of j
        int node = lvl < K ? e : -1, np = n_parent;
#pragma unroll
        for (int i = 0; i < K - 1; ++i) {
            if (i < lvl && node >= 0) {
                const int s = node * A + ((j >> (lvl - i)) & 1);
                np = t.visit[s];
                node = t.expansion[s];
            }
        }
        // 2.-3. this lane's child: tree_select's score
        const int a_own = j & 1;
        const int slot_k = node * A + a_own;
        const bool root_level = (node == 0);            // only the round's level 0 can sit at the root
        const bool valid = node >= 0 && (!root_level || ((t.legal >> a_own) & 1u));
        double score = -INFINITY;
        int nc = 0, child_exp_k = -1;
        float reward_k = 0.0f;
        if (valid) {
            nc = t.visit[slot_k];
            child_exp_k = t.expansion[slot_k];
            const double pr = root_level ? t.root_prior[a_own] : (double)t.prior[slot_k];
            double pbc;
            if (c.ucb) {
                pbc = __ldg(c.ucb + np * (c.N + 2) + nc);
            } else {
                const double q = __ddiv_rn(c.sqrtn[np], (double)(nc + 1));
                pbc = __dmul_rn(c.pbc[np], q);
            }
            score = __dmul_rn(pbc, pr);
            if (nc > 0) {
                reward_k = t.reward[slot_k];
                const double v = value_range_normalize(t.mval[slot_k], t.lo, t.hi);
                score = __dadd_rn(score, v);
            } else {
                score = __dadd_rn(score, 0.0);
            }
        }
        // 4. sibling max of every level at once (siblings are lanes 2i, 2i+1), then one ballot for all levels
        const double best = fmax(score, shfl_xor_f64(LaneGroup<G>::mask(), score, 1, G));
        const unsigned tied = LaneGroup<G>::ballot(valid && score == best);
        const unsigned expanded = LaneGroup<G>::ballot(child_exp_k >= 0);
        // 5. resolve the path (uniform); the lane that scored a picked child writes its path entry
        int pl = 0;
        int p = 0;                                       // local index of the path node inside the next level
#pragma unroll
        for (int l = 0; l < K; ++l) {
            const int pair = (2 << l) - 2 + 2 * p;       // first lane of the sibling pair below the path node
            const unsigned tl = (tied >> pair) & 3u;
            const int n_tied = __popc(tl);
            int pick;
            if (n_tied <= 1) {
                pick = max(__ffs(tl) - 1, 0);
            } else {
                int idx;
                const int d = depth + l;
                if (sim == 0 && d == 0 && first_index >= 0) {
                    idx = first_index < n_tied ? first_index : n_tied - 1;
                } else {
                    idx = philox_tie_index(c.seed, game_id, move, sim, d, n_tied);
                    if (!(sim == 0 && d == 0)) t.ties += 1;
                }
                pick = nth_set_bit(tl, idx);
            }
            pl = pair + pick;
            if (k == pl) { t.path[depth + l + 1] = slot_k; t.path_reward[depth + l + 1] = reward_k; }
            if (!((expanded >> pl) & 1u)) break;
            p = 2 * p + pick;
        }
        // 6. continue below the last pick, or stop at it
        const int child_exp = LaneGroup<G>::bcast(child_exp_k, pl);
        const int child_visits = LaneGroup<G>::bcast(nc, pl);
        const int slot = LaneGroup<G>::bcast(slot_k, pl);
        depth += 31 - __clz(pl + 2);                     // levels resolved in this round: level of lane pl, plus one
        if (child_exp < 0) {
            leaf.depth = depth;
            leaf.parent_exp = (A == 2) ? (slot >> 1) : slot;
            leaf.action = (A == 2) ? (slot & 1) : 0;
            leaf.slot = slot;
            break;
        }
        n_parent = child_visits;
        e = child_exp;
    }
    LaneGroup<G>::sync();
    return leaf;
}

// ------------------------------------------------------------------------------------------
// Expansion of the selected leaf with the network outputs (self_play.py:345-351, 451-465).
// prior_f32: this lane's fp32 softmax prior (lane k <-> action k).
// ------------------------------------------------------------------------------------------
template <int G>
MZ_DEVINL int tree_expand(const TreeConst& c, GameTree& t, const Leaf& leaf, float reward, float prior_f32) {
    const int k = LaneGroup<G>::lane();
    const int e = t.n_expanded;
    if (k == 0) {
        t.expansion[leaf.slot] = e;
        t.reward[leaf.slot] = reward;
        t.path_reward[leaf.depth] = reward;
    }
    if (k < c.A) {
        const int s = e * c.A + k;
        t.visit[s] = 0;
        t.vsum[s] = 0.0;
        t.reward[s] = 0.0f;
        t.prior[s] = prior_f32;
        t.expansion[s] = -1;
    }
    t.n_expanded = e + 1;
    LaneGroup<G>::sync();
    return e;
}

// ------------------------------------------------------------------------------------------
// Backup along path[0..depth] (self_play.py:406-430).  The discounted value recurrence is a
// serial chain (2 fp64 ops per level, run redundantly by every lane); the per-node updates
// (value_sum, visit, running min/max) are independent: lane j updates node j, all at once, after
// the recurrence handed every lane the value its node saw.
// ------------------------------------------------------------------------------------------
template <int G>
MZ_DEVINL void tree_backup(const TreeConst& c, GameTree& t, const Leaf& leaf, float leaf_value) {
    const int k = LaneGroup<G>::lane();
    const int L = leaf.depth;                         // path indices 0..L
    double lo = INFINITY, hi = -INFINITY;
    double v = (double)leaf_value;                    // value seen by node j, starting at j = L
    double root_vsum = t.root_vsum;
    // lane j holds (slot, reward) of path node j when the path fits in the group: the serial recurrence
    // then runs on shuffles instead of a dependent chain of loads
    const bool packed = (L < G);
    int my_slot = -1;
    float my_reward = 0.0f;
    if (packed && k <= L) { my_slot = t.path[k]; my_reward = t.path_reward[k]; }
    if (packed) {
        // The recurrence runs on shuffles and every lane keeps the value its own node saw; the node updates then happen
        // ONCE, all lanes in parallel (a divergent owner block inside the loop would be issued L + 1 times, one lane each).
        double myv = 0.0;
        for (int j = L; j >= 0; --j) {
            const double r = (double)LaneGroup<G>::bcast(my_reward, j);
            const bool same = (c.P == 1) || (((L - j) & 1) == 0);
            if (j == k) myv = v;
            const double rr = (c.P == 1) ? r : (same ? -r : r);
            v = __dadd_rn(rr, __dmul_rn(c.discount, v));
        }
        if (k <= L) {
            const bool same = (c.P == 1) || (((L - k) & 1) == 0);
            const double add = same ? myv : -myv;
            double q;
            if (k == 0) {
                root_vsum = __dadd_rn(t.root_vsum, add);
                q = __ddiv_rn(root_vsum, (double)(t.root_visit + 1));
            } else {
                const double s = __dadd_rn(t.vsum[my_slot], add);
                const int n = t.visit[my_slot] + 1;
                t.vsum[my_slot] = s;
                t.visit[my_slot] = n;
                q = __ddiv_rn(s, (double)n);
            }
            const double m = __dadd_rn((double)my_reward, __dmul_rn(c.discount, (c.P == 1) ? q : -q));
            if (k > 0) t.mval[my_slot] = m;           // what the next selection will normalise for this child
            lo = m;
            hi = m;
        }
    } else {
    for (int j = L; j >= 0; --j) {
        const int slot = t.path[j];
        const float rf = t.path_reward[j];
        const double r = (double)rf;
        // node.to_play == to_play  <=>  (L - j) even (players alternate every level)
        const bool same = (c.P == 1) || (((L - j) & 1) == 0);
        if ((j % G) == k) {
            const double add = same ? v : -v;
            double q;
            if (j == 0) {
                root_vsum = __dadd_rn(t.root_vsum, add);
                q = __ddiv_rn(root_vsum, (double)(t.root_visit + 1));
            } else {
                const double s = __dadd_rn(t.vsum[slot], add);
                const int n = t.visit[slot] + 1;
                t.vsum[slot] = s;
                t.visit[slot] = n;
                q = __ddiv_rn(s, (double)n);
            }
            const double m = __dadd_rn(r, __dmul_rn(c.discount, (c.P == 1) ? q : -q));
            if (j > 0) t.mval[slot] = m;           // what the next selection will normalise for this child
            lo = fmin(lo, m);
            hi = fmax(hi, m);
        }
        // value = (same ? -reward : reward) + discount * value     (P == 2)
        // value = reward + discount * value                        (P == 1)
        const double rr = (c.P == 1) ? r : (same ? -r : r);
        v = __dadd_rn(rr, __dmul_rn(c.discount, v));
    }
    }
    // only lanes 0..L hold candidates: reduce over the smallest power of two covering them,
    // then broadcast lane 0's result (lanes beyond the reduced width hold partial values)
    const int width = (L + 1 >= G) ? G : pow2_ceil(L + 1);
    const unsigned gm = LaneGroup<G>::mask();
    if (width >= 2) {
        // minimum and maximum in ONE butterfly: after the first exchange the lower half of the `width` lanes carries minimum
        // candidates and the upper half maximum candidates (each lane sends the one it does not keep), the remaining steps
        // stay inside the halves; lane 0 ends with the minimum, lane width/2 with the maximum (exact: no rounding involved)
        const int half = width >> 1;
        const bool up = (k & half) != 0;
        const double got = shfl_xor_f64(gm, up ? lo : hi, half, G);
        double val = up ? fmax(hi, got) : fmin(lo, got);
        for (int off = half >> 1; off > 0; off >>= 1) {
            const double r = shfl_xor_f64(gm, val, off, G);
            val = up ? fmax(val, r) : fmin(val, r);
        }
        lo = shfl_f64(gm, val, 0, G);
        hi = shfl_f64(gm, val, half, G);
    } else {
        lo = shfl_f64(gm, lo, 0, G);
        hi = shfl_f64(gm, hi, 0, G);
    }
    root_vsum = shfl_f64(gm, root_vsum, 0, G);
    t.root_vsum = root_vsum;
    t.root_visit += 1;
    t.lo = fmin(t.lo, lo);
    t.hi = fmax(t.hi, hi);
    LaneGroup<G>::sync();
}

}  // namespace mz
