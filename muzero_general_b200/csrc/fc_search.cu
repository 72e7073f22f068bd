// Persistent fused search kernel for fully-connected MuZero networks.
//
// One launch runs the reference's whole MCTS.run (self_play.py:260-361) - root inference,
// root expansion + Dirichlet mixing, N x {select, recurrent inference, support_to_scalar,
// expand, backup} - for every game of the batch.  A group of G lanes owns one game from the
// first to the last simulation: its tree (child slots, hidden states, path) lives in shared
// memory next to the network weights, so the only HBM traffic is the observation in and
// the visit counts / root values out.  Groups never synchronise with each other; the grid
// is persistent (one wave) and groups stride over the games.
#include "fc_net.cuh"
#include "tree.cuh"
#include "kernels.h"

#include <stdlib.h>

namespace mz {

struct GameSmem {
    // byte offsets inside one game's region
    int vsum, mval, root_prior, visit, expansion, reward, prior, path, path_reward, hidden, act, bytes;
};

__host__ __device__ inline GameSmem game_smem_layout(int N, int A, int E, int maxw, bool keep_hidden) {
    GameSmem L;
    const int S = (N + 1) * A;
    const int Epad = (E + 3) & ~3;
    int off = 0;
    auto take = [&](int bytes) { int o = off; off = (off + bytes + 15) & ~15; return o; };
    L.vsum = take(S * 8);
    L.mval = take(S * 8);
    L.root_prior = take(A * 8);
    L.visit = take(S * 4);
    L.expansion = take(S * 4);
    L.reward = take(S * 4);
    L.prior = take(S * 4);
    L.path = take((N + 2) * 4);
    L.path_reward = take((N + 2) * 4);
    L.hidden = take((keep_hidden ? (N + 1) * Epad : 0) * 4);
    L.act = take(9 * maxw * 4);        // s0 s1 s2 + three heads x (ping, pong)
    off += 16;          // odd multiple of 16 B between games: spreads games over banks
    L.bytes = off;
    return L;
}

// SH: FcFixedShape<E, H, S, A> runs the per-simulation network call through the fully unrolled fixed-shape code
// (fc_net.cuh::fc_recurrent_fixed, bit-identical to the generic descriptors walk), FcGenericShape through the latter.
template <int G, bool kTeacher, typename SH>
__global__ void __launch_bounds__(kFcMaxThreads) fc_search_kernel(const __grid_constant__ FcSearchArgs a) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int N = a.N, A = a.A;
    // ---- CTA-shared: tables + weights
    double* s_pbc = reinterpret_cast<double*>(smem);
    double* s_sqrt = s_pbc + (N + 2);
    float* s_blob = reinterpret_cast<float*>(s_sqrt + (N + 2));
    for (int i = threadIdx.x; i < N + 2; i += blockDim.x) { s_pbc[i] = a.pbc[i]; s_sqrt[i] = a.sqrtn[i]; }
    if (!kTeacher)
        for (int i = threadIdx.x; i < a.net.blob_floats; i += blockDim.x) s_blob[i] = a.blob[i];
    __syncthreads();

    const int shared_bytes = ((2 * (N + 2) * 8 + (kTeacher ? 0 : a.net.blob_floats) * 4) + 15) & ~15;
    const GameSmem L = game_smem_layout(N, A, a.net.E, a.net.maxw, !kTeacher);
    const int groups_per_cta = blockDim.x / G;
    const int gi = threadIdx.x / G;
    const int lane = LaneGroup<G>::lane();
    unsigned char* mine = smem + shared_bytes + (size_t)gi * L.bytes;

    TreeConst c;
    c.A = A; c.N = N; c.P = a.P; c.discount = a.discount; c.noise_frac = a.noise_frac; c.noise_alpha = a.noise_alpha; c.seed = a.seed;
    c.pbc = s_pbc; c.sqrtn = s_sqrt; c.ucb = a.ucb;

    GameTree t;
    t.vsum = reinterpret_cast<double*>(mine + L.vsum);
    t.mval = reinterpret_cast<double*>(mine + L.mval);
    t.root_prior = reinterpret_cast<double*>(mine + L.root_prior);
    t.visit = reinterpret_cast<int*>(mine + L.visit);
    t.expansion = reinterpret_cast<int*>(mine + L.expansion);
    t.reward = reinterpret_cast<float*>(mine + L.reward);
    t.prior = reinterpret_cast<float*>(mine + L.prior);
    t.path = reinterpret_cast<int*>(mine + L.path);
    t.path_reward = reinterpret_cast<float*>(mine + L.path_reward);
    float* s_hidden = reinterpret_cast<float*>(mine + L.hidden);
    float* s_act = reinterpret_cast<float*>(mine + L.act);
    const int E = a.net.E, F = a.net.F, S = a.net.S, maxw = a.net.maxw;
    const int Epad = (E + 3) & ~3;
    float* s0 = s_act;
    float* s1 = s_act + maxw;
    float* s2 = s_act + 2 * maxw;
    float* const hb[3][2] = {{s_act + 3 * maxw, s_act + 4 * maxw}, {s_act + 5 * maxw, s_act + 6 * maxw},
                             {s_act + 7 * maxw, s_act + 8 * maxw}};
    const bool fused_heads = (a.net.rew.n == a.net.pol.n) && (a.net.pol.n == a.net.val.n);

    for (int g = blockIdx.x * groups_per_cta + gi; g < a.n_games; g += gridDim.x * groups_per_cta) {
        const int64_t game_id = a.game_id ? a.game_id[g] : (int64_t)g;
        const int move = a.move_index ? a.move_index[g] : 0;
        const int to_play0 = a.to_play ? a.to_play[g] : 0;
        const int first_index = a.first_index ? a.first_index[g] : -1;
        unsigned legal = 0;
        for (int k = 0; k < A; ++k) legal |= (a.legal_mask == nullptr || a.legal_mask[(size_t)g * A + k]) ? (1u << k) : 0u;
        t.legal = legal;
        (void)to_play0;

        // ------------------------------------------------------------------ root
        float root_value, root_reward, logit = 0.0f;
        if (kTeacher) {
            root_value = a.teacher.root_value[g];
            root_reward = a.teacher.root_reward[g];
        } else {
            // representation (models.py:133-145) -> hidden[0]
            load_vector<G>(a.obs + (size_t)g * a.net.obs_elems, s1, a.net.obs_elems);
            float* raw = mlp_forward<G>(a.net.rep, s_blob, s1, s0, s1, s2);
            rescale_unit_range<G>(raw, s_hidden, E);
            // prediction (models.py:128-131)
            float* pol = mlp_forward<G>(a.net.pol, s_blob, s_hidden, s0, s1, s2);
            logit = (lane < A) ? pol[lane] : 0.0f;
            LaneGroup<G>::sync();
            float* val = mlp_forward<G>(a.net.val, s_blob, s_hidden, s0, s1, s2);
            root_value = support_to_scalar_group<G>(val, S);
            LaneGroup<G>::sync();
            root_reward = inverse_value_transform(0.0f);     // log(one-hot centre), models.py:176-183
        }
        float prior;
        if (kTeacher) prior = (lane < A) ? a.teacher.root_priors[(size_t)g * A + lane] : 0.0f;
        else prior = group_softmax_masked<G>(logit, lane < A && ((legal >> lane) & 1u));
        if (a.trace.root_priors_raw && lane < A) a.trace.root_priors_raw[(size_t)g * A + lane] = ((legal >> lane) & 1u) ? prior : 0.0f;
        if (a.trace.root_reward && lane == 0) a.trace.root_reward[g] = root_reward;
        tree_init_root<G>(c, t, prior, root_reward,
                          (a.add_noise && a.noise) ? a.noise + (size_t)g * A : nullptr, a.add_noise && !a.noise,
                          game_id, move, a.trace.noise ? a.trace.noise + (size_t)g * A : nullptr);

        // ------------------------------------------------------------------ simulations
        int max_depth = 0;
        for (int sim = 0; sim < N; ++sim) {
            Leaf leaf;
            if constexpr (lookahead_levels<G>() >= 2) {
                if (a.lookahead) leaf = tree_select_lookahead<G>(c, t, sim, game_id, move, first_index);
                else leaf = tree_select<G>(c, t, sim, game_id, move, first_index);
            } else {
                leaf = tree_select<G>(c, t, sim, game_id, move, first_index);
            }
            float value, reward;
            if (kTeacher) {
                value = a.teacher.value[(size_t)g * N + sim];
                reward = a.teacher.reward[(size_t)g * N + sim];
                prior = (lane < A) ? a.teacher.priors[((size_t)g * N + sim) * A + lane] : 0.0f;
            } else {
                // dynamics (models.py:147-170)
                const float* h = s_hidden + (size_t)leaf.parent_exp * Epad;
                float* hn = s_hidden + (size_t)t.n_expanded * Epad;
                if constexpr (SH::kEnabled) {
                    fc_recurrent_fixed<G, SH>(a.net, s_blob, h, leaf.action, hn, s0, s1, hb[0][0], hb[1][0], hb[2][0], logit, value, reward);
                } else {
                float* raw = mlp_forward<G>(a.net.dyn, s_blob, h, s0, s1, s2, leaf.action);
                if (fused_heads) {
                    // rescale first, then reward (raw state), policy and value (rescaled state) side by side
                    rescale_unit_range<G>(raw, hn, E);
                    const MlpDesc* const ds[3] = {&a.net.rew, &a.net.pol, &a.net.val};
                    const float* const xs[3] = {raw, hn, hn};
                    float* outs[3];
                    mlp_forward_multi<G, 3>(ds, s_blob, xs, hb, outs);
                    logit = (lane < A) ? outs[1][lane] : 0.0f;
                    support_to_scalar_group2<G>(outs[2], outs[0], S, value, reward);
                    LaneGroup<G>::sync();
                } else {
                    // reward head reads the un-normalised next state
                    float* rl = mlp_forward<G>(a.net.rew, s_blob, raw, s0, s1, nullptr);
                    reward = support_to_scalar_group<G>(rl, S);
                    LaneGroup<G>::sync();
                    rescale_unit_range<G>(raw, hn, E);
                    float* pol = mlp_forward<G>(a.net.pol, s_blob, hn, s0, s1, s2);
                    logit = (lane < A) ? pol[lane] : 0.0f;
                    LaneGroup<G>::sync();
                    float* vl = mlp_forward<G>(a.net.val, s_blob, hn, s0, s1, s2);
                    value = support_to_scalar_group<G>(vl, S);
                    LaneGroup<G>::sync();
                }
                }
                if constexpr (SH::kEnabled) prior = group_softmax_masked_w<G, pow2_ceil_c(SH::A)>(logit, lane < A);
                else prior = group_softmax_masked<G>(logit, lane < A);
            }
            if (a.trace.depth) {
                const size_t ti = (size_t)g * N + sim;
                if (lane == 0) { a.trace.depth[ti] = leaf.depth; a.trace.value[ti] = value; a.trace.reward[ti] = reward; }
                if (lane < A) a.trace.priors[ti * A + lane] = prior;
                for (int j = lane; j < leaf.depth && j < a.trace.max_depth; j += G)
                    a.trace.actions[ti * a.trace.max_depth + j] = (uint8_t)(t.path[j + 1] % A);
            }
            tree_expand<G>(c, t, leaf, reward, prior);
            tree_backup<G>(c, t, leaf, value);
            max_depth = max(max_depth, leaf.depth);
        }

        // ------------------------------------------------------------------ results
        if (lane < A) {
            const bool ok = (legal >> lane) & 1u;
            if (a.visit_counts) a.visit_counts[(size_t)g * A + lane] = ok ? t.visit[lane] : 0;
            if (a.root_priors) a.root_priors[(size_t)g * A + lane] = t.root_prior[lane];
        }
        if (lane == 0) {
            if (a.root_value) a.root_value[g] = (t.root_visit == 0) ? 0.0 : __ddiv_rn(t.root_vsum, (double)t.root_visit);
            if (a.root_predicted_value) a.root_predicted_value[g] = root_value;
            if (a.max_tree_depth) a.max_tree_depth[g] = max_depth;
            if (a.tie_count) a.tie_count[g] = t.ties;
            if (a.value_range) { a.value_range[2 * g] = t.lo; a.value_range[2 * g + 1] = t.hi; }
        }
        if (a.pool.visit) {      // MZ_FLAG_KEEP_TREE: spill the shared-memory tree to the HBM node pool
            const int slots = (N + 1) * A;
            const size_t pb = (size_t)g * slots;
            for (int s = lane; s < t.n_expanded * A; s += G) {
                a.pool.visit[pb + s] = t.visit[s];
                a.pool.vsum[pb + s] = t.vsum[s];
                a.pool.reward[pb + s] = t.reward[s];
                a.pool.prior[pb + s] = t.prior[s];
                a.pool.expansion[pb + s] = t.expansion[s];
            }
            if (lane < A) a.pool.root_prior[(size_t)g * A + lane] = t.root_prior[lane];
            if (!kTeacher && a.pool.hidden)
                for (int i = lane; i < t.n_expanded * E; i += G)
                    a.pool.hidden[(size_t)g * (N + 1) * E + i] = s_hidden[(i / E) * Epad + (i % E)];
            if (lane == 0) {
                a.pool.root_visit[g] = t.root_visit;
                a.pool.root_vsum[g] = t.root_vsum;
                a.pool.n_expanded[g] = t.n_expanded;
            }
        }
        LaneGroup<G>::sync();
    }
    (void)F;
}

// ------------------------------------------------------------------------------------------
// host launcher
// ------------------------------------------------------------------------------------------
template <int G, bool T, typename SH>
static cudaError_t launch_one(const FcSearchArgs& a, int sm_count, size_t smem_cap, cudaStream_t stream, FcLaunchInfo* info) {
    const GameSmem L = game_smem_layout(a.N, a.A, a.net.E, a.net.maxw, !T);
    const size_t shared_bytes = ((2 * (size_t)(a.N + 2) * 8 + (T ? 0 : (size_t)a.net.blob_floats) * 4) + 15) & ~(size_t)15;
    const int threads = a.threads;
    const int groups = threads / G;
    if (groups < 1) return cudaErrorInvalidValue;
    const size_t smem = shared_bytes + (size_t)groups * L.bytes;
    if (smem > smem_cap) return cudaErrorInvalidConfiguration;
    auto kern = fc_search_kernel<G, T, SH>;
    cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (err != cudaSuccess) return err;
    int per_sm = 0;
    err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, smem);
    if (err != cudaSuccess) return err;
    if (per_sm < 1) return cudaErrorInvalidConfiguration;
    const int want = (a.n_games + groups - 1) / groups;
    const int grid = want < per_sm * sm_count ? want : per_sm * sm_count;
    if (info) { info->grid = grid; info->block = threads; info->smem = smem; info->ctas_per_sm = per_sm; info->group = G; }
    kern<<<grid, threads, smem, stream>>>(a);
    return cudaGetLastError();
}

// shapes with a fully unrolled network path: games/cartpole.py (encoding 8, hidden 16, support 10, 2 actions)
using CartPoleShape = FcFixedShape<8, 16, 10, 2>;

cudaError_t launch_fc_search(const FcSearchArgs& args, int group, bool teacher, int sm_count, size_t smem_cap,
                             cudaStream_t stream, FcLaunchInfo* info) {
    FcSearchArgs a = args;
    const char* la = getenv("MZ_FC_LOOKAHEAD");                // A/B switch: 0 selects one tree level per round
    a.lookahead = (a.A <= 2 && !(la && la[0] == '0')) ? 1 : 0;
    const char* generic = getenv("MZ_FC_GENERIC");             // A/B switch: always walk the layer descriptors
    if (!teacher && !(generic && generic[0] == '1') && fc_matches_fixed<CartPoleShape>(a.net)) {
        if (group == 16) return launch_one<16, false, CartPoleShape>(a, sm_count, smem_cap, stream, info);
        if (group == 32) return launch_one<32, false, CartPoleShape>(a, sm_count, smem_cap, stream, info);
    }
#define MZ_CASE(GG)                                                                                     \
    case GG:                                                                                            \
        return teacher ? launch_one<GG, true, FcGenericShape>(a, sm_count, smem_cap, stream, info)      \
                       : launch_one<GG, false, FcGenericShape>(a, sm_count, smem_cap, stream, info);
    switch (group) {
        MZ_CASE(4)
        MZ_CASE(8)
        MZ_CASE(16)
        MZ_CASE(32)
    }
#undef MZ_CASE
    return cudaErrorInvalidValue;
}

size_t fc_search_smem_bytes(const FcSearchArgs& a, int group, bool teacher) {
    const GameSmem L = game_smem_layout(a.N, a.A, a.net.E, a.net.maxw, !teacher);
    const size_t shared_bytes = ((2 * (size_t)(a.N + 2) * 8 + (teacher ? 0 : (size_t)a.net.blob_floats) * 4) + 15) & ~(size_t)15;
    return shared_bytes + (size_t)(a.threads / group) * L.bytes;
}

}  // namespace mz
