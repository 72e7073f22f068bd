// Internal interface between the host side of the library (abi.cu) and the kernel files.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "../../include/mzb200.h"
#include "fc_net.cuh"

namespace mz {

constexpr int kFcThreads = 128;      // fc_inference_kernel block
constexpr int kFcMaxThreads = 128;   // upper bound of the fused search kernel's block

// HBM node pool, game-major: game g owns slots [g*(N+1)*A, (g+1)*(N+1)*A).
struct NodePool {
    int* visit;            // [B, (N+1)*A]
    double* vsum;          // [B, (N+1)*A]
    double* mval;          // [B, (N+1)*A] cached reward + discount * (+/-)mean of every visited child (tree.cuh)
    float* reward;         // [B, (N+1)*A]
    float* prior;          // [B, (N+1)*A]
    int* expansion;        // [B, (N+1)*A]
    double* root_prior;    // [B, A]
    float* hidden;         // [B, N+1, hidden_elems]
    int* root_visit;       // [B]
    double* root_vsum;     // [B]
    float* root_reward;    // [B]
    double* range;         // [B, 2]
    int* n_expanded;       // [B]
    int* ties;             // [B]
    int* max_depth;        // [B]
    unsigned* legal;       // [B]
    int* path;             // [B, N+2]
    float* path_reward;    // [B, N+2]
    // leaf of the simulation in flight
    int* leaf_depth;       // [B]
    int* leaf_parent;      // [B]
    int* leaf_action;      // [B]
    int* leaf_slot;        // [B]
    // network outputs of the evaluation in flight (step-wise pipeline)
    float* net_value;      // [B]
    float* net_reward;     // [B]
    float* net_policy;     // [B, A]
};

struct DevTeacher { const float *root_value, *root_reward, *root_priors, *value, *reward, *priors; };
struct DevTrace {
    int max_depth;
    int* depth; uint8_t* actions; float *value, *reward, *priors, *root_priors_raw, *root_reward;
    double* noise;         // [n, A] Dirichlet noise actually mixed in (host-given or device-drawn)
};

struct FcSearchArgs {
    int n_games, N, A, P;
    int threads;           // block size of the launch (multiple of 32)
    double discount, noise_frac, noise_alpha;
    uint64_t seed;
    const double* pbc;
    const double* sqrtn;
    const double* ucb;
    FcNet net;
    const float* blob;
    // inputs (device)
    const float* obs;
    const uint8_t* legal_mask;
    const int32_t* to_play;
    int add_noise;
    const double* noise;
    const int32_t* first_index;
    const int64_t* game_id;
    const int32_t* move_index;
    // outputs (device)
    int32_t* visit_counts;
    double* root_value;
    float* root_predicted_value;
    int32_t* max_tree_depth;
    int32_t* tie_count;
    double* root_priors;
    double* value_range;
    DevTeacher teacher;
    DevTrace trace;
    NodePool pool;         // pool.visit == nullptr unless MZ_FLAG_KEEP_TREE
    int lookahead;         // set by launch_fc_search: several tree levels per selection round (|A| <= 2, tree.cuh)
};

struct FcInferArgs {
    int n, recurrent;
    FcNet net;
    const float* blob;
    const float* in;          // obs [n, obs_elems] (initial) or hidden [n, E] (recurrent)
    const int32_t* action;    // [n] (recurrent)
    // pool mode: sample g reads pool_hidden[(g*pool_stride + gather_parent[g])*E ...] and writes its
    // new state to pool_hidden[(g*pool_stride + out_slot)*E ...]
    const int32_t* gather_parent;
    float* pool_hidden;
    int pool_stride, out_slot;
    float *value_logits, *reward_logits, *policy_logits, *hidden, *value, *reward;
};
cudaError_t launch_fc_inference(const FcInferArgs& a, int group, int sm_count, cudaStream_t stream);

struct FcLaunchInfo { int grid, block, ctas_per_sm, group; size_t smem; };

cudaError_t launch_fc_search(const FcSearchArgs& a, int group, bool teacher, int sm_count, size_t smem_cap,
                             cudaStream_t stream, FcLaunchInfo* info);
size_t fc_search_smem_bytes(const FcSearchArgs& a, int group, bool teacher);

}  // namespace mz
