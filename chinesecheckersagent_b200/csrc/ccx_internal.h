// ccx_internal.h — the opaque handle behind include/ccx.h and the launch helpers shared by the .cu files.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include "../../include/ccx.h"

struct ccx_scratch {
    void *ptr = nullptr;
    size_t bytes = 0;
};

struct ccx_net;     // ccx_net.cu
struct ccx_trees;   // ccx_mcts.cu
struct ccx_net_tc;  // ccx_net_tc.cu
struct ccx_net_acc; // ccx_net_tc.cu (accurate split-precision mode)

struct ccx_handle {
    int device = 0;
    int num_sms = 148;
    cudaStream_t stream = nullptr;
    int64_t launches = 0;
    char cuda_err[256] = {0};
    // device scratch for the *_host entry points (grown on demand, freed in ccx_destroy)
    ccx_scratch d_state, d_aux0, d_aux1, d_aux2;
    ccx_net *net = nullptr;
    ccx_trees *trees = nullptr;
    ccx_net_tc *net_tc = nullptr;
    ccx_net_acc *net_acc = nullptr;
    uint8_t *jump_table = nullptr;   // CCX_JT_BYTES, device: ray-jump lookup table (ccx_device.cuh)
    uint8_t *jump_table3 = nullptr;  // CCX_JT3_BYTES, device: row / column / diagonal answer tables of the three-layout kernels
    uint8_t *jump_table_wide = nullptr;   // CCX_JTW_BYTES, device: the same answers per cell, placed on the board (one-wave carry kernel)
    bool carry_wide_smem = false;    // the one-wave carry kernel's dynamic shared-memory limit is raised (per device, so per handle)
    const int64_t *slot_ids = nullptr;   // device, caller-owned: identities of a compacted batch (ccx_set_slot_ids)
    int tie_mode = 0;           // PUCT tie rule of this handle's searches (ccx_mcts_set_tiebreak)
    uint64_t tie_seed = 0;
    int64_t tie_uid0 = 0;
    int net_mode = 0;           // 0 = fp32 SIMT kernel, 1 = 16-bit tcgen05 kernels, 2 = split-precision tcgen05 kernels (ccx_net_set_mode)
    int sym_mode = 0;           // mirror-symmetric net evaluation (ccx_net_set_symmetry): 0 off, 1 random orientation, 2 mean of both
    uint64_t sym_seed = 0;      // Philox key of the random orientation
    int acc_ctx = -1;           // tiles in flight per CTA of the accurate trunk (ccx_net_set_acc_contexts); -1 = take CCX_ACC_CTX / the default on first use
    // second stream + fork/join events of the two-half round pipeline (ccx_mcts_run_net), created on first use
    cudaStream_t stream2 = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    // CUDA-graph replay of the round loop (ccx_mcts_run_net): `epoch` changes whenever a device buffer the loop's kernels
    // receive is (re)allocated or the evaluator changes, which invalidates the cached graph
    uint64_t epoch = 0;
    // tree reuse (ccx_mcts_begin_reuse): `pool_gen` changes whenever the trees' contents stop being a valid start for the next
    // search (the pool was reallocated, the net was loaded or its mode changed); every begin records the generation and tree
    // count of the search it starts, and a reuse begin carries subtrees only from a search of the current generation
    uint64_t pool_gen = 1;
    uint64_t search_gen = 0;
    int64_t search_n = 0;
    void *round_graph = nullptr;     // ccx_round_graph (ccx_mcts.cu)
    void *leaf_pool = nullptr;       // ccx_leaf_pool (ccx_mcts.cu): per-leaf storage of the leaf-parallel rounds, freed with the trees
    void *reuse_pool = nullptr;      // ccx_reuse_pool (ccx_mcts.cu): scratch of the tree-reuse gather, freed with the trees
    // Gumbel search (ccx_mcts_set_gumbel): the mode and its parameters; gumbel_pool (ccx_gumbel_pool, ccx_mcts.cu) holds the
    // per-node values, root draws and schedule table, allocated by the first begin in the mode and freed with the trees
    int gumbel = 0;
    int32_t gumbel_m = 16;
    double gumbel_scale = 1.0, gumbel_c_visit = 50.0, gumbel_c_scale = 0.1;
    uint64_t gumbel_seed = 0;
    void *gumbel_pool = nullptr;
    cudaStream_t cap_stream = nullptr;
    int graph_off = 0;
    int64_t graph_replays = 0;
};

static inline int ccx_fail(ccx_handle *h, cudaError_t e)
{
    if (h) snprintf(h->cuda_err, sizeof(h->cuda_err), "%s: %s", cudaGetErrorName(e), cudaGetErrorString(e));
    return e == cudaErrorMemoryAllocation ? CCX_ERR_NOMEM : CCX_ERR_CUDA;
}

#define CCX_CUDA(h, call)                                   \
    do {                                                    \
        cudaError_t e__ = (call);                           \
        if (e__ != cudaSuccess) return ccx_fail((h), e__);  \
    } while (0)

// after a kernel launch: count it and surface launch-configuration errors
#define CCX_LAUNCHED(h)                                     \
    do {                                                    \
        (h)->launches++;                                    \
        cudaError_t e__ = cudaGetLastError();               \
        if (e__ != cudaSuccess) return ccx_fail((h), e__);  \
    } while (0)

static inline int ccx_reserve(ccx_handle *h, ccx_scratch &s, size_t bytes)
{
    if (s.bytes >= bytes) return CCX_OK;
    if (s.ptr) { CCX_CUDA(h, cudaFree(s.ptr)); s.ptr = nullptr; s.bytes = 0; }
    size_t want = bytes + bytes / 4;
    CCX_CUDA(h, cudaMalloc(&s.ptr, want));
    s.bytes = want;
    return CCX_OK;
}

// scratch of the net evaluator (planes uint8[n][343], logits float[n][294], value float[n]) and the forward pass in
// the active mode (ccx_net_set_mode) — used by ccx_net_eval and by the fused MCTS round loop (ccx_mcts_run_net)
int ccx_net_scratch(ccx_handle *h, int64_t n, uint8_t **planes, float **logits, float **value);
int ccx_net_forward_active(ccx_handle *h, int64_t n, const uint8_t *planes, float *logits, float *value);
// tensor-core forward on an explicit stream, rows [row0, row0 + n) of the evaluator scratch (capacity reserved by the caller)
int ccx_net_forward_tc_on(ccx_handle *h, cudaStream_t stream, int64_t cap, int64_t row0, int64_t n, const uint8_t *planes, float *logits,
                          float *value);

int ccx_net_forward_acc_on(ccx_handle *h, cudaStream_t stream, int64_t cap, int64_t row0, int64_t n, const uint8_t *planes, float *logits,
                           float *value, const float *b_pold);
const float *ccx_net_pold_bias(const ccx_handle *h);     // fp32 policy-dense bias inside the SIMT weight blob (ccx_net.cu)

// sub-module teardown hooks (defined where the sub-module lives)
void ccx_net_free(ccx_handle *h);
void ccx_trees_free(ccx_handle *h);
void ccx_trees_set_uids(ccx_handle *h, const int64_t *uids);     // tie-rule identities of the trees (ccx_set_slot_ids)
void ccx_round_graph_free(ccx_handle *h);
void ccx_net_tc_free(ccx_handle *h);
void ccx_net_acc_free(ccx_handle *h);
extern "C" int ccx_net_forward_acc(ccx_handle *h, int64_t n, const uint8_t *planes, float *logits, float *value, const float *w_pold,
                                   const float *b_pold);
