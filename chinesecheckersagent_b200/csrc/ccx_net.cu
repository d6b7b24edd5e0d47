// ccx_net.cu — policy/value network inference (model.py:58-145 via Model.predict, model.py:21-24).
//
// Stage-1 kernel ("simt"): fp32 SIMT, one warp per position, the whole 33-layer graph fused in one
// kernel with every activation of a position resident in shared memory (never written to HBM);
// BatchNorm is folded into the conv weights/biases on the host (chinesecheckersagent_b200/model.py).
// HBM traffic per position = 343 B of input planes in, 1,180 B of logits+value out; the 0.98 MB of
// folded fp32 weights are read through L1/L2.  This kernel doubles as the on-device fp32 reference for
// the bf16 tensor-core kernel.
//
// Packed weight blob (fp32, BN folded), offsets in floats — must match model.py `pack_weights`:
//   conv1   W[63][64]  b[64]                k = (dy*3+dx)*7  + cin          (model.py:62, 'valid')
//   block b (9x): A W[64][32] b[32] | B W[288][32] b[32] (k = (dy*3+dx)*32 + cin, 'same') | C W[32][64] b[64]
//   policy  conv W[64][16] b[16] | dense W[400][294] b[294]   (flatten (y,x,c), model.py:107-117)
//   value   conv W[64] b[1] | dense_1 W[25][32] b[32] | value_head W[32] b[1]   (model.py:90-104)
#include <cuda_bf16.h>
#include "ccx_device.cuh"
#include "ccx_internal.h"
#include "ccx_sym.cuh"
#include <new>

namespace netl {
constexpr int CONV1_W = 0, CONV1_B = CONV1_W + 63 * 64;
constexpr int BLOCK0 = CONV1_B + 64;
constexpr int BA_W = 0, BA_B = BA_W + 64 * 32, BB_W = BA_B + 32, BB_B = BB_W + 288 * 32, BC_W = BB_B + 32, BC_B = BC_W + 32 * 64;
constexpr int BLOCK_STRIDE = BC_B + 64;
constexpr int POLC_W = BLOCK0 + 9 * BLOCK_STRIDE, POLC_B = POLC_W + 64 * 16;
constexpr int POLD_W = POLC_B + 16, POLD_B = POLD_W + 400 * 294;
constexpr int VALC_W = POLD_B + 294, VALC_B = VALC_W + 64;
constexpr int D1_W = VALC_B + 1, D1_B = D1_W + 25 * 32;
constexpr int VH_W = D1_B + 32, VH_B = VH_W + 32;
constexpr int TOTAL = VH_B + 1;
static_assert(TOTAL == 244920, "packed weight count");
}  // namespace netl

struct ccx_net {
    float *w = nullptr;           // packed fp32 weights on the device
    float *logits = nullptr;      // scratch for ccx_net_eval: [cap][294]
    float *value = nullptr;       // [cap]
    uint8_t *planes = nullptr;    // [cap][343]
    int64_t cap = 0;
};

#define NET_G 8                    // positions (= warps) per CTA
#define XLD 68                     // row stride of the 64-channel activation (floats): 16-byte aligned rows

// out[row][lane (+32)] for the 25 rows of this warp's position: A (25 x K, row stride lda) times W (K x N)
template <int K, int N, bool RELU, bool RESIDUAL>
__device__ __forceinline__ void layer_1x1(const float *A, int lda, const float *__restrict__ W, const float *__restrict__ bias,
                                          float *out, int ldo, int lane)
{
    constexpr int NJ = N / 32;
    float acc[25][NJ];
#pragma unroll
    for (int r = 0; r < 25; r++)
#pragma unroll
        for (int j = 0; j < NJ; j++) acc[r][j] = __ldg(bias + lane + 32 * j);
    for (int k = 0; k < K; k += 4) {
        float w[4][NJ];
#pragma unroll
        for (int q = 0; q < 4; q++)
#pragma unroll
            for (int j = 0; j < NJ; j++) w[q][j] = __ldg(W + (k + q) * N + lane + 32 * j);
#pragma unroll
        for (int r = 0; r < 25; r++) {
            float4 a = *reinterpret_cast<const float4 *>(A + r * lda + k);
#pragma unroll
            for (int j = 0; j < NJ; j++) {
                acc[r][j] = fmaf(a.x, w[0][j], acc[r][j]); acc[r][j] = fmaf(a.y, w[1][j], acc[r][j]);
                acc[r][j] = fmaf(a.z, w[2][j], acc[r][j]); acc[r][j] = fmaf(a.w, w[3][j], acc[r][j]);
            }
        }
    }
    __syncwarp();          // RESIDUAL reads `out` (the block input) before overwriting it
#pragma unroll
    for (int r = 0; r < 25; r++)
#pragma unroll
        for (int j = 0; j < NJ; j++) {
            float v = acc[r][j];
            if (RESIDUAL) v += out[r * ldo + lane + 32 * j];          // model.py:143 add([x, block_input])
            if (RELU) v = fmaxf(v, 0.f);
            out[r * ldo + lane + 32 * j] = v;
        }
    __syncwarp();
}

// 3x3 'same' conv on the 5x5x32 grid (model.py:129-135): 9 shifted K=32 accumulations
__device__ __forceinline__ void layer_3x3(const float *A, const float *__restrict__ W, const float *__restrict__ bias,
                                          float *out, int lane)
{
    float acc[25];
#pragma unroll
    for (int r = 0; r < 25; r++) acc[r] = __ldg(bias + lane);
#pragma unroll
    for (int tap = 0; tap < 9; tap++) {
        const int dy = tap / 3 - 1, dx = tap % 3 - 1;
        for (int c = 0; c < 32; c += 4) {
            float w0 = __ldg(W + (tap * 32 + c + 0) * 32 + lane), w1 = __ldg(W + (tap * 32 + c + 1) * 32 + lane);
            float w2 = __ldg(W + (tap * 32 + c + 2) * 32 + lane), w3 = __ldg(W + (tap * 32 + c + 3) * 32 + lane);
#pragma unroll
            for (int r = 0; r < 25; r++) {
                const int y = r / 5 + dy, x = r % 5 + dx;
                if (y < 0 || y > 4 || x < 0 || x > 4) continue;          // zero padding (compile-time per r, tap)
                float4 a = *reinterpret_cast<const float4 *>(A + (y * 5 + x) * 32 + c);
                acc[r] = fmaf(a.x, w0, acc[r]); acc[r] = fmaf(a.y, w1, acc[r]);
                acc[r] = fmaf(a.z, w2, acc[r]); acc[r] = fmaf(a.w, w3, acc[r]);
            }
        }
    }
#pragma unroll
    for (int r = 0; r < 25; r++) out[r * 32 + lane] = fmaxf(acc[r], 0.f);
    __syncwarp();
}

template <typename TIN> __device__ __forceinline__ float plane_val(TIN v);
template <> __device__ __forceinline__ float plane_val<uint8_t>(uint8_t v) { return (float)v; }
template <> __device__ __forceinline__ float plane_val<float>(float v) { return v; }
template <> __device__ __forceinline__ float plane_val<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }

template <typename TIN>
__global__ void __launch_bounds__(32 * NET_G)
k_net_forward_simt(const float *__restrict__ wts, const TIN *__restrict__ planes, int64_t n,
                   float *__restrict__ logits, float *__restrict__ value, const int32_t *__restrict__ count)
{
    if (count) n = min(n, (int64_t)*count);        // compacted batch: the row count on the device
    if ((int64_t)blockIdx.x * NET_G >= n) return;
    extern __shared__ float4 smem_f4[];
    float *smem = reinterpret_cast<float *>(smem_f4);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t pos = (int64_t)blockIdx.x * NET_G + warp;
    // per-warp regions: X[25][XLD] | M1[25][32] | M2[25][32]   (xin[343] aliases M1+M2)
    constexpr int PER_WARP = 25 * XLD + 25 * 32 + 25 * 32;
    float *X = smem + warp * PER_WARP, *M1 = X + 25 * XLD, *M2 = M1 + 25 * 32;
    float *xin = M1;
    const bool live = pos < n;
    if (live) {
        for (int i = lane; i < 343; i += 32) xin[i] = plane_val<TIN>(planes[pos * 343 + i]);
        __syncwarp();
        // conv1: 3x3 'valid' on (7,7,7) -> (5,5,64), BN folded, relu   (model.py:62-64)
        {
            float acc[25][2];
#pragma unroll
            for (int r = 0; r < 25; r++) { acc[r][0] = __ldg(wts + netl::CONV1_B + lane); acc[r][1] = __ldg(wts + netl::CONV1_B + lane + 32); }
#pragma unroll
            for (int tap = 0; tap < 9; tap++) {
                const int dy = tap / 3, dx = tap % 3;
                for (int c = 0; c < 7; c++) {
                    float w0 = __ldg(wts + netl::CONV1_W + (tap * 7 + c) * 64 + lane);
                    float w1 = __ldg(wts + netl::CONV1_W + (tap * 7 + c) * 64 + lane + 32);
#pragma unroll
                    for (int r = 0; r < 25; r++) {
                        float a = xin[((r / 5 + dy) * 7 + (r % 5 + dx)) * 7 + c];
                        acc[r][0] = fmaf(a, w0, acc[r][0]); acc[r][1] = fmaf(a, w1, acc[r][1]);
                    }
                }
            }
            __syncwarp();
#pragma unroll
            for (int r = 0; r < 25; r++) { X[r * XLD + lane] = fmaxf(acc[r][0], 0.f); X[r * XLD + lane + 32] = fmaxf(acc[r][1], 0.f); }
            __syncwarp();
        }
        // 9 bottleneck residual blocks (model.py:120-145)
        for (int b = 0; b < 9; b++) {
            const float *bw = wts + netl::BLOCK0 + b * netl::BLOCK_STRIDE;
            layer_1x1<64, 32, true, false>(X, XLD, bw + netl::BA_W, bw + netl::BA_B, M1, 32, lane);
            layer_3x3(M1, bw + netl::BB_W, bw + netl::BB_B, M2, lane);
            layer_1x1<32, 64, true, true>(M2, 32, bw + netl::BC_W, bw + netl::BC_B, X, XLD, lane);
        }
        // policy conv 1x1 64->16 + relu -> M1 as flat[400] in (y, x, c) order (model.py:108-111)
        {
            const int c = lane & 15, half = lane >> 4;
            for (int r = half; r < 25; r += 2) {
                float acc = __ldg(wts + netl::POLC_B + c);
                for (int k = 0; k < 64; k++) acc = fmaf(X[r * XLD + k], __ldg(wts + netl::POLC_W + k * 16 + c), acc);
                M1[r * 16 + c] = fmaxf(acc, 0.f);
            }
        }
        // value conv 1x1 64->1 + relu -> M2[0..24]; dense_1 25->32 relu; value_head 32->1 tanh (model.py:91-104)
        if (lane < 25) {
            float acc = __ldg(wts + netl::VALC_B);
            for (int k = 0; k < 64; k++) acc = fmaf(X[lane * XLD + k], __ldg(wts + netl::VALC_W + k), acc);
            M2[lane] = fmaxf(acc, 0.f);
        }
        __syncwarp();
        {
            float acc = __ldg(wts + netl::D1_B + lane);
            for (int k = 0; k < 25; k++) acc = fmaf(M2[k], __ldg(wts + netl::D1_W + k * 32 + lane), acc);
            float t = fmaxf(acc, 0.f) * __ldg(wts + netl::VH_W + lane);
#pragma unroll
            for (int off = 16; off; off >>= 1) t += __shfl_xor_sync(0xFFFFFFFFu, t, off);
            if (lane == 0) value[pos] = tanhf(t + __ldg(wts + netl::VH_B));
        }
    }
    __syncthreads();
    // policy dense 400 -> 294 for the CTA's 8 positions together: thread t owns logits t and t + 256
    {
        const int t = threadIdx.x;
        const bool second = t + 256 < 294;
        float acc0[NET_G], acc1[NET_G];
        const float b0 = __ldg(wts + netl::POLD_B + t), b1 = second ? __ldg(wts + netl::POLD_B + t + 256) : 0.f;
#pragma unroll
        for (int g = 0; g < NET_G; g++) { acc0[g] = b0; acc1[g] = b1; }
        const float *Wd = wts + netl::POLD_W;
        for (int k = 0; k < 400; k += 4) {
            float w0[4], w1[4];
#pragma unroll
            for (int q = 0; q < 4; q++) { w0[q] = __ldg(Wd + (k + q) * 294 + t); w1[q] = second ? __ldg(Wd + (k + q) * 294 + t + 256) : 0.f; }
#pragma unroll
            for (int g = 0; g < NET_G; g++) {
                float4 a = *reinterpret_cast<const float4 *>(smem + g * PER_WARP + 25 * XLD + k);      // that warp's M1 = flat[400]
                acc0[g] = fmaf(a.x, w0[0], acc0[g]); acc0[g] = fmaf(a.y, w0[1], acc0[g]);
                acc0[g] = fmaf(a.z, w0[2], acc0[g]); acc0[g] = fmaf(a.w, w0[3], acc0[g]);
                acc1[g] = fmaf(a.x, w1[0], acc1[g]); acc1[g] = fmaf(a.y, w1[1], acc1[g]);
                acc1[g] = fmaf(a.z, w1[2], acc1[g]); acc1[g] = fmaf(a.w, w1[3], acc1[g]);
            }
        }
#pragma unroll
        for (int g = 0; g < NET_G; g++) {
            int64_t p = (int64_t)blockIdx.x * NET_G + g;
            if (p < n) {
                logits[p * 294 + t] = acc0[g];
                if (second) logits[p * 294 + t + 256] = acc1[g];
            }
        }
    }
}

// Model.predict's utils.softmax in float64 over all 294 logits, no legality mask (model.py:21-24, utils.py:187-192), one warp
// per position; also widens v to float64 for the tree statistics.  SYM != SYM_OFF (ccx_net_set_symmetry): position i owns net
// rows [i * SymRows, (i + 1) * SymRows) and st = its state words [5][n] (SYM_RANDOM's orientation); SYM_OFF reads no state words.
template <int SYM>
__global__ void __launch_bounds__(128)
k_softmax_f64(const float *__restrict__ logits, const float *__restrict__ value, const uint64_t *__restrict__ st, int64_t n, uint32_t k0,
              uint32_t k1, double *__restrict__ p, double *__restrict__ v)
{
    constexpr int R = SymRows<SYM>::value;
    const int64_t pos = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (pos >= n) return;
    const bool mir = SYM == SYM_RANDOM && sym_mirrored(k0, k1, st[0 * n + pos], st[1 * n + pos], st[4 * n + pos]);
    sym_priors<SYM>(lane, logits + pos * R * 294, mir, p + pos * 294);
    if (v && lane == 0) v[pos] = sym_value<SYM>(value + pos * R);
}

// ---- mirror-symmetric evaluation (ccx_net_set_symmetry): the planes of leaf i go to rows [i * SymRows, (i + 1) * SymRows)
// of the net batch, one warp per position, the encode of the fused MCTS kernels (ccx_sym.cuh)
template <int SYM>
__global__ void __launch_bounds__(128)
k_encode_sym(const uint64_t *__restrict__ st, int64_t n, uint32_t k0, uint32_t k1, uint8_t *__restrict__ planes)
{
    __shared__ __align__(16) uint8_t sP[4][352];
    const int64_t pos = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
    if (pos >= n) return;
    const bool p2 = (st[4 * n + pos] >> 48) & 1;
    Game g;
    g.meta = st[4 * n + pos];
    g.occ_me = st[(p2 ? 1 : 0) * n + pos]; g.occ_op = st[(p2 ? 0 : 1) * n + pos];
    g.cells_me = st[(p2 ? 3 : 2) * n + pos]; g.cells_op = st[(p2 ? 2 : 3) * n + pos];
    sym_encode<SYM>(g, threadIdx.x & 31, k0, k1, sP[threadIdx.x >> 5], planes + pos * SymRows<SYM>::value * 343);
}

// ---- host side ------------------------------------------------------------------------------------------

void ccx_net_free(ccx_handle *h)
{
    ccx_net *nt = h->net;
    if (!nt) return;
    void *ptrs[] = {nt->w, nt->logits, nt->value, nt->planes};
    for (void *p : ptrs) if (p) cudaFree(p);
    delete nt;
    h->net = nullptr;
}

static constexpr int NET_SMEM = NET_G * (25 * XLD + 25 * 32 + 25 * 32) * 4;

extern "C" {

int ccx_net_num_weights(void) { return netl::TOTAL; }

int ccx_net_load(ccx_handle *h, const float *packed_host, int64_t count)
{
    if (!h || !packed_host || count != netl::TOTAL) return CCX_ERR_ARG;
    if (!h->net) {
        h->net = new (std::nothrow) ccx_net();
        if (!h->net) return CCX_ERR_NOMEM;
    }
    h->epoch++;
    h->pool_gen++;                                   // trees searched with the old weights are no start for a reuse begin
    if (!h->net->w) CCX_CUDA(h, cudaMalloc(&h->net->w, sizeof(float) * netl::TOTAL));
    CCX_CUDA(h, cudaMemcpyAsync(h->net->w, packed_host, sizeof(float) * netl::TOTAL, cudaMemcpyHostToDevice, h->stream));
    CCX_CUDA(h, cudaStreamSynchronize(h->stream));
    CCX_CUDA(h, cudaFuncSetAttribute(k_net_forward_simt<uint8_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, NET_SMEM));
    CCX_CUDA(h, cudaFuncSetAttribute(k_net_forward_simt<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, NET_SMEM));
    CCX_CUDA(h, cudaFuncSetAttribute(k_net_forward_simt<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, NET_SMEM));
    return CCX_OK;
}

int ccx_net_forward(ccx_handle *h, int64_t n, const void *planes, int dtype, float *logits, float *value)
{
    if (!h || n < 0 || (n && (!planes || !logits || !value))) return CCX_ERR_ARG;
    if (!h->net || !h->net->w) return CCX_ERR_STATE;
    if (n == 0) return CCX_OK;
    unsigned grid = (unsigned)((n + NET_G - 1) / NET_G);
    switch (dtype) {
    case CCX_DTYPE_U8:
        k_net_forward_simt<uint8_t><<<grid, 32 * NET_G, NET_SMEM, h->stream>>>(h->net->w, (const uint8_t *)planes, n, logits, value, nullptr);
        break;
    case CCX_DTYPE_BF16:
        k_net_forward_simt<__nv_bfloat16><<<grid, 32 * NET_G, NET_SMEM, h->stream>>>(h->net->w, (const __nv_bfloat16 *)planes, n, logits, value, nullptr);
        break;
    case CCX_DTYPE_F32:
        k_net_forward_simt<float><<<grid, 32 * NET_G, NET_SMEM, h->stream>>>(h->net->w, (const float *)planes, n, logits, value, nullptr);
        break;
    default:
        return CCX_ERR_ARG;
    }
    CCX_LAUNCHED(h);
    return CCX_OK;
}

int ccx_softmax_f64(ccx_handle *h, int64_t n, const float *logits, const float *value, double *p, double *v)
{
    if (!h || n < 0 || (n && (!logits || !p)) || (v && !value)) return CCX_ERR_ARG;
    if (n == 0) return CCX_OK;
    k_softmax_f64<SYM_OFF><<<(unsigned)((n + 3) / 4), 128, 0, h->stream>>>(logits, value, nullptr, n, 0, 0, p, v);
    CCX_LAUNCHED(h);
    return CCX_OK;
}

int ccx_net_set_mode(ccx_handle *h, int32_t mode)
{
    if (!h || (mode != 0 && mode != 1 && mode != 2)) return CCX_ERR_ARG;
    if (mode == 1 && !h->net_tc) return CCX_ERR_STATE;
    if (mode == 2 && (!h->net_tc || !h->net_acc || !h->net || !h->net->w)) return CCX_ERR_STATE;
    if (h->net_mode != mode) { h->epoch++; h->pool_gen++; }      // a cached round graph holds the old mode's kernels; the trees hold its values
    h->net_mode = mode;
    return CCX_OK;
}

int ccx_net_set_symmetry(ccx_handle *h, int32_t mode, uint64_t seed)
{
    if (!h || mode < SYM_OFF || mode > SYM_MEAN) return CCX_ERR_ARG;
    if (h->sym_mode != mode || h->sym_seed != seed) { h->epoch++; h->pool_gen++; }   // another evaluator: no cached round graph, no carried tree
    h->sym_mode = mode;
    h->sym_seed = seed;
    return CCX_OK;
}

// Model.predict for a batch of packed states (leaf_state = words 0-4, plane-major [5][n]):
// to_model_input -> net -> float64 softmax.  The MCTS round loop's evaluator.
int ccx_net_eval(ccx_handle *h, int64_t n, const uint64_t *leaf_state, double *p, double *v)
{
    if (!h || n < 0 || (n && (!leaf_state || !p || !v))) return CCX_ERR_ARG;
    if (!h->net || !h->net->w) return CCX_ERR_STATE;
    if (n == 0) return CCX_OK;
    uint8_t *planes; float *logits, *value;
    int rc;
    if (h->sym_mode != SYM_OFF) {
        const int64_t rows = h->sym_mode == SYM_MEAN ? 2 * n : n;
        const uint32_t k0 = (uint32_t)h->sym_seed, k1 = (uint32_t)(h->sym_seed >> 32);
        const unsigned grid = (unsigned)((n + 3) / 4);
        if ((rc = ccx_net_scratch(h, rows, &planes, &logits, &value))) return rc;
        if (h->sym_mode == SYM_MEAN) k_encode_sym<SYM_MEAN><<<grid, 128, 0, h->stream>>>(leaf_state, n, k0, k1, planes);
        else k_encode_sym<SYM_RANDOM><<<grid, 128, 0, h->stream>>>(leaf_state, n, k0, k1, planes);
        CCX_LAUNCHED(h);
        if ((rc = ccx_net_forward_active(h, rows, planes, logits, value))) return rc;
        if (h->sym_mode == SYM_MEAN) k_softmax_f64<SYM_MEAN><<<grid, 128, 0, h->stream>>>(logits, value, leaf_state, n, k0, k1, p, v);
        else k_softmax_f64<SYM_RANDOM><<<grid, 128, 0, h->stream>>>(logits, value, leaf_state, n, k0, k1, p, v);
        CCX_LAUNCHED(h);
        return CCX_OK;
    }
    if ((rc = ccx_net_scratch(h, n, &planes, &logits, &value))) return rc;
    if ((rc = ccx_encode(h, n, leaf_state, planes, CCX_DTYPE_U8))) return rc;
    if ((rc = ccx_net_forward_active(h, n, planes, logits, value))) return rc;
    return ccx_softmax_f64(h, n, logits, value, p, v);
}

}  // extern "C"

int ccx_net_scratch(ccx_handle *h, int64_t n, uint8_t **planes, float **logits, float **value)
{
    if (!h->net || !h->net->w) return CCX_ERR_STATE;
    ccx_net *nt = h->net;
    if (nt->cap < n) {
        h->epoch++;
        void *ptrs[] = {nt->logits, nt->value, nt->planes};
        for (void *q : ptrs) if (q) CCX_CUDA(h, cudaFree(q));
        nt->logits = nullptr; nt->value = nullptr; nt->planes = nullptr; nt->cap = 0;
        CCX_CUDA(h, cudaMalloc(&nt->logits, sizeof(float) * 294 * (size_t)n));
        CCX_CUDA(h, cudaMalloc(&nt->value, sizeof(float) * (size_t)n));
        CCX_CUDA(h, cudaMalloc(&nt->planes, 343 * (size_t)n + 16));
        nt->cap = n;
    }
    *planes = nt->planes; *logits = nt->logits; *value = nt->value;
    return CCX_OK;
}

extern "C" int ccx_net_forward_u8(ccx_handle *h, int64_t n, const uint8_t *planes, float *logits, float *value)
{
    if (!h || n < 0 || (n && (!planes || !logits || !value))) return CCX_ERR_ARG;
    if (!h->net || !h->net->w) return CCX_ERR_STATE;
    return ccx_net_forward_active(h, n, planes, logits, value);
}

const float *ccx_net_pold_bias(const ccx_handle *h) { return (h && h->net && h->net->w) ? h->net->w + netl::POLD_B : nullptr; }

int ccx_net_forward_active(ccx_handle *h, int64_t n, const uint8_t *planes, float *logits, float *value, const int32_t *count)
{
    if (h->net_mode == 1) return count ? ccx_net_forward_tc_on(h, h->stream, n, 0, n, planes, logits, value, count)
                                       : ccx_net_forward_tc(h, n, planes, logits, value);
    if (h->net_mode == 2) return count ? ccx_net_forward_acc_on(h, h->stream, n, 0, n, planes, logits, value, h->net->w + netl::POLD_B, count)
                                       : ccx_net_forward_acc(h, n, planes, logits, value, h->net->w + netl::POLD_W, h->net->w + netl::POLD_B);
    if (!count) return ccx_net_forward(h, n, planes, CCX_DTYPE_U8, logits, value);
    if (!h->net || !h->net->w) return CCX_ERR_STATE;
    if (n == 0) return CCX_OK;
    k_net_forward_simt<uint8_t><<<(unsigned)((n + NET_G - 1) / NET_G), 32 * NET_G, NET_SMEM, h->stream>>>(h->net->w, planes, n, logits, value, count);
    CCX_LAUNCHED(h);
    return CCX_OK;
}
