// ccx_net_tc.cu — tensor-core (tcgen05 + TMEM) path of the policy/value net (model.py:58-145): tcgen05 self-tests,
// the trunk kernel (k_net_trunk_tc4), the policy dense kernel (k_policy_dense_tc3) and their C-ABI entry points.
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include "ccx_device.cuh"
#include "ccx_internal.h"
#include "ccx_umma.cuh"
#include <new>
#include <cstdlib>

// ---- self-test of the UMMA plumbing: D[128 x N] = A[128 x K] * Bt[N x K]^T -------------------------------
__global__ void __launch_bounds__(128)
k_umma_selftest(const __nv_bfloat16 *__restrict__ A, const __nv_bfloat16 *__restrict__ Bt, int K, int N, float *__restrict__ D)
{
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ uint64_t bar;
    __shared__ uint32_t tmem_slot;
    uint8_t *sa = smem, *sb = smem + umma::op_bytes(128, K);
    const int t = threadIdx.x, warp = t >> 5;
    for (int i = t; i < 128 * K; i += 128) {
        int r = i / K, k = i % K;
        *reinterpret_cast<__nv_bfloat16 *>(sa + umma::op_offset(r, k, K)) = A[i];
    }
    for (int i = t; i < N * K; i += 128) {
        int r = i / K, k = i % K;
        *reinterpret_cast<__nv_bfloat16 *>(sb + umma::op_offset(r, k, K)) = Bt[i];
    }
    if (t == 0) umma::mbar_init(&bar, 1);
    if (warp == 0) umma::tmem_alloc(&tmem_slot, 64);
    umma::fence_async_smem();
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = tmem_slot;
    if (t == 0) {
        umma::gemm_issue(tmem, umma::smem_u32(sa), K, 0, umma::smem_u32(sb), K, 0, K, N, false);
        umma::commit(&bar);
    }
    umma::mbar_wait(&bar, 0);
    umma::fence_after_sync();
    for (int c = 0; c < N; c += 32) {
        float v[32];
        umma::tmem_ld32(tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)c, v);
#pragma unroll
        for (int j = 0; j < 32; j++) if (c + j < N) D[t * N + c + j] = v[j];
    }
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 0) umma::tmem_free(tmem, 64);
}

// Second self-test: the A operand in the ROW-CONTIGUOUS layout the 3x3 conv uses — element (r, k) at
// (k/8)*LBO + r*16 + (k%8)*2 with LBO = rows*16, SBO = 128 — and a descriptor whose start address is moved by
// `shift` rows (16 B each, NOT a multiple of the 128-byte core matrix): D = A[shift .. shift+127] * Bt^T.
__global__ void __launch_bounds__(128)
k_umma_selftest_rows(const __nv_bfloat16 *__restrict__ A, int rows, int shift, const __nv_bfloat16 *__restrict__ Bt, int K, int N,
                     float *__restrict__ D)
{
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ uint64_t bar;
    __shared__ uint32_t tmem_slot;
    uint8_t *sa = smem, *sb = smem + (size_t)rows * K * 2;
    const int t = threadIdx.x, warp = t >> 5;
    for (int i = t; i < rows * K; i += 128) {
        int r = i / K, k = i % K;
        *reinterpret_cast<__nv_bfloat16 *>(sa + (k >> 3) * rows * 16 + r * 16 + (k & 7) * 2) = A[i];
    }
    for (int i = t; i < N * K; i += 128) {
        int r = i / K, k = i % K;
        *reinterpret_cast<__nv_bfloat16 *>(sb + umma::op_offset(r, k, K)) = Bt[i];
    }
    if (t == 0) umma::mbar_init(&bar, 1);
    if (warp == 0) umma::tmem_alloc(&tmem_slot, 64);
    umma::fence_async_smem();
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = tmem_slot;
    if (t == 0) {
        const uint32_t idesc = umma::make_idesc(N, false);
        for (int s = 0; s < K / 16; s++) {
            uint64_t ad = umma::make_desc(umma::smem_u32(sa) + (uint32_t)(2 * s) * rows * 16u + (uint32_t)shift * 16u, (uint32_t)rows * 16u, 128u);
            uint64_t bd = umma::make_desc(umma::smem_u32(sb) + (uint32_t)(2 * s) * 128u, 128u, (uint32_t)(K >> 3) * 128u);
            umma::mma_bf16(tmem, ad, bd, idesc, s > 0);
        }
        umma::commit(&bar);
    }
    umma::mbar_wait(&bar, 0);
    umma::fence_after_sync();
    for (int c = 0; c < N; c += 32) {
        float v[32];
        umma::tmem_ld32(tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)c, v);
#pragma unroll
        for (int j = 0; j < 32; j++) if (c + j < N) D[t * N + c + j] = v[j];
    }
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 0) umma::tmem_free(tmem, 64);
}

// Third self-test: the A operand read from TMEM (packed 16-bit pairs written with tcgen05.st): D = A * Bt^T, K = 64.
__global__ void __launch_bounds__(128)
k_umma_selftest_ts(const __nv_bfloat16 *__restrict__ A, const __nv_bfloat16 *__restrict__ Bt, int N, float *__restrict__ D)
{
    constexpr int K = 64;
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ uint64_t bar;
    __shared__ uint32_t tmem_slot;
    const int t = threadIdx.x, warp = t >> 5;
    for (int i = t; i < N * K; i += 128) {
        int r = i / K, k = i % K;
        *reinterpret_cast<__nv_bfloat16 *>(smem + umma::op_offset(r, k, K)) = Bt[i];
    }
    if (t == 0) umma::mbar_init(&bar, 1);
    if (warp == 0) umma::tmem_alloc(&tmem_slot, 128);
    umma::fence_async_smem();
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = tmem_slot;
    const uint32_t trow = tmem + ((uint32_t)(warp * 32) << 16);
    {
        uint32_t w[32];
#pragma unroll
        for (int j = 0; j < 32; j++) w[j] = reinterpret_cast<const uint32_t *>(A + (size_t)t * K)[j];   // elements 2j (low), 2j+1 (high)
        umma::tmem_st32(trow + 64, w);
        umma::tmem_wait_st();
    }
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 0) {
        umma::fence_after_sync();
        if (umma::elect_one()) {
            umma::gemm_issue_ts<K>(tmem, tmem + 64, umma::desc_base(umma::smem_u32(smem), 128u, K / 8 * 128u), 0, umma::make_idesc(N, false), false);
            umma::commit(&bar);
        }
        __syncwarp();
    }
    umma::mbar_wait(&bar, 0);
    umma::fence_after_sync();
    for (int c = 0; c < N; c += 16) {
        float v[16];
        umma::tmem_ld16(trow + (uint32_t)c, v);
#pragma unroll
        for (int j = 0; j < 16; j++) D[t * N + c + j] = v[j];
    }
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 0) umma::tmem_free(tmem, 128);
}

extern "C" {

int ccx_debug_umma_gemm_ts(ccx_handle *h, const void *A, const void *Bt, int32_t N, float *D)
{
    if (!h || !A || !Bt || !D || N % 16 || N < 16 || N > 64) return CCX_ERR_ARG;
    size_t smem = umma::op_bytes(N, 64);
    k_umma_selftest_ts<<<1, 128, smem, h->stream>>>((const __nv_bfloat16 *)A, (const __nv_bfloat16 *)Bt, N, D);
    CCX_LAUNCHED(h);
    return CCX_OK;
}

int ccx_debug_umma_gemm_rows(ccx_handle *h, const void *A, int32_t rows, int32_t shift, const void *Bt, int32_t K, int32_t N, float *D)
{
    if (!h || !A || !Bt || !D || K % 16 || K < 16 || K > 128 || N % 16 || N < 16 || N > 64 || rows % 8 || shift < 0 || shift + 128 > rows)
        return CCX_ERR_ARG;
    size_t smem = (size_t)rows * K * 2 + umma::op_bytes(N, K);
    if (smem > 200 * 1024) return CCX_ERR_ARG;
    CCX_CUDA(h, cudaFuncSetAttribute(k_umma_selftest_rows, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_umma_selftest_rows<<<1, 128, smem, h->stream>>>((const __nv_bfloat16 *)A, rows, shift, (const __nv_bfloat16 *)Bt, K, N, D);
    CCX_LAUNCHED(h);
    return CCX_OK;
}

int ccx_debug_umma_gemm(ccx_handle *h, const void *A, const void *Bt, int32_t K, int32_t N, float *D)
{
    if (!h || !A || !Bt || !D || K % 16 || K < 16 || K > 512 || N % 16 || N < 16 || N > 64) return CCX_ERR_ARG;
    size_t smem = umma::op_bytes(128, K) + umma::op_bytes(N, K);
    CCX_CUDA(h, cudaFuncSetAttribute(k_umma_selftest, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_umma_selftest<<<1, 128, smem, h->stream>>>((const __nv_bfloat16 *)A, (const __nv_bfloat16 *)Bt, K, N, D);
    CCX_LAUNCHED(h);
    return CCX_OK;
}

}  // extern "C"

// =====================================================================================================
// Tensor-core forward pass (model.py:58-145).  Weight blobs (built by model.py pack_weights_tc):
//   16-bit operand blob, every matrix stored TRANSPOSED [N][K + 16] in the UMMA K-major core-matrix layout; the 16
//   extra K columns carry the layer's bias as (hi, lo, 0, ...) so that one more MMA against a constant "ones" operand
//   adds it inside the tensor core (hi + lo of a 16-bit split: the bias keeps ~22 bits):
//     CONV1 (N64,K80) | HEADS (N32,K80: 16 policy-conv cols, value-conv col, zeros) |
//     9 x [A (N32,K80) | B (N32,K304) | C (N64,K48)] | policy dense: 2 N-halves x [K 0..207 (N160,K208) | K 208..399 (N160,K192)]
//   fp32 blob: conv1_b[64] heads_b[32] 9 x (a_b[32] b_b[32] c_b[64]) pold_b[320] d1_w[25][32] d1_b[32] vh_w[32] vh_b[1]
//   (the trunk kernel reads only the value-head dense from it; the policy dense kernel reads pold_b)
namespace tcl {
constexpr int KB = 16;                                         // bias columns appended to every trunk operand
constexpr int B_CONV1 = 64 * (64 + KB) * 2, B_HEADS = 32 * (64 + KB) * 2;
constexpr int B_A = 32 * (64 + KB) * 2, B_B = 32 * (288 + KB) * 2, B_C = 64 * (32 + KB) * 2;
constexpr int W_CONV1 = 0, W_HEADS = B_CONV1, W_BLOCK0 = W_HEADS + B_HEADS, W_BLOCK = B_A + B_B + B_C;
constexpr int W_BA = 0, W_BB = B_A, W_BC = B_A + B_B;
constexpr int W_POLD = W_BLOCK0 + 9 * W_BLOCK;
constexpr int POLD_C0 = 160 * 208 * 2, POLD_C1 = 160 * 192 * 2, POLD_HALF = POLD_C0 + POLD_C1;
constexpr int W_TOTAL = W_POLD + 2 * POLD_HALF;
constexpr int F_CONV1 = 0, F_HEADS = 64, F_BLOCK0 = 96, F_BLOCK = 128, F_POLD = F_BLOCK0 + 9 * F_BLOCK;
constexpr int F_D1W = F_POLD + 320, F_D1B = F_D1W + 800, F_VHW = F_D1B + 32, F_VHB = F_VHW + 32, F_TOTAL = F_VHB + 1;
}  // namespace tcl

struct ccx_net_tc {
    uint8_t *wb = nullptr;      // bf16 operand blob
    float *fb = nullptr;        // fp32 biases + value-head dense
    __nv_bfloat16 *polc = nullptr;   // policy-conv activations between the two kernels: 128-position tiles in the dense kernel's operand layout (pd3)
    int64_t cap = 0;
    int fp16 = 0;               // 0 = bf16 operands, 1 = IEEE half operands (same kernels, other instruction descriptor)
};


// two fp32 -> one 32-bit word of 16-bit operands: bf16 (FP16 = false) or IEEE half (FP16 = true)
template <bool FP16> __device__ __forceinline__ uint32_t pack2(float a, float b)
{
    if (FP16) { __half2 h = __floats2half2_rn(a, b); return *reinterpret_cast<uint32_t *>(&h); }
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t *>(&h);
}

// ReLU after the 16-bit pack: round(max(x, 0)) == max(round(x), 0) bit for bit (rounding is monotonic and keeps the sign),
// and one packed max handles two values
template <bool FP16> __device__ __forceinline__ uint32_t relu_pack2(float a, float b)
{
    uint32_t p = pack2<FP16>(a, b), r;
    if (FP16) asm("max.f16x2 %0, %1, %2;" : "=r"(r) : "r"(p), "r"(0u));
    else asm("max.bf16x2 %0, %1, %2;" : "=r"(r) : "r"(p), "r"(0u));
    return r;
}


// layout of the policy-conv activations handed from the trunk kernel to the policy dense kernel (see k_policy_dense_tc3)
namespace pd3 {
constexpr int NQ = 80;
constexpr int A0_B = 128 * 208 * 2, A1_B = 128 * 192 * 2, TILE_B = A0_B + A1_B;        // 102,400 B per 128 positions
constexpr int W0_B = NQ * 208 * 2, W1_B = NQ * 192 * 2;
constexpr int S_A0 = 0, S_A1 = S_A0 + A0_B, S_W0 = S_A1 + A1_B, S_W1 = S_W0 + W0_B;
constexpr int S_TOTAL = S_W1 + W1_B;                    // 166,400 B
constexpr int OUT_LD = NQ + 1;                          // fp32 staging [128][81] over the A region once the MMAs are done
static_assert(128 * OUT_LD * 4 <= S_W0, "staging fits in the A region");
}  // namespace pd3

// =====================================================================================================
// Trunk kernel v4 = v3 with the 1x1 convs' A operands and the residual stream moved into TENSOR MEMORY:
//  * the fp32 residual x lives in TMEM columns [0,64): conv C accumulates straight onto it (D += m2 * Wc with
//    D = x), its epilogue applies bias + ReLU in place and writes the 16-bit copy of x that conv A of the next
//    block reads — also in TMEM (columns [64,96), two channels per column, tcgen05.mma "ts" form).  conv B's
//    output goes the same way to conv C (columns [64,80)).  Only the 3x3 conv still reads its A operand from
//    shared memory (the three row-shifted copies), so a block's tensor-core operand traffic out of shared
//    memory drops from 122 KB to 98 KB per tile and two of its three epilogues need no shared-memory store and
//    no generic->async proxy fence;
//  * no residual registers and no [128 x 64] shared operand: 70 KB of shared memory, <= 85 registers,
//    128 TMEM columns per CTA -> THREE CTAs (24 warps) per SM instead of two.
//  * biases are added by the tensor core: every weight operand carries 16 extra K columns (bias hi, bias lo, zeros) and
//    each layer issues one more MMA against a constant [128 x 16] "ones" operand, so the epilogues are ReLU + pack only.
// TMEM columns: X fp32 [0,64) | XB: 16-bit x [64,96), reused as M2B: 16-bit conv-B output [64,80) |
//               AO: conv A / conv B / heads accumulator [96,128).
// Tried and dropped (r01f, both bit-identical to v4; the code is in the history, commit "Experiment: trunk v5 ... v6"):
//  * v5: two tiles in flight per CTA, the same 256 threads running one tile's epilogue while the other's MMAs execute
//    (256 TMEM columns, 101 KB, two CTAs = four tiles per SM): 1.27 ms per 65,536 positions against 1.00 ms — the epilogues of
//    the two tiles serialise on the same threads, and the MMA latency they were meant to hide is only ~0.2 of an epilogue;
//  * v6: the same with two independent 256-thread contexts per CTA (named barriers, weight slots shared and refilled by the
//    second context to finish a layer, 64 registers): 0.971 ms per 65,536 (+2.7 %), 90.0 us against 85.6 us per 4,096 and
//    19.2 ms against 18.3 ms per self-play ply.  Four tiles per SM instead of three buy nothing: the tile rate is not set by
//    per-tile latency with idle resources but by what the tiles share on the SM (shared-memory operand traffic of the N = 32
//    MMAs and the epilogues' TMEM / shared-memory round trips).
namespace tc4 {
constexpr int THREADS = 256, POS = 4, POS_ROWS = 30, LIVE_ROWS = 120;
constexpr int YROWS = 130, Y_LBO = YROWS * 16, Y_COPY = 4 * Y_LBO;        // 1 guard row + 128 + 1 guard row
constexpr int T_X = 0, T_XB = 64, T_AO = 96;
constexpr int S_Y = 0;
constexpr int S_WC1 = S_Y + 3 * Y_COPY;                  // conv1 weights, resident
constexpr int S_WA = S_WC1 + tcl::B_CONV1, S_WB = S_WA + tcl::B_A, S_WC = S_WB + tcl::B_B;      // streamed per layer (A slot also: heads)
constexpr int S_ONES = S_WC + tcl::B_C;                  // [128 x 16] operand, columns 0 and 1 = 1.0: multiplies the bias columns
constexpr int S_F = S_ONES + 128 * 16 * 2;               // value-head dense: floats [F_D1W, F_TOTAL)
constexpr int NF = tcl::F_TOTAL - tcl::F_D1W;
constexpr int F_BYTES = ((NF * 4 + 15) / 16) * 16;
constexpr int FO_D1W = 0, FO_D1B = FO_D1W + 800, FO_VHW = FO_D1B + 32, FO_VHB = FO_VHW + 32;
constexpr int S_PLANES = S_F + F_BYTES;
constexpr int S_VALC = S_PLANES + 1376;
constexpr int S_TOTAL = S_VALC + 512;
static_assert(S_TOTAL <= 74 * 1024, "three CTAs per SM");
static_assert(S_WC1 % 128 == 0 && S_WA % 128 == 0 && S_WB % 128 == 0 && S_WC % 128 == 0 && S_ONES % 128 == 0 && S_F % 16 == 0 &&
              S_PLANES % 16 == 0, "alignment");
}  // namespace tc4

// COUNTED: a compacted batch (count != NULL), a separate instantiation so that the uncounted one keeps n in the parameter bank
template <bool FP16, bool COUNTED = false>
__global__ void __launch_bounds__(tc4::THREADS, 3)
k_net_trunk_tc4(const uint8_t *__restrict__ wb, const float *__restrict__ fb, const uint8_t *__restrict__ planes, int64_t n,
                __nv_bfloat16 *__restrict__ polc, float *__restrict__ value, const int32_t *__restrict__ count)
{
    using namespace tc4;
    if constexpr (COUNTED) {
        n = min(n, (int64_t)*count);                 // the row count on the device, capped by the host's capacity
        if ((int64_t)blockIdx.x * POS >= n) return;  // no tile for this CTA
    }
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ uint64_t bar, barW[4];                // MMAs of a phase done; weight slots A, B, C and conv1 landed
    __shared__ uint32_t tmem_slot;
    const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
    const int rg = warp & 3, h = warp >> 2;                  // TMEM lane group, column half
    const int r = rg * 32 + lane;                            // operand row of this thread
    const int p_local = r / POS_ROWS, rem = r % POS_ROWS, cy = rem / 6, cx = rem % 6;
    const bool live = r < LIVE_ROWS && cx < 5;
    const int cell = cy * 5 + cx;
    const uint32_t sbase = umma::smem_u32(smem);
    const float *sF = reinterpret_cast<const float *>(smem + S_F);
    const int64_t n_tiles = (n + POS - 1) / POS;
    const bool planes_aligned = (reinterpret_cast<uintptr_t>(planes) & 3) == 0;

    // weight slots are refilled by ONE lane with a bulk copy (TMA engine); only the MMA-issuing lane ever waits for them
    auto refill_slot = [&](int slot, int dst, const uint8_t *src, uint32_t bytes) {
        umma::mbar_expect_tx(&barW[slot], bytes);
        umma::bulk_g2s(sbase + dst, src, bytes, &barW[slot]);
    };
    // words t and 256 + t (< 343) of a tile's input planes; bytes past the last position read as zero
    auto load_planes = [&](int64_t tile, uint32_t (&w)[2]) {
        const int bytes = (int)min((int64_t)POS, n - tile * POS) * 343;
        const uint8_t *src = planes + tile * (POS * 343);
        w[0] = 0u; w[1] = 0u;
        if (bytes == POS * 343 && planes_aligned) {
            w[0] = __ldg(reinterpret_cast<const uint32_t *>(src) + t);
            if (t < 343 - THREADS) w[1] = __ldg(reinterpret_cast<const uint32_t *>(src) + THREADS + t);
        } else {
#pragma unroll
            for (int q = 0; q < 2; q++)
                for (int k = 0; k < 4; k++) {
                    const int byte = (q * THREADS + t) * 4 + k;
                    if (byte < bytes) w[q] |= (uint32_t)__ldg(src + byte) << (8 * k);
                }
        }
    };
    auto store_planes = [&](const uint32_t (&w)[2]) {
#pragma unroll
        for (int q = 0; q < 2; q++) {
            const int idx = q * THREADS + t;
            if (idx < 344) reinterpret_cast<uint32_t *>(smem + S_PLANES)[idx] = w[q];
        }
    };

    for (int i = t; i < S_WC1 / 16; i += THREADS) reinterpret_cast<uint4 *>(smem)[i] = make_uint4(0, 0, 0, 0);   // guard rows stay zero
    for (int i = t; i < NF; i += THREADS) reinterpret_cast<float *>(smem + S_F)[i] = __ldg(fb + tcl::F_D1W + i);
    for (int i = t; i < 128 * 2; i += THREADS) {             // ones operand: row r, columns (0,1) = (1,1), the rest 0 (standard layout, K = 16)
        const int r = i >> 1, chunk = i & 1;                 // chunk = which 8-column core matrix of the row
        *reinterpret_cast<uint4 *>(smem + S_ONES + umma::op_offset(r, chunk * 8, 16)) = make_uint4(chunk == 0 ? pack2<FP16>(1.f, 1.f) : 0u, 0u, 0u, 0u);
    }
    {
        uint32_t w0[2];
        load_planes(blockIdx.x, w0);
        store_planes(w0);
    }
    if (t == 0) {
        umma::mbar_init(&bar, 1);
#pragma unroll
        for (int q = 0; q < 4; q++) umma::mbar_init(&barW[q], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        refill_slot(3, S_WC1, wb + tcl::W_CONV1, tcl::B_CONV1);
        refill_slot(0, S_WA, wb + tcl::W_BLOCK0 + tcl::W_BA, tcl::B_A);
        refill_slot(1, S_WB, wb + tcl::W_BLOCK0 + tcl::W_BB, tcl::B_B);
        refill_slot(2, S_WC, wb + tcl::W_BLOCK0 + tcl::W_BC, tcl::B_C);
    }
    if (warp == 0) umma::tmem_alloc(&tmem_slot, 128);
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    uint32_t phW0 = 0, phW1 = 0, phW2 = 0;           // parities of the weight-slot barriers (tracked by the issuing lane)
    bool conv1_ready = false;
    const uint32_t tmem = tmem_slot;
    const uint32_t trow = tmem + ((uint32_t)(rg * 32) << 16);
    uint32_t phase = 0;
    const umma::DescBase dY = umma::desc_base(sbase + S_Y, Y_LBO, 128u);
    const umma::DescBase dWC1 = umma::desc_base(sbase + S_WC1, 128u, (64 + tcl::KB) / 8 * 128u), dWA = umma::desc_base(sbase + S_WA, 128u, (64 + tcl::KB) / 8 * 128u);
    const umma::DescBase dWB = umma::desc_base(sbase + S_WB, 128u, (288 + tcl::KB) / 8 * 128u), dWC = umma::desc_base(sbase + S_WC, 128u, (32 + tcl::KB) / 8 * 128u);
    const umma::DescBase dONES = umma::desc_base(sbase + S_ONES, 128u, 16 / 8 * 128u);
    constexpr uint32_t ID32 = umma::make_idesc(32, FP16), ID64 = umma::make_idesc(64, FP16);

    // operands written to TMEM: make the stores visible to the tensor core, then the CTA barrier
    auto tmem_sync = [&]() {
        umma::tmem_wait_st();
        umma::fence_before_sync();
        __syncthreads();
    };
    // operands written to shared memory (conv A's output copies)
    auto smem_sync = [&]() {
        umma::fence_async_smem();
        umma::fence_before_sync();
        __syncthreads();
    };
    auto wait_mma = [&]() {
        umma::mbar_wait(&bar, phase); phase ^= 1;
        umma::fence_after_sync();
    };
    auto pack8 = [&](const float *rr) {
        return make_uint4(pack2<FP16>(rr[0], rr[1]), pack2<FP16>(rr[2], rr[3]), pack2<FP16>(rr[4], rr[5]), pack2<FP16>(rr[6], rr[7]));
    };
    // this thread's 32 residual columns: ReLU in place in TMEM X (fp32) and the 16-bit copy XB, 16 columns at a time
    auto finish_x = [&]() {
#pragma unroll
        for (int half = 0; half < 2; half++) {
            float v[16];
            umma::tmem_ld16(trow + T_X + h * 32 + half * 16, v);
            uint32_t f[16], pk[8];
#pragma unroll
            for (int j = 0; j < 16; j++) { v[j] = fmaxf(v[j], 0.f); f[j] = __float_as_uint(v[j]); }
#pragma unroll
            for (int j = 0; j < 8; j++) pk[j] = pack2<FP16>(v[2 * j], v[2 * j + 1]);
            umma::tmem_st16(trow + T_X + h * 32 + half * 16, f);
            umma::tmem_st8(trow + T_XB + h * 16 + half * 8, pk);
        }
    };
    // bias MMA of a layer: D (+)= ones[128 x 16] * W[., K .. K+16)^T  (columns K, K+1 of the weight operand = bias hi, lo)
    auto bias_mma = [&](uint32_t tmem_d, umma::DescBase w, int K, uint32_t idesc, bool accumulate) {
        umma::mma_bf16(tmem_d, umma::desc_at(dONES, 0u), umma::desc_at(w, (uint32_t)(K / 8) * 128u), idesc, accumulate);
    };

    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t pos0 = tile * POS;
        const int n_pos = (int)min((int64_t)POS, n - pos0);
        uint32_t pw[2] = {0u, 0u};
        if (tile + gridDim.x < n_tiles) load_planes(tile + gridDim.x, pw);       // lands while this tile computes
        // ---- conv1 operand: im2col of the 3x3 'valid' window, K = 63 (+1 zero) (model.py:62), packed into TMEM XB
        {
            const uint8_t *pl = smem + S_PLANES + (live ? p_local * 343 : 0);
#pragma unroll
            for (int c8 = 0; c8 < 2; c8++) {
                uint32_t pk[8];
#pragma unroll
                for (int q = 0; q < 8; q++) {
                    float v2[2];
#pragma unroll
                    for (int e = 0; e < 2; e++) {
                        const int kk = h * 32 + c8 * 16 + q * 2 + e;
                        const int tap = kk / 7, ch = kk % 7, dy = tap / 3, dx = tap % 3;
                        v2[e] = (live && kk < 63) ? (float)pl[((cy + dy) * 7 + (cx + dx)) * 7 + ch] : 0.f;
                    }
                    pk[q] = pack2<FP16>(v2[0], v2[1]);
                }
                umma::tmem_st8(trow + T_XB + h * 16 + c8 * 8, pk);
            }
        }
        tmem_sync();
        if (warp == 0) {
            umma::fence_after_sync();
            if (umma::elect_one()) {
                if (!conv1_ready) { umma::mbar_wait(&barW[3], 0); conv1_ready = true; }
                bias_mma(tmem + T_X, dWC1, 64, ID64, false);
                umma::gemm_issue_ts<64>(tmem + T_X, tmem + T_XB, dWC1, 0, ID64, true);
                umma::commit(&bar);
            }
            __syncwarp();
        }
        wait_mma();
        finish_x();
        // ---- 9 bottleneck residual blocks (model.py:120-145) --------------------------------------------------
        for (int b = 0; b < 9; b++) {
            const uint8_t *wnext = wb + tcl::W_BLOCK0 + ((b + 1) % 9) * tcl::W_BLOCK;
            // A: 1x1 conv 64 -> 32, ReLU; A operand = XB in TMEM
            tmem_sync();
            if (warp == 0) {
                umma::fence_after_sync();
                if (umma::elect_one()) {
                    umma::mbar_wait(&barW[0], phW0); phW0 ^= 1;
                    bias_mma(tmem + T_AO, dWA, 64, ID32, false);
                    umma::gemm_issue_ts<64>(tmem + T_AO, tmem + T_XB, dWA, 0, ID32, true);
                    umma::commit(&bar);
                }
                __syncwarp();
            }
            wait_mma();
            if (warp == 0 && umma::elect_one()) refill_slot(0, S_WA, b < 8 ? wnext + tcl::W_BA : wb + tcl::W_HEADS, tcl::B_A);
            {
                float v[16];
                umma::tmem_ld16(trow + T_AO + h * 16, v);
                const uint4 o0 = make_uint4(relu_pack2<FP16>(v[0], v[1]), relu_pack2<FP16>(v[2], v[3]), relu_pack2<FP16>(v[4], v[5]), relu_pack2<FP16>(v[6], v[7]));
                const uint4 o1 = make_uint4(relu_pack2<FP16>(v[8], v[9]), relu_pack2<FP16>(v[10], v[11]), relu_pack2<FP16>(v[12], v[13]), relu_pack2<FP16>(v[14], v[15]));
                if (live) {
                    // copy d serves kernel row dy = d - 1: output cell (y - dy, x) reads this cell, so the value goes to row r - 6*dy
#pragma unroll
                    for (int d = 0; d < 3; d++) {
                        const int oy = cy - (d - 1);
                        if (oy >= 0 && oy <= 4) {
                            uint8_t *dst = smem + S_Y + d * Y_COPY + (2 * h) * Y_LBO + (1 + r - 6 * (d - 1)) * 16;
                            *reinterpret_cast<uint4 *>(dst) = o0;
                            *reinterpret_cast<uint4 *>(dst + Y_LBO) = o1;
                        }
                    }
                }
            }
            // B: 3x3 'same' conv 32 -> 32 = nine accumulating K = 32 GEMMs on row-shifted views of the three copies
            smem_sync();
            if (warp == 0) {
                umma::fence_after_sync();
                if (umma::elect_one()) {
                    umma::mbar_wait(&barW[1], phW1); phW1 ^= 1;
                    bias_mma(tmem + T_AO, dWB, 288, ID32, false);
#pragma unroll
                    for (int d = 0; d < 3; d++)
#pragma unroll
                        for (int dxi = 0; dxi < 3; dxi++)
#pragma unroll
                            for (int ks = 0; ks < 2; ks++)
                                umma::mma_bf16(tmem + T_AO, umma::desc_at(dY, (uint32_t)(d * Y_COPY + dxi * 16 + 2 * ks * Y_LBO)),
                                               umma::desc_at(dWB, (uint32_t)(((d * 3 + dxi) * 32 / 8 + 2 * ks) * 128)), ID32, true);
                    umma::commit(&bar);
                }
                __syncwarp();
            }
            wait_mma();
            if (warp == 0 && umma::elect_one()) refill_slot(1, S_WB, wnext + tcl::W_BB, tcl::B_B);
            {
                float v[16];
                umma::tmem_ld16(trow + T_AO + h * 16, v);
                uint32_t pk[8];
#pragma unroll
                for (int q = 0; q < 8; q++)
                    pk[q] = relu_pack2<FP16>(v[2 * q], v[2 * q + 1]);
                umma::tmem_st8(trow + T_XB + h * 8, pk);         // M2B: 32 channels = 16 columns
            }
            // C: 1x1 conv 32 -> 64 accumulated onto the residual (model.py:137-144): X += M2B * Wc, then bias + ReLU in place
            tmem_sync();
            if (warp == 0) {
                umma::fence_after_sync();
                if (umma::elect_one()) {
                    umma::mbar_wait(&barW[2], phW2); phW2 ^= 1;
                    bias_mma(tmem + T_X, dWC, 32, ID64, true);
                    umma::gemm_issue_ts<32>(tmem + T_X, tmem + T_XB, dWC, 0, ID64, true);
                    umma::commit(&bar);
                }
                __syncwarp();
            }
            wait_mma();
            if (warp == 0 && umma::elect_one()) refill_slot(2, S_WC, wnext + tcl::W_BC, tcl::B_C);
            finish_x();
        }
        // ---- heads: policy conv 64 -> 16 and value conv 64 -> 1 in one N = 32 GEMM (model.py:91, 108); weights in the A slot
        tmem_sync();
        if (warp == 0) {
            umma::fence_after_sync();
            if (umma::elect_one()) {
                umma::mbar_wait(&barW[0], phW0); phW0 ^= 1;
                bias_mma(tmem + T_AO, dWA, 64, ID32, false);
                umma::gemm_issue_ts<64>(tmem + T_AO, tmem + T_XB, dWA, 0, ID32, true);
                umma::commit(&bar);
            }
            __syncwarp();
        }
        wait_mma();
        if (warp == 0 && umma::elect_one()) refill_slot(0, S_WA, wb + tcl::W_BLOCK0 + tcl::W_BA, tcl::B_A);   // conv A of block 0 for the next tile
        {
            float v[16];
            umma::tmem_ld16(trow + T_AO + h * 16, v);
            if (live && p_local < n_pos) {
                if (h == 0) {
#pragma unroll
                    for (int q = 0; q < 16; q++) v[q] = fmaxf(v[q], 0.f);
                    // Flatten in (y, x, c) order = K index cell * 16 + c, stored straight in the policy dense kernel's A-operand
                    // layout: 128-position tiles, each [K 0..207 | K 208..399] in the UMMA core-matrix layout, so that kernel
                    // fetches a tile with two bulk copies
                    const int64_t pos = pos0 + p_local;
                    const int k = cell * 16, chunk = k >= 208, kk = k - chunk * 208;
                    uint8_t *dst = reinterpret_cast<uint8_t *>(polc) + (pos >> 7) * pd3::TILE_B + (chunk ? pd3::A0_B : 0) +
                                   umma::op_offset((int)(pos & 127), kk, chunk ? 192 : 208);
                    *reinterpret_cast<uint4 *>(dst) = pack8(v);
                    *reinterpret_cast<uint4 *>(dst + 128) = pack8(v + 8);
                } else {
                    reinterpret_cast<float *>(smem + S_VALC)[p_local * 25 + cell] = fmaxf(v[0], 0.f);
                }
            }
        }
        store_planes(pw);
        umma::fence_before_sync();
        __syncthreads();
        // ---- value head: dense_1 25 -> 32 ReLU, value_head 32 -> 1 tanh (model.py:95-103), fp32 ---------------------
        if (warp < n_pos) {
            const float *valc = reinterpret_cast<const float *>(smem + S_VALC) + warp * 25;
            float acc = sF[FO_D1B + lane];
            for (int k = 0; k < 25; k++) acc = fmaf(valc[k], sF[FO_D1W + k * 32 + lane], acc);
            float sv = fmaxf(acc, 0.f) * sF[FO_VHW + lane];
#pragma unroll
            for (int off = 16; off; off >>= 1) sv += __shfl_xor_sync(0xFFFFFFFFu, sv, off);
            if (lane == 0) value[pos0 + warp] = tanhf(sv + sF[FO_VHB]);
        }
    }
    // the last refills (block 0's weights for a tile that never comes) must land before the CTA's shared memory is released
    if (warp == 0 && umma::elect_one()) {
        umma::mbar_wait(&barW[0], phW0); umma::mbar_wait(&barW[1], phW1); umma::mbar_wait(&barW[2], phW2);
        if (!conv1_ready) umma::mbar_wait(&barW[3], 0);
    }
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 0) umma::tmem_free(tmem, 128);
}

// Policy dense v3: logits[B x 294] = flat(policy conv)[B x 400] * W + b as 128-position x 80-output tiles (grid = row tiles x
// 4 column quarters: 128 CTAs at the self-play batch of 4,096).  Both operands of a tile arrive as FOUR bulk copies issued by
// one thread (the trunk kernel already wrote the activations in the operand layout; the quarter's weight rows are a contiguous
// slice of the blob) — v2 spent ~3 K instructions per thread on 16-byte cp.async address arithmetic, 12 us per launch.
// The K chunks land on two mbarriers, so the first chunk's MMAs run while the second is in flight; logits are staged through
// shared memory for coalesced stores.
template <bool FP16>
__global__ void __launch_bounds__(128, 1)
k_policy_dense_tc3(const uint8_t *__restrict__ wb, const float *__restrict__ fb, const uint8_t *__restrict__ polc, int64_t n,
                   float *__restrict__ logits, const int32_t *__restrict__ count)
{
    using namespace pd3;
    if (count) n = min(n, (int64_t)*count);        // compacted batch: the row count on the device, capped by the host's capacity
    if ((int64_t)blockIdx.x * 128 >= n) return;      // past the last row (only with a count)
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ uint64_t bar, barL[2];
    __shared__ uint32_t tmem_slot;
    const int t = threadIdx.x, warp = t >> 5;
    const int quarter = blockIdx.y, half = quarter >> 1, c0 = (quarter & 1) * NQ;
    const int64_t row0 = (int64_t)blockIdx.x * 128;
    const uint32_t sbase = umma::smem_u32(smem);
    if (t == 0) {
        umma::mbar_init(&bar, 1); umma::mbar_init(&barL[0], 1); umma::mbar_init(&barL[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        const uint8_t *a = polc + (int64_t)blockIdx.x * TILE_B;
        // this quarter's 80 weight rows are a contiguous slice of the half's [160 x Kc] operand
        const uint8_t *w0 = wb + tcl::W_POLD + half * tcl::POLD_HALF + (c0 / 8) * (208 / 8) * 128;
        const uint8_t *w1 = wb + tcl::W_POLD + half * tcl::POLD_HALF + tcl::POLD_C0 + (c0 / 8) * (192 / 8) * 128;
        umma::mbar_expect_tx(&barL[0], A0_B + W0_B);
        umma::bulk_g2s(sbase + S_A0, a, A0_B, &barL[0]);
        umma::bulk_g2s(sbase + S_W0, w0, W0_B, &barL[0]);
        umma::mbar_expect_tx(&barL[1], A1_B + W1_B);
        umma::bulk_g2s(sbase + S_A1, a + A0_B, A1_B, &barL[1]);
        umma::bulk_g2s(sbase + S_W1, w1, W1_B, &barL[1]);
    }
    if (warp == 0) umma::tmem_alloc(&tmem_slot, 128);
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = tmem_slot;
    constexpr uint32_t ID = umma::make_idesc(NQ, FP16);
    if (warp == 0) {
        if (umma::elect_one()) {
            umma::mbar_wait(&barL[0], 0);
            umma::gemm_issue_d<208>(tmem, umma::desc_base(sbase + S_A0, 128u, 208 / 8 * 128u), 0, umma::desc_base(sbase + S_W0, 128u, 208 / 8 * 128u), 0, ID, false);
            umma::mbar_wait(&barL[1], 0);
            umma::gemm_issue_d<192>(tmem, umma::desc_base(sbase + S_A1, 128u, 192 / 8 * 128u), 0, umma::desc_base(sbase + S_W1, 128u, 192 / 8 * 128u), 0, ID, true);
            umma::commit(&bar);
        }
        __syncwarp();
    }
    umma::mbar_wait(&bar, 0);
    umma::fence_after_sync();
    float *stage = reinterpret_cast<float *>(smem);
#pragma unroll
    for (int c = 0; c < NQ; c += 16) {
        float v[16];
        umma::tmem_ld16(tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)c, v);
#pragma unroll
        for (int j = 0; j < 16; j++) stage[t * OUT_LD + c + j] = v[j];
    }
    umma::fence_before_sync();
    __syncthreads();
    const int col_base = half * 160 + c0;
    for (int i = t; i < 128 * NQ; i += 128) {
        const int r = i / NQ, c = i % NQ, col = col_base + c;
        if (row0 + r < n && col < CCX_NUM_ACTIONS) logits[(row0 + r) * CCX_NUM_ACTIONS + col] = stage[r * OUT_LD + c] + __ldg(fb + tcl::F_POLD + col);
    }
    if (warp == 0) umma::tmem_free(tmem, 128);
}

static ccx_net_tc *tc_of(ccx_handle *h, bool create)
{
    if (!h->net_tc && create) h->net_tc = new (std::nothrow) ccx_net_tc();
    return h->net_tc;
}

void ccx_net_tc_free(ccx_handle *h)
{
    ccx_net_tc *tc = h->net_tc;
    if (!tc) return;
    cudaFree(tc->wb); cudaFree(tc->fb); cudaFree(tc->polc);
    delete tc;
    h->net_tc = nullptr;
}

extern "C" {

int ccx_net_tc_blob_bytes(void) { return tcl::W_TOTAL; }
int ccx_net_tc_num_floats(void) { return tcl::F_TOTAL; }

int ccx_net_load_tc(ccx_handle *h, const void *bf16_blob_host, int64_t blob_bytes, const float *f32_host, int64_t n_floats,
                    int32_t fp16)
{
    if (!h || !bf16_blob_host || !f32_host || blob_bytes != tcl::W_TOTAL || n_floats != tcl::F_TOTAL || (fp16 != 0 && fp16 != 1))
        return CCX_ERR_ARG;
    ccx_net_tc *tc = tc_of(h, true);
    if (!tc) return CCX_ERR_NOMEM;
    h->epoch++;
    h->pool_gen++;
    if (!tc->wb) CCX_CUDA(h, cudaMalloc(&tc->wb, tcl::W_TOTAL));
    if (!tc->fb) CCX_CUDA(h, cudaMalloc(&tc->fb, sizeof(float) * tcl::F_TOTAL));
    CCX_CUDA(h, cudaMemcpyAsync(tc->wb, bf16_blob_host, tcl::W_TOTAL, cudaMemcpyHostToDevice, h->stream));
    CCX_CUDA(h, cudaMemcpyAsync(tc->fb, f32_host, sizeof(float) * tcl::F_TOTAL, cudaMemcpyHostToDevice, h->stream));
    CCX_CUDA(h, cudaStreamSynchronize(h->stream));
    tc->fp16 = fp16;
    CCX_CUDA(h, cudaFuncSetAttribute(k_policy_dense_tc3<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, pd3::S_TOTAL));
    CCX_CUDA(h, cudaFuncSetAttribute(k_policy_dense_tc3<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, pd3::S_TOTAL));
    CCX_CUDA(h, cudaFuncSetAttribute(k_net_trunk_tc4<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc4::S_TOTAL));
    CCX_CUDA(h, cudaFuncSetAttribute(k_net_trunk_tc4<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc4::S_TOTAL));
    CCX_CUDA(h, cudaFuncSetAttribute(k_net_trunk_tc4<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc4::S_TOTAL));
    CCX_CUDA(h, cudaFuncSetAttribute(k_net_trunk_tc4<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc4::S_TOTAL));
    return CCX_OK;
}

// planes: uint8 (n,7,7,7) on the device -> logits float32[n][294], value float32[n]
int ccx_net_forward_tc(ccx_handle *h, int64_t n, const uint8_t *planes, float *logits, float *value)
{
    if (!h || n < 0 || (n && (!planes || !logits || !value))) return CCX_ERR_ARG;
    if (n == 0) return tc_of(h, false) && tc_of(h, false)->wb ? CCX_OK : CCX_ERR_STATE;
    return ccx_net_forward_tc_on(h, h->stream, n, 0, n, planes, logits, value);
}

}  // extern "C"

// planes / logits / value point at the FIRST of the n rows to evaluate; row0 only selects the rows of the internal
// policy-conv scratch (so two halves of a batch can be in flight on two streams)
int ccx_net_forward_tc_on(ccx_handle *h, cudaStream_t stream, int64_t cap, int64_t row0, int64_t n, const uint8_t *planes, float *logits,
                          float *value, const int32_t *count)
{
    ccx_net_tc *tc = tc_of(h, false);
    if (!tc || !tc->wb) return CCX_ERR_STATE;
    if (tc->cap < cap) {
        h->epoch++;
        CCX_CUDA(h, cudaDeviceSynchronize());          // another stream may still read the old scratch
        if (tc->polc) CCX_CUDA(h, cudaFree(tc->polc));
        tc->polc = nullptr; tc->cap = 0;
        const size_t bytes = (size_t)((cap + 127) / 128) * pd3::TILE_B;         // whole 128-position tiles
        CCX_CUDA(h, cudaMalloc(&tc->polc, bytes));
        CCX_CUDA(h, cudaMemsetAsync(tc->polc, 0, bytes, stream));                  // rows past n of the last tile stay finite
        tc->cap = cap;
    }
    if (n == 0) return CCX_OK;                         // (a call with n = 0 only reserves the scratch)
    if (row0 % 128) return CCX_ERR_ARG;
    __nv_bfloat16 *polc = reinterpret_cast<__nv_bfloat16 *>(reinterpret_cast<uint8_t *>(tc->polc) + (row0 / 128) * pd3::TILE_B);
    {
        int64_t tiles = (n + tc4::POS - 1) / tc4::POS;
        unsigned grid = (unsigned)(tiles < 3 * h->num_sms ? tiles : 3 * h->num_sms);     // three resident CTAs per SM
#define CCX_TC4(F, C) k_net_trunk_tc4<F, C><<<grid, tc4::THREADS, tc4::S_TOTAL, stream>>>(tc->wb, tc->fb, planes, n, polc, value, count)
        if (tc->fp16) { if (count) CCX_TC4(true, true); else CCX_TC4(true, false); }
        else { if (count) CCX_TC4(false, true); else CCX_TC4(false, false); }
#undef CCX_TC4
    }
    CCX_LAUNCHED(h);
    {
        dim3 g2((unsigned)((n + 127) / 128), 4);
        if (tc->fp16) k_policy_dense_tc3<true><<<g2, 128, pd3::S_TOTAL, stream>>>(tc->wb, tc->fb, (const uint8_t *)polc, n, logits, count);
        else k_policy_dense_tc3<false><<<g2, 128, pd3::S_TOTAL, stream>>>(tc->wb, tc->fb, (const uint8_t *)polc, n, logits, count);
    }
    CCX_LAUNCHED(h);
    return CCX_OK;
}

// =====================================================================================================
// Accurate tensor-core mode (ccx_net_set_mode(2)): same network, same tile geometry and phase structure as
// k_net_trunk_tc4, but every product is evaluated in split precision — activations a = a_hi + a_lo and weights
// w = w_hi + w_lo, each term an IEEE half — as  a_hi*w_hi + a_lo*w_hi + a_hi*w_lo  accumulated in fp32 by the tensor
// core (the dropped a_lo*w_lo term is ~2^-22 relative).  A 16-bit-operand pass through the 29 layers leaves up to
// 3.2e-3 on the largest probabilities (every layer group contributes: DESIGN.md §3); this mode brings the tensor-core
// path to the fp32 restatement's ~1e-5 at three times the MMAs and twice the operand storage (one CTA per SM).
// Operand blob (model.py pack_weights_acc): per matrix [hi: N x (K+16) with the bias columns][lo: N x K], UMMA layout:
//   CONV1 | HEADS | 9 x [A | B | C] | policy dense (see acl::W_POLD).  Biases of the policy dense come from the fp32 weights (ccx_net_load).
namespace acl {
__host__ __device__ constexpr int hi_b(int N, int K) { return N * (K + 16) * 2; }
__host__ __device__ constexpr int lo_b(int N, int K) { return N * K * 2; }
constexpr int B_CONV1 = hi_b(64, 64) + lo_b(64, 64), B_HEADS = hi_b(32, 64) + lo_b(32, 64);
constexpr int B_A = hi_b(32, 64) + lo_b(32, 64), B_C = hi_b(64, 32) + lo_b(64, 32);
constexpr int B_B = hi_b(64, 288);       // conv B: ONE [64 x 304] operand, rows 0-31 = hi (+ bias columns), rows 32-63 = lo: a_hi * [w_hi | w_lo] is a single N = 64 MMA
constexpr int W_CONV1 = 0, W_HEADS = B_CONV1, W_BLOCK0 = W_HEADS + B_HEADS, W_BLOCK = B_A + B_B + B_C;
constexpr int W_BA = 0, W_BB = B_A, W_BC = B_A + B_B;
constexpr int W_POLD = W_BLOCK0 + 9 * W_BLOCK;                 // policy dense: 2 N-halves x 4 K-chunks (112, 96, 96, 96) x [hi (N160, Kc) | lo (N160, Kc)]
__host__ __device__ constexpr int pd_kc(int c) { return c == 0 ? 112 : 96; }          // multiples of 16 (one MMA = K 16)
__host__ __device__ constexpr int pd_k0(int c) { return c == 0 ? 0 : c == 1 ? 112 : c == 2 ? 208 : 304; }
constexpr int POLD_HALF = 2 * 160 * 400 * 2;
__host__ __device__ constexpr int pd_w_off(int half, int c) { return W_POLD + half * POLD_HALF + 2 * 160 * pd_k0(c) * 2; }   // hi slice; lo follows at + 160*Kc*2
constexpr int W_TOTAL = W_POLD + 2 * POLD_HALF;
constexpr int PD_TILE_B = 128 * 400 * 2;                       // one 128-position tile of policy-conv activations (hi or lo), 4 K-chunks
__host__ __device__ constexpr int pd_a_off(int c) { return 128 * pd_k0(c) * 2; }
constexpr int THREADS = 256, POS = 4, POS_ROWS = 30, LIVE_ROWS = 120;
constexpr int YROWS = 130, Y_LBO = YROWS * 16, Y_COPY = 4 * Y_LBO;
constexpr int T_X = 0, T_XH = 64, T_XL = 96, T_AO = 128;                   // TMEM columns (256 allocated); AO is 64 wide for conv B
constexpr int S_YH = 0, S_YL = S_YH + 3 * Y_COPY;
constexpr int S_WA = S_YL + 3 * Y_COPY, S_WB = S_WA + B_A, S_WC = S_WB + B_B;     // slot B also carries conv1's weights at tile starts
constexpr int S_ONES = S_WC + B_C;
constexpr int S_PLANES = S_ONES + 128 * 16 * 2;
constexpr int S_VALC = S_PLANES + 1376;
constexpr int S_TOTAL = S_VALC + 512;
static_assert(B_CONV1 <= B_B, "conv1's weights fit in slot B");
static_assert(S_TOTAL <= 113 * 1024, "two CTAs per SM");
static_assert(S_YL % 128 == 0 && S_WA % 128 == 0 && S_WB % 128 == 0 && S_WC % 128 == 0 && S_ONES % 128 == 0 && S_PLANES % 16 == 0, "alignment");
}  // namespace acl

// (hi, lo) halves of two fp32 values: hi = round16(x), lo = round16(x - hi)
__device__ __forceinline__ void split2(float a, float b, uint32_t &hi, uint32_t &lo)
{
    __half2 h = __floats2half2_rn(a, b);
    float2 hf = __half22float2(h);
    __half2 l = __floats2half2_rn(a - hf.x, b - hf.y);
    hi = *reinterpret_cast<uint32_t *>(&h);
    lo = *reinterpret_cast<uint32_t *>(&l);
}

__global__ void __launch_bounds__(acl::THREADS, 2)
k_net_trunk_acc(const uint8_t *__restrict__ wb, const float *__restrict__ fb, const uint8_t *__restrict__ planes, int64_t n,
                uint8_t *__restrict__ polc_h, uint8_t *__restrict__ polc_l, float *__restrict__ value, const int32_t *__restrict__ count)
{
    using namespace acl;
    if (count) n = min(n, (int64_t)*count);        // compacted batch: the row count on the device, capped by the host's capacity
    if ((int64_t)blockIdx.x * POS >= n) return;
    constexpr bool FP16 = true;
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ uint64_t bar, barW[4];
    __shared__ uint32_t tmem_slot;
    const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
    const int rg = warp & 3, h = warp >> 2;
    const int r = rg * 32 + lane;
    const int p_local = r / POS_ROWS, rem = r % POS_ROWS, cy = rem / 6, cx = rem % 6;
    const bool live = r < LIVE_ROWS && cx < 5;
    const int cell = cy * 5 + cx;
    const uint32_t sbase = umma::smem_u32(smem);
    const int64_t n_tiles = (n + POS - 1) / POS;

    auto refill_slot = [&](int slot, int dst, const uint8_t *src, uint32_t bytes) {
        umma::mbar_expect_tx(&barW[slot], bytes);
        umma::bulk_g2s(sbase + dst, src, bytes, &barW[slot]);
    };
    auto stage_planes = [&](int64_t tile) {
        const int bytes = (int)min((int64_t)POS, n - tile * POS) * 343;
        const uint8_t *src = planes + tile * (POS * 343);
        for (int i = t; i < POS * 343; i += THREADS) smem[S_PLANES + i] = i < bytes ? __ldg(src + i) : (uint8_t)0;
    };

    for (int i = t; i < S_WA / 16; i += THREADS) reinterpret_cast<uint4 *>(smem)[i] = make_uint4(0, 0, 0, 0);   // guard rows of both copy sets
    for (int i = t; i < 128 * 2; i += THREADS) {
        const int rr = i >> 1, chunk = i & 1;
        *reinterpret_cast<uint4 *>(smem + S_ONES + umma::op_offset(rr, chunk * 8, 16)) = make_uint4(chunk == 0 ? pack2<FP16>(1.f, 1.f) : 0u, 0u, 0u, 0u);
    }
    if (t == 0) {
        umma::mbar_init(&bar, 1);
#pragma unroll
        for (int q = 0; q < 4; q++) umma::mbar_init(&barW[q], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        refill_slot(1, S_WB, wb + W_CONV1, B_CONV1);                     // slot B: conv1 first, conv B of block 0 right after it
        refill_slot(0, S_WA, wb + W_BLOCK0 + W_BA, B_A);
        refill_slot(2, S_WC, wb + W_BLOCK0 + W_BC, B_C);
    }
    if (warp == 0) umma::tmem_alloc(&tmem_slot, 256);
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    uint32_t phW0 = 0, phW1 = 0, phW2 = 0;
    const uint32_t tmem = tmem_slot;
    const uint32_t trow = tmem + ((uint32_t)(rg * 32) << 16);
    uint32_t phase = 0;
    // operand descriptors: hi parts carry the 16 bias columns (K + 16 layout), lo parts follow them in the slot (K layout)
    const umma::DescBase dYH = umma::desc_base(sbase + S_YH, Y_LBO, 128u), dYL = umma::desc_base(sbase + S_YL, Y_LBO, 128u);
    const umma::DescBase dC1H = umma::desc_base(sbase + S_WB, 128u, 80 / 8 * 128u), dC1L = umma::desc_base(sbase + S_WB + hi_b(64, 64), 128u, 64 / 8 * 128u);
    const umma::DescBase dAH = umma::desc_base(sbase + S_WA, 128u, 80 / 8 * 128u), dAL = umma::desc_base(sbase + S_WA + hi_b(32, 64), 128u, 64 / 8 * 128u);
    const umma::DescBase dBH = umma::desc_base(sbase + S_WB, 128u, 304 / 8 * 128u);          // rows 0-31 hi, rows 32-63 lo
    const umma::DescBase dCH = umma::desc_base(sbase + S_WC, 128u, 48 / 8 * 128u), dCL = umma::desc_base(sbase + S_WC + hi_b(64, 32), 128u, 32 / 8 * 128u);
    const umma::DescBase dONES = umma::desc_base(sbase + S_ONES, 128u, 16 / 8 * 128u);
    constexpr uint32_t ID32 = umma::make_idesc(32, FP16), ID64 = umma::make_idesc(64, FP16);

    auto tmem_sync = [&]() { umma::tmem_wait_st(); umma::fence_before_sync(); __syncthreads(); };
    auto smem_sync = [&]() { umma::fence_async_smem(); umma::fence_before_sync(); __syncthreads(); };
    auto wait_mma = [&]() { umma::mbar_wait(&bar, phase); phase ^= 1; umma::fence_after_sync(); };
    auto bias_mma = [&](uint32_t tmem_d, umma::DescBase w, int K, uint32_t idesc, bool accumulate) {
        umma::mma_bf16(tmem_d, umma::desc_at(dONES, 0u), umma::desc_at(w, (uint32_t)(K / 8) * 128u), idesc, accumulate);
    };
    // this thread's 32 residual columns: ReLU in place in TMEM X (fp32) and the split 16-bit copies XH / XL
    auto finish_x = [&]() {
#pragma unroll
        for (int half = 0; half < 2; half++) {
            float v[16];
            umma::tmem_ld16(trow + T_X + h * 32 + half * 16, v);
            uint32_t f[16], ph[8], pl[8];
#pragma unroll
            for (int j = 0; j < 16; j++) { v[j] = fmaxf(v[j], 0.f); f[j] = __float_as_uint(v[j]); }
#pragma unroll
            for (int j = 0; j < 8; j++) split2(v[2 * j], v[2 * j + 1], ph[j], pl[j]);
            umma::tmem_st16(trow + T_X + h * 32 + half * 16, f);
            umma::tmem_st8(trow + T_XH + h * 16 + half * 8, ph);
            umma::tmem_st8(trow + T_XL + h * 16 + half * 8, pl);
        }
    };

    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t pos0 = tile * POS;
        const int n_pos = (int)min((int64_t)POS, n - pos0);
        stage_planes(tile);
        __syncthreads();
        // conv1 operand: the uint8 plane values are exact in half precision, so only the weights are split (a_lo = 0)
        {
            const uint8_t *pl = smem + S_PLANES + (live ? p_local * 343 : 0);
#pragma unroll
            for (int c8 = 0; c8 < 2; c8++) {
                uint32_t pk[8];
#pragma unroll
                for (int q = 0; q < 8; q++) {
                    float v2[2];
#pragma unroll
                    for (int e = 0; e < 2; e++) {
                        const int kk = h * 32 + c8 * 16 + q * 2 + e;
                        const int tap = kk / 7, ch = kk % 7, dy = tap / 3, dx = tap % 3;
                        v2[e] = (live && kk < 63) ? (float)pl[((cy + dy) * 7 + (cx + dx)) * 7 + ch] : 0.f;
                    }
                    pk[q] = pack2<FP16>(v2[0], v2[1]);
                }
                umma::tmem_st8(trow + T_XH + h * 16 + c8 * 8, pk);
            }
        }
        tmem_sync();
        if (warp == 0) {
            umma::fence_after_sync();
            if (umma::elect_one()) {
                umma::mbar_wait(&barW[1], phW1); phW1 ^= 1;
                bias_mma(tmem + T_X, dC1H, 64, ID64, false);
                umma::gemm_issue_ts<64>(tmem + T_X, tmem + T_XH, dC1H, 0, ID64, true);
                umma::gemm_issue_ts<64>(tmem + T_X, tmem + T_XH, dC1L, 0, ID64, true);
                umma::commit(&bar);
            }
            __syncwarp();
        }
        wait_mma();
        if (warp == 0 && umma::elect_one()) refill_slot(1, S_WB, wb + W_BLOCK0 + W_BB, B_B);       // conv B of block 0 (needed two phases from now)
        finish_x();
        for (int b = 0; b < 9; b++) {
            const uint8_t *wnext = wb + W_BLOCK0 + ((b + 1) % 9) * W_BLOCK;
            // A: 1x1 conv 64 -> 32
            tmem_sync();
            if (warp == 0) {
                umma::fence_after_sync();
                if (umma::elect_one()) {
                    umma::mbar_wait(&barW[0], phW0); phW0 ^= 1;
                    bias_mma(tmem + T_AO, dAH, 64, ID32, false);
                    umma::gemm_issue_ts<64>(tmem + T_AO, tmem + T_XH, dAH, 0, ID32, true);
                    umma::gemm_issue_ts<64>(tmem + T_AO, tmem + T_XL, dAH, 0, ID32, true);
                    umma::gemm_issue_ts<64>(tmem + T_AO, tmem + T_XH, dAL, 0, ID32, true);
                    umma::commit(&bar);
                }
                __syncwarp();
            }
            wait_mma();
            if (warp == 0 && umma::elect_one()) refill_slot(0, S_WA, b < 8 ? wnext + W_BA : wb + W_HEADS, B_A);
            {
                float v[16];
                umma::tmem_ld16(trow + T_AO + h * 16, v);
                uint32_t ph[8], pl[8];
#pragma unroll
                for (int q = 0; q < 8; q++) split2(fmaxf(v[2 * q], 0.f), fmaxf(v[2 * q + 1], 0.f), ph[q], pl[q]);
                if (live) {
#pragma unroll
                    for (int d = 0; d < 3; d++) {
                        const int oy = cy - (d - 1);
                        if (oy >= 0 && oy <= 4) {
                            const int off = d * Y_COPY + (2 * h) * Y_LBO + (1 + r - 6 * (d - 1)) * 16;
                            *reinterpret_cast<uint4 *>(smem + S_YH + off) = make_uint4(ph[0], ph[1], ph[2], ph[3]);
                            *reinterpret_cast<uint4 *>(smem + S_YH + off + Y_LBO) = make_uint4(ph[4], ph[5], ph[6], ph[7]);
                            *reinterpret_cast<uint4 *>(smem + S_YL + off) = make_uint4(pl[0], pl[1], pl[2], pl[3]);
                            *reinterpret_cast<uint4 *>(smem + S_YL + off + Y_LBO) = make_uint4(pl[4], pl[5], pl[6], pl[7]);
                        }
                    }
                }
            }
            // B: 3x3 conv 32 -> 32: (hi, hi) + (lo, hi) + (hi, lo) over the nine row-shifted taps
            smem_sync();
            if (warp == 0) {
                umma::fence_after_sync();
                if (umma::elect_one()) {
                    umma::mbar_wait(&barW[1], phW1); phW1 ^= 1;
                    // columns [0,32) of AO: bias + a_hi*w_hi + a_lo*w_hi; columns [32,64): a_hi*w_lo (summed in the epilogue)
                    bias_mma(tmem + T_AO, dBH, 288, ID64, false);
#pragma unroll
                    for (int d = 0; d < 3; d++)
#pragma unroll
                        for (int dxi = 0; dxi < 3; dxi++)
#pragma unroll
                            for (int ks = 0; ks < 2; ks++) {
                                const uint32_t ao = (uint32_t)(d * Y_COPY + dxi * 16 + 2 * ks * Y_LBO), wo = (uint32_t)(((d * 3 + dxi) * 32 / 8 + 2 * ks) * 128);
                                umma::mma_bf16(tmem + T_AO, umma::desc_at(dYH, ao), umma::desc_at(dBH, wo), ID64, true);
                                umma::mma_bf16(tmem + T_AO, umma::desc_at(dYL, ao), umma::desc_at(dBH, wo), ID32, true);
                            }
                    umma::commit(&bar);
                }
                __syncwarp();
            }
            wait_mma();
            if (warp == 0 && umma::elect_one()) {
                if (b < 8) refill_slot(1, S_WB, wnext + W_BB, B_B);
                else refill_slot(1, S_WB, wb + W_CONV1, B_CONV1);           // conv1 of the next tile
            }
            {
                float v[16], u[16];
                umma::tmem_ld16(trow + T_AO + h * 16, v);
                umma::tmem_ld16(trow + T_AO + 32 + h * 16, u);
                uint32_t ph[8], pl[8];
#pragma unroll
                for (int q = 0; q < 8; q++) split2(fmaxf(v[2 * q] + u[2 * q], 0.f), fmaxf(v[2 * q + 1] + u[2 * q + 1], 0.f), ph[q], pl[q]);
                umma::tmem_st8(trow + T_XH + h * 8, ph);         // conv C's operand: 32 channels = 16 columns, hi and lo
                umma::tmem_st8(trow + T_XL + h * 8, pl);
            }
            // C: 1x1 conv 32 -> 64 accumulated onto the residual
            tmem_sync();
            if (warp == 0) {
                umma::fence_after_sync();
                if (umma::elect_one()) {
                    umma::mbar_wait(&barW[2], phW2); phW2 ^= 1;
                    bias_mma(tmem + T_X, dCH, 32, ID64, true);
                    umma::gemm_issue_ts<32>(tmem + T_X, tmem + T_XH, dCH, 0, ID64, true);
                    umma::gemm_issue_ts<32>(tmem + T_X, tmem + T_XL, dCH, 0, ID64, true);
                    umma::gemm_issue_ts<32>(tmem + T_X, tmem + T_XH, dCL, 0, ID64, true);
                    umma::commit(&bar);
                }
                __syncwarp();
            }
            wait_mma();
            if (warp == 0 && umma::elect_one()) refill_slot(2, S_WC, wnext + W_BC, B_C);
            finish_x();
        }
        // heads
        tmem_sync();
        if (warp == 0) {
            umma::fence_after_sync();
            if (umma::elect_one()) {
                umma::mbar_wait(&barW[0], phW0); phW0 ^= 1;
                bias_mma(tmem + T_AO, dAH, 64, ID32, false);
                umma::gemm_issue_ts<64>(tmem + T_AO, tmem + T_XH, dAH, 0, ID32, true);
                umma::gemm_issue_ts<64>(tmem + T_AO, tmem + T_XL, dAH, 0, ID32, true);
                umma::gemm_issue_ts<64>(tmem + T_AO, tmem + T_XH, dAL, 0, ID32, true);
                umma::commit(&bar);
            }
            __syncwarp();
        }
        wait_mma();
        if (warp == 0 && umma::elect_one()) refill_slot(0, S_WA, wb + W_BLOCK0 + W_BA, B_A);
        {
            float v[16];
            umma::tmem_ld16(trow + T_AO + h * 16, v);
            if (live && p_local < n_pos) {
                if (h == 0) {
                    // Flatten in (y, x, c) order = K index cell * 16 + c, written as hi / lo halves straight in the accurate policy
                    // dense kernel's A-operand layout (128-position tiles of four K-chunks)
                    uint32_t ph[8], pl[8];
#pragma unroll
                    for (int q = 0; q < 8; q++) split2(fmaxf(v[2 * q], 0.f), fmaxf(v[2 * q + 1], 0.f), ph[q], pl[q]);
                    const int64_t pos = pos0 + p_local;
#pragma unroll
                    for (int part = 0; part < 2; part++) {               // the cell's channels 0-7 and 8-15 may fall into different chunks
                        const int k = cell * 16 + part * 8;
                        const int c = k >= 304 ? 3 : k >= 208 ? 2 : k >= 112 ? 1 : 0;
                        const int64_t off = (pos >> 7) * PD_TILE_B + pd_a_off(c) + umma::op_offset((int)(pos & 127), k - pd_k0(c), pd_kc(c));
                        *reinterpret_cast<uint4 *>(polc_h + off) = make_uint4(ph[4 * part], ph[4 * part + 1], ph[4 * part + 2], ph[4 * part + 3]);
                        *reinterpret_cast<uint4 *>(polc_l + off) = make_uint4(pl[4 * part], pl[4 * part + 1], pl[4 * part + 2], pl[4 * part + 3]);
                    }
                } else {
                    reinterpret_cast<float *>(smem + S_VALC)[p_local * 25 + cell] = fmaxf(v[0], 0.f);
                }
            }
        }
        umma::fence_before_sync();
        __syncthreads();
        if (warp < n_pos) {
            const float *valc = reinterpret_cast<const float *>(smem + S_VALC) + warp * 25;
            float acc = __ldg(fb + tcl::F_D1B + lane);
            for (int k = 0; k < 25; k++) acc = fmaf(valc[k], __ldg(fb + tcl::F_D1W + k * 32 + lane), acc);
            float sv = fmaxf(acc, 0.f) * __ldg(fb + tcl::F_VHW + lane);
#pragma unroll
            for (int off = 16; off; off >>= 1) sv += __shfl_xor_sync(0xFFFFFFFFu, sv, off);
            if (lane == 0) value[pos0 + warp] = tanhf(sv + __ldg(fb + tcl::F_VHB));
        }
        __syncthreads();
    }
    if (warp == 0 && umma::elect_one()) {
        umma::mbar_wait(&barW[0], phW0); umma::mbar_wait(&barW[1], phW1); umma::mbar_wait(&barW[2], phW2);
    }
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 0) umma::tmem_free(tmem, 256);
}

// =====================================================================================================
// Accurate trunk, multi-context form (r02 second session): ONE CTA per SM runs NCTX independent 256-thread contexts, one
// tile each, that SHARE the streamed weight slots.  k_net_trunk_acc keeps a private 58 KB weight copy per CTA, so only two
// tiles fit on an SM; its ncu profile (profiles/r02c_kernels_ncu.md) shows every context waiting for the tensor core half of
// its time while the tensor core is busy 55 % of the time — two contexts are not enough to keep it fed.  Sharing the slots
// makes room for three (221 KB of shared memory, 3 x 160 of the 512 TMEM columns, 80 registers):
//  * TMEM per context: X fp32 [64] | XH|XL split 16-bit residual [32+32], REUSED as conv B's N = 64 accumulator (conv A has
//    consumed XH / XL by then) | AO [32]: conv A / heads output, REUSED for conv C's operand (hi 16 | lo 16).  The three
//    regions of all contexts are laid out region-major so that every accumulator starts at a multiple of its width.
//  * weight slots: a layer's operand lands once per CTA; each context's issuing lane waits for the slot's "full" barrier
//    before its MMAs and counts itself off after they complete; the last of the contexts still working in this round
//    streams the next layer in.  A context runs at most one slot use ahead of the slowest one.
//  * tiles: tile = round * (grid * NCTX) + ctx * grid + block, so the last, partial round is spread over the SMs instead of
//    filling some CTAs' three contexts; contexts without a tile leave (the counts above use the round's active contexts).
//  * the next tile's input planes are prefetched into registers while the current tile computes (k_net_trunk_acc staged them
//    byte by byte at the tile start: 8 % of its time), the value-head dense lives in shared memory.
//  * rows of a tile in board-row-major order (ROWMAJ, see namespace acm): the 3x3 conv reads ONE operand buffer through row-shifted
//    descriptors instead of three copies; the conv A epilogue stores a third of the bytes (SPLIT_A then has nothing to split).
// Arithmetic per tile is k_net_trunk_acc's, bit for bit (tests/test_gpu_net.py::test_acc_multi_context_equals_single).
namespace acm {
using namespace acl;
constexpr int CTX_T = 256;
// Row order of a tile's 128 operand rows and the 3x3 conv's operand buffers, per ROWMAJ:
//  false: position-major rows r = p*30 + y*6 + x and THREE row-shifted copies (one per kernel row dy, rows that would leak into the
//         neighbouring position dropped) of the hi and of the lo half — k_net_trunk_acc's layout;
//  true:  board-row-major rows r = y*24 + p*6 + x (the four positions' rows y side by side): a vertical step is +-24 rows and
//         lands in the zero guard rows before / after the tile for y = 0 / y = 4, a horizontal step lands in the guard cell x = 5,
//         so ONE buffer (25 guard rows + 128 + 25) serves all nine taps through the descriptor's start row: a third of the
//         epilogue's shared-memory stores and of the buffer space.
constexpr int G2 = 25, YROWS2 = 128 + 2 * G2, Y_LBO2 = YROWS2 * 16, Y_BUF2 = 4 * Y_LBO2;          // 11,392 B per half
__host__ __device__ constexpr int c_yl(bool rowmaj) { return rowmaj ? Y_BUF2 : 3 * Y_COPY; }
__host__ __device__ constexpr int c_planes(bool rowmaj) { return 2 * c_yl(rowmaj); }
__host__ __device__ constexpr int c_valc(bool rowmaj) { return c_planes(rowmaj) + 1376; }
__host__ __device__ constexpr int ctx_b(bool rowmaj) { return ((c_valc(rowmaj) + 512 + 127) / 128) * 128; }     // 51,840 / 24,704 B per context
constexpr int NF = tcl::F_TOTAL - tcl::F_D1W, F_BYTES = ((NF * 4 + 15) / 16) * 16;
constexpr int FO_D1W = 0, FO_D1B = 800, FO_VHW = 832, FO_VHB = 864;
__host__ __device__ constexpr int s_wa(int nctx, bool rowmaj) { return nctx * ctx_b(rowmaj); }
__host__ __device__ constexpr int s_wb(int nctx, bool rowmaj) { return s_wa(nctx, rowmaj) + B_A; }
__host__ __device__ constexpr int s_wc(int nctx, bool rowmaj) { return s_wb(nctx, rowmaj) + B_B; }
__host__ __device__ constexpr int s_ones(int nctx, bool rowmaj) { return s_wc(nctx, rowmaj) + B_C; }
__host__ __device__ constexpr int s_f(int nctx, bool rowmaj) { return s_ones(nctx, rowmaj) + 128 * 16 * 2; }
__host__ __device__ constexpr int s_total(int nctx, bool rowmaj) { return s_f(nctx, rowmaj) + F_BYTES; }
__host__ __device__ constexpr int tmem_cols(int nctx) { return nctx * 160 <= 256 ? 256 : 512; }
static_assert(s_total(3, false) <= 227 * 1024 && s_total(3, true) <= 227 * 1024, "three contexts fit in one SM's shared memory");
static_assert(B_A % 128 == 0 && B_B % 128 == 0 && B_C % 128 == 0 && c_yl(false) % 128 == 0 && c_yl(true) % 128 == 0 && c_planes(false) % 16 == 0 && c_planes(true) % 16 == 0, "alignment");
}  // namespace acm

template <int NCTX, bool SPLIT_A, bool ROWMAJ, bool COUNTED = false>     // COUNTED: as k_net_trunk_tc4
__global__ void __launch_bounds__(NCTX * acm::CTX_T, 1)
k_net_trunk_accm(const uint8_t *__restrict__ wb, const float *__restrict__ fb, const uint8_t *__restrict__ planes, int64_t n,
                 uint8_t *__restrict__ polc_h, uint8_t *__restrict__ polc_l, float *__restrict__ value, const int32_t *__restrict__ count)
{
    using namespace acm;
    if constexpr (COUNTED) {
        n = min(n, (int64_t)*count);                 // the row count on the device, capped by the host's capacity
        if ((int64_t)blockIdx.x * POS >= n) return;  // tile_of(0, 0) = blockIdx.x: no tile for any context of this CTA
    }
    constexpr bool FP16 = true;
    constexpr int S_WA = s_wa(NCTX, ROWMAJ), S_WB = s_wb(NCTX, ROWMAJ), S_WC = s_wc(NCTX, ROWMAJ), S_ONES = s_ones(NCTX, ROWMAJ), S_F = s_f(NCTX, ROWMAJ);
    constexpr int CTX_B = ctx_b(ROWMAJ), C_YH = 0, C_YL = c_yl(ROWMAJ), C_PLANES = c_planes(ROWMAJ), C_VALC = c_valc(ROWMAJ);
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ uint64_t bar[NCTX], barW[3];            // per context: MMAs of a phase done; weight slots A, B, C landed
    __shared__ unsigned slot_done[3];                  // contexts that have finished with a slot's current layer, cumulative
    __shared__ uint32_t tmem_slot;
    const int ctx = threadIdx.x >> 8;
    const int t = threadIdx.x & 255, warp = t >> 5, lane = t & 31;
    const int rg = warp & 3, h = warp >> 2;
    const int r = rg * 32 + lane;
    const int p_local = ROWMAJ ? (r % 24) / 6 : r / POS_ROWS, cy = ROWMAJ ? r / 24 : (r % POS_ROWS) / 6, cx = r % 6;     // (30 and 24 are multiples of 6)
    const bool live = r < LIVE_ROWS && cx < 5;
    const int cell = cy * 5 + cx;
    const uint32_t sbase = umma::smem_u32(smem);
    uint8_t *const sctx = smem + ctx * CTX_B;
    const float *sF = reinterpret_cast<const float *>(smem + S_F);
    const int64_t n_tiles = (n + POS - 1) / POS;
    const int64_t round_tiles = (int64_t)gridDim.x * NCTX;
    const bool planes_aligned = (reinterpret_cast<uintptr_t>(planes) & 3) == 0;
    auto tile_of = [&](int64_t round, int c) { return round * round_tiles + (int64_t)c * gridDim.x + blockIdx.x; };
    // contexts of this CTA that have a tile in `round` (tile_of grows with the context index: they are contexts 0 .. count-1)
    auto active_in = [&](int64_t round) {
        unsigned a = 0;
#pragma unroll
        for (int c = 0; c < NCTX; c++) a += tile_of(round, c) < n_tiles ? 1u : 0u;
        return a;
    };

    auto refill_slot = [&](int slot, int dst, const uint8_t *src, uint32_t bytes) {
        umma::mbar_expect_tx(&barW[slot], bytes);
        umma::bulk_g2s(sbase + dst, src, bytes, &barW[slot]);
    };
    // words t and 256 + t (< 343) of a tile's input planes; bytes past the last position read as zero
    auto load_planes = [&](int64_t tile, uint32_t (&w)[2]) {
        w[0] = 0u; w[1] = 0u;
        if (tile >= n_tiles) return;
        const int bytes = (int)min((int64_t)POS, n - tile * POS) * 343;
        const uint8_t *src = planes + tile * (POS * 343);
        if (bytes == POS * 343 && planes_aligned) {
            w[0] = __ldg(reinterpret_cast<const uint32_t *>(src) + t);
            if (t < 343 - CTX_T) w[1] = __ldg(reinterpret_cast<const uint32_t *>(src) + CTX_T + t);
        } else {
#pragma unroll
            for (int q = 0; q < 2; q++)
                for (int k = 0; k < 4; k++) {
                    const int byte = (q * CTX_T + t) * 4 + k;
                    if (byte < bytes) w[q] |= (uint32_t)__ldg(src + byte) << (8 * k);
                }
        }
    };
    auto store_planes = [&](const uint32_t (&w)[2]) {
#pragma unroll
        for (int q = 0; q < 2; q++) {
            const int idx = q * CTX_T + t;
            if (idx < 344) reinterpret_cast<uint32_t *>(sctx + C_PLANES)[idx] = w[q];
        }
    };

    for (int i = threadIdx.x; i < NCTX * CTX_B / 16; i += NCTX * CTX_T) reinterpret_cast<uint4 *>(smem)[i] = make_uint4(0, 0, 0, 0);   // guard rows of every copy set
    for (int i = threadIdx.x; i < NF; i += NCTX * CTX_T) reinterpret_cast<float *>(smem + S_F)[i] = __ldg(fb + tcl::F_D1W + i);
    for (int i = threadIdx.x; i < 128 * 2; i += NCTX * CTX_T) {
        const int rr = i >> 1, chunk = i & 1;
        *reinterpret_cast<uint4 *>(smem + S_ONES + umma::op_offset(rr, chunk * 8, 16)) = make_uint4(chunk == 0 ? pack2<FP16>(1.f, 1.f) : 0u, 0u, 0u, 0u);
    }
    __syncthreads();                                   // the zero fill above covers the plane staging areas written next
    {
        uint32_t w0[2];
        load_planes(tile_of(0, ctx), w0);
        store_planes(w0);
    }
    if (threadIdx.x == 0) {
        slot_done[0] = 0u; slot_done[1] = 0u; slot_done[2] = 0u;
#pragma unroll
        for (int q = 0; q < NCTX; q++) umma::mbar_init(&bar[q], 1);
#pragma unroll
        for (int q = 0; q < 3; q++) umma::mbar_init(&barW[q], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        refill_slot(1, S_WB, wb + W_CONV1, B_CONV1);                     // slot B: conv1 first, conv B of block 0 right after it
        refill_slot(0, S_WA, wb + W_BLOCK0 + W_BA, B_A);
        refill_slot(2, S_WC, wb + W_BLOCK0 + W_BC, B_C);
    }
    if (threadIdx.x < 32) umma::tmem_alloc(&tmem_slot, tmem_cols(NCTX));
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    uint32_t phW0 = 0, phW1 = 0, phW2 = 0;             // parities of the weight-slot barriers (tracked by each context's issuing lane)
    unsigned due0 = 0, due1 = 0, due2 = 0;             // cumulative count at which a slot's current layer has been consumed by everyone
    // TMEM columns, region-major over the contexts: X [ctx*64, +64) | XH|XL = conv B accumulator [NCTX*64 + ctx*64, +64) | AO [NCTX*128 + ctx*32, +32)
    const uint32_t tmem = tmem_slot;
    const uint32_t T_Xc = (uint32_t)(ctx * 64), T_XHc = (uint32_t)(NCTX * 64 + ctx * 64), T_XLc = T_XHc + 32u, T_BOc = T_XHc;
    const uint32_t T_AOc = (uint32_t)(NCTX * 128 + ctx * 32), T_CHc = T_AOc, T_CLc = T_AOc + 16u;
    const uint32_t trow = tmem + ((uint32_t)(rg * 32) << 16);
    uint32_t phase = 0;
    constexpr int YLBO = ROWMAJ ? Y_LBO2 : Y_LBO;
    const umma::DescBase dYH = umma::desc_base(sbase + ctx * CTX_B + C_YH, YLBO, 128u), dYL = umma::desc_base(sbase + ctx * CTX_B + C_YL, YLBO, 128u);
    const umma::DescBase dC1H = umma::desc_base(sbase + S_WB, 128u, 80 / 8 * 128u), dC1L = umma::desc_base(sbase + S_WB + hi_b(64, 64), 128u, 64 / 8 * 128u);
    const umma::DescBase dAH = umma::desc_base(sbase + S_WA, 128u, 80 / 8 * 128u), dAL = umma::desc_base(sbase + S_WA + hi_b(32, 64), 128u, 64 / 8 * 128u);
    const umma::DescBase dBH = umma::desc_base(sbase + S_WB, 128u, 304 / 8 * 128u);          // rows 0-31 hi, rows 32-63 lo
    const umma::DescBase dCH = umma::desc_base(sbase + S_WC, 128u, 48 / 8 * 128u), dCL = umma::desc_base(sbase + S_WC + hi_b(64, 32), 128u, 32 / 8 * 128u);
    const umma::DescBase dONES = umma::desc_base(sbase + S_ONES, 128u, 16 / 8 * 128u);
    constexpr uint32_t ID32 = umma::make_idesc(32, FP16), ID64 = umma::make_idesc(64, FP16);

    auto ctx_barrier = [&]() { asm volatile("bar.sync %0, 256;" :: "r"(1 + ctx) : "memory"); };        // this context's 8 warps only
    auto tmem_sync = [&]() { umma::tmem_wait_st(); umma::fence_before_sync(); ctx_barrier(); };
    auto smem_sync = [&]() { umma::fence_async_smem(); umma::fence_before_sync(); ctx_barrier(); };
    auto wait_mma = [&]() { umma::mbar_wait(&bar[ctx], phase); phase ^= 1; umma::fence_after_sync(); };
    auto bias_mma = [&](uint32_t tmem_d, umma::DescBase w, int K, uint32_t idesc, bool accumulate) {
        umma::mma_bf16(tmem_d, umma::desc_at(dONES, 0u), umma::desc_at(w, (uint32_t)(K / 8) * 128u), idesc, accumulate);
    };
    // this context's MMAs of the slot's current layer are complete: count it off; the last one streams the next layer in
    auto slot_release = [&](int slot, unsigned &due, unsigned nact, int dst, const uint8_t *src, uint32_t bytes, bool wanted) {
        due += nact;
        if (warp == 0 && umma::elect_one()) {
            if (atomicAdd(&slot_done[slot], 1u) + 1u == due && wanted) refill_slot(slot, dst, src, bytes);
        }
    };
    // this thread's 32 residual columns: ReLU in place in TMEM X (fp32) and the split 16-bit copies XH / XL
    auto finish_x = [&]() {
#pragma unroll
        for (int half = 0; half < 2; half++) {
            float v[16];
            umma::tmem_ld16(trow + T_Xc + h * 32 + half * 16, v);
            uint32_t f[16], ph[8], pl[8];
#pragma unroll
            for (int j = 0; j < 16; j++) { v[j] = fmaxf(v[j], 0.f); f[j] = __float_as_uint(v[j]); }
#pragma unroll
            for (int j = 0; j < 8; j++) split2(v[2 * j], v[2 * j + 1], ph[j], pl[j]);
            umma::tmem_st16(trow + T_Xc + h * 32 + half * 16, f);
            umma::tmem_st8(trow + T_XHc + h * 16 + half * 8, ph);
            umma::tmem_st8(trow + T_XLc + h * 16 + half * 8, pl);
        }
    };

#ifdef CCX_ACC_TIMING
    long long ts[128]; int nts = 0;
#define ACC_TS() do { if (threadIdx.x == 0 && blockIdx.x == 0 && nts < 128) ts[nts++] = clock64(); } while (0)
#else
#define ACC_TS() do { } while (0)
#endif
    for (int64_t round = 0; tile_of(round, ctx) < n_tiles; round++) {
#ifdef CCX_ACC_TIMING
        nts = 0;
        ACC_TS();
#endif
        const int64_t tile = tile_of(round, ctx);
        const int64_t pos0 = tile * POS;
        const int n_pos = (int)min((int64_t)POS, n - pos0);
        const unsigned nact = active_in(round);
        const bool more = tile_of(round + 1, 0) < n_tiles;             // somebody in this CTA works in the next round
        uint32_t pw[2];
        load_planes(tile_of(round + 1, ctx), pw);                      // lands while this tile computes
        // conv1 operand: the uint8 plane values are exact in half precision, so only the weights are split (a_lo = 0)
        {
            const uint8_t *pl = sctx + C_PLANES + (live ? p_local * 343 : 0);
#pragma unroll
            for (int c8 = 0; c8 < 2; c8++) {
                uint32_t pk[8];
#pragma unroll
                for (int q = 0; q < 8; q++) {
                    float v2[2];
#pragma unroll
                    for (int e = 0; e < 2; e++) {
                        const int kk = h * 32 + c8 * 16 + q * 2 + e;
                        const int tap = kk / 7, ch = kk % 7, dy = tap / 3, dx = tap % 3;
                        v2[e] = (live && kk < 63) ? (float)pl[((cy + dy) * 7 + (cx + dx)) * 7 + ch] : 0.f;
                    }
                    pk[q] = pack2<FP16>(v2[0], v2[1]);
                }
                umma::tmem_st8(trow + T_XHc + h * 16 + c8 * 8, pk);
            }
        }
        tmem_sync(); ACC_TS();
        if (warp == 0) {
            umma::fence_after_sync();
            if (umma::elect_one()) {
                umma::mbar_wait(&barW[1], phW1); phW1 ^= 1;
                bias_mma(tmem + T_Xc, dC1H, 64, ID64, false);
                umma::gemm_issue_ts<64>(tmem + T_Xc, tmem + T_XHc, dC1H, 0, ID64, true);
                umma::gemm_issue_ts<64>(tmem + T_Xc, tmem + T_XHc, dC1L, 0, ID64, true);
                umma::commit(&bar[ctx]);
            }
            __syncwarp();
        }
        wait_mma(); ACC_TS();
        slot_release(1, due1, nact, S_WB, wb + W_BLOCK0 + W_BB, B_B, true);              // conv B of block 0
        finish_x();
        for (int b = 0; b < 9; b++) {
            const uint8_t *wnext = wb + W_BLOCK0 + ((b + 1) % 9) * W_BLOCK;
            // A: 1x1 conv 64 -> 32
            tmem_sync(); ACC_TS();
            if (warp == 0) {
                umma::fence_after_sync();
                if (umma::elect_one()) {
                    umma::mbar_wait(&barW[0], phW0); phW0 ^= 1;
                    bias_mma(tmem + T_AOc, dAH, 64, ID32, false);
                    umma::gemm_issue_ts<64>(tmem + T_AOc, tmem + T_XHc, dAH, 0, ID32, true);
                    umma::gemm_issue_ts<64>(tmem + T_AOc, tmem + T_XLc, dAH, 0, ID32, true);
                    umma::gemm_issue_ts<64>(tmem + T_AOc, tmem + T_XHc, dAL, 0, ID32, true);
                    umma::commit(&bar[ctx]);
                }
                __syncwarp();
            }
            wait_mma(); ACC_TS();
            slot_release(0, due0, nact, S_WA, b < 8 ? wnext + W_BA : wb + W_HEADS, B_A, true);
            {
                float v[16];
                umma::tmem_ld16(trow + T_AOc + h * 16, v);
                uint32_t ph[8], pl[8];
#pragma unroll
                for (int q = 0; q < 8; q++) split2(fmaxf(v[2 * q], 0.f), fmaxf(v[2 * q + 1], 0.f), ph[q], pl[q]);
                // B: 3x3 conv 32 -> 32: (hi, hi) + (lo, hi) + (hi, lo) over the nine row-shifted taps; the N = 64 accumulator
                // takes the place of XH | XL, which conv A has consumed.  SPLIT_A: the copy of kernel row dy = -1 is written
                // first and its three taps' MMAs are in flight while the other two copies are written (same MMA order).
                auto store_copy = [&](int d) {
                    const int oy = cy - (d - 1);
                    if (live && (ROWMAJ || (oy >= 0 && oy <= 4))) {
                        const int off = ROWMAJ ? (2 * h) * YLBO + (G2 + r) * 16 : d * Y_COPY + (2 * h) * YLBO + (1 + r - 6 * (d - 1)) * 16;
                        *reinterpret_cast<uint4 *>(sctx + C_YH + off) = make_uint4(ph[0], ph[1], ph[2], ph[3]);
                        *reinterpret_cast<uint4 *>(sctx + C_YH + off + YLBO) = make_uint4(ph[4], ph[5], ph[6], ph[7]);
                        *reinterpret_cast<uint4 *>(sctx + C_YL + off) = make_uint4(pl[0], pl[1], pl[2], pl[3]);
                        *reinterpret_cast<uint4 *>(sctx + C_YL + off + YLBO) = make_uint4(pl[4], pl[5], pl[6], pl[7]);
                    }
                };
                auto issue_taps = [&](int d0, int d1) {
#pragma unroll
                    for (int d = d0; d < d1; d++)
#pragma unroll
                        for (int dxi = 0; dxi < 3; dxi++)
#pragma unroll
                            for (int ks = 0; ks < 2; ks++) {
                                // input row = output row + 24 (or 6) * dy + dx, dy = d - 1, dx = dxi - 1: the start row of the A operand
                                const uint32_t ao = ROWMAJ ? (uint32_t)((G2 + 24 * (d - 1) + (dxi - 1)) * 16 + 2 * ks * YLBO)
                                                           : (uint32_t)(d * Y_COPY + dxi * 16 + 2 * ks * YLBO);
                                const uint32_t wo = (uint32_t)(((d * 3 + dxi) * 32 / 8 + 2 * ks) * 128);
                                umma::mma_bf16(tmem + T_BOc, umma::desc_at(dYH, ao), umma::desc_at(dBH, wo), ID64, true);
                                umma::mma_bf16(tmem + T_BOc, umma::desc_at(dYL, ao), umma::desc_at(dBH, wo), ID32, true);
                            }
                };
                store_copy(0);
                if (SPLIT_A && !ROWMAJ) {
                    smem_sync(); ACC_TS();
                    if (warp == 0) {
                        umma::fence_after_sync();
                        if (umma::elect_one()) {
                            umma::mbar_wait(&barW[1], phW1); phW1 ^= 1;
                            bias_mma(tmem + T_BOc, dBH, 288, ID64, false);
                            issue_taps(0, 1);
                        }
                        __syncwarp();
                    }
                }
                if (!ROWMAJ) { store_copy(1); store_copy(2); }
                smem_sync(); ACC_TS();
                if (warp == 0) {
                    umma::fence_after_sync();
                    if (umma::elect_one()) {
                        if (!SPLIT_A || ROWMAJ) {
                            umma::mbar_wait(&barW[1], phW1); phW1 ^= 1;
                            bias_mma(tmem + T_BOc, dBH, 288, ID64, false);
                            issue_taps(0, 1);
                        }
                        issue_taps(1, 3);
                        umma::commit(&bar[ctx]);
                    }
                    __syncwarp();
                }
            }
            wait_mma(); ACC_TS();
            if (b < 8) slot_release(1, due1, nact, S_WB, wnext + W_BB, B_B, true);
            else slot_release(1, due1, nact, S_WB, wb + W_CONV1, B_CONV1, more);         // conv1 of the next round's tiles
            {
                float v[16], u[16];
                umma::tmem_ld16(trow + T_BOc + h * 16, v);
                umma::tmem_ld16(trow + T_BOc + 32 + h * 16, u);
                uint32_t ph[8], pl[8];
#pragma unroll
                for (int q = 0; q < 8; q++) split2(fmaxf(v[2 * q] + u[2 * q], 0.f), fmaxf(v[2 * q + 1] + u[2 * q + 1], 0.f), ph[q], pl[q]);
                umma::tmem_st8(trow + T_CHc + h * 8, ph);        // conv C's operand: 32 channels = 16 columns, hi and lo
                umma::tmem_st8(trow + T_CLc + h * 8, pl);
            }
            // C: 1x1 conv 32 -> 64 accumulated onto the residual
            tmem_sync(); ACC_TS();
            if (warp == 0) {
                umma::fence_after_sync();
                if (umma::elect_one()) {
                    umma::mbar_wait(&barW[2], phW2); phW2 ^= 1;
                    bias_mma(tmem + T_Xc, dCH, 32, ID64, true);
                    umma::gemm_issue_ts<32>(tmem + T_Xc, tmem + T_CHc, dCH, 0, ID64, true);
                    umma::gemm_issue_ts<32>(tmem + T_Xc, tmem + T_CLc, dCH, 0, ID64, true);
                    umma::gemm_issue_ts<32>(tmem + T_Xc, tmem + T_CHc, dCL, 0, ID64, true);
                    umma::commit(&bar[ctx]);
                }
                __syncwarp();
            }
            wait_mma(); ACC_TS();
            slot_release(2, due2, nact, S_WC, wnext + W_BC, B_C, b < 8 || more);
            finish_x();
        }
        // heads
        tmem_sync(); ACC_TS();
        if (warp == 0) {
            umma::fence_after_sync();
            if (umma::elect_one()) {
                umma::mbar_wait(&barW[0], phW0); phW0 ^= 1;
                bias_mma(tmem + T_AOc, dAH, 64, ID32, false);
                umma::gemm_issue_ts<64>(tmem + T_AOc, tmem + T_XHc, dAH, 0, ID32, true);
                umma::gemm_issue_ts<64>(tmem + T_AOc, tmem + T_XLc, dAH, 0, ID32, true);
                umma::gemm_issue_ts<64>(tmem + T_AOc, tmem + T_XHc, dAL, 0, ID32, true);
                umma::commit(&bar[ctx]);
            }
            __syncwarp();
        }
        wait_mma(); ACC_TS();
        slot_release(0, due0, nact, S_WA, wb + W_BLOCK0 + W_BA, B_A, more);
        {
            float v[16];
            umma::tmem_ld16(trow + T_AOc + h * 16, v);
            if (live && p_local < n_pos) {
                if (h == 0) {
                    // Flatten in (y, x, c) order = K index cell * 16 + c, written as hi / lo halves straight in the accurate policy
                    // dense kernel's A-operand layout (128-position tiles of four K-chunks)
                    uint32_t ph[8], pl[8];
#pragma unroll
                    for (int q = 0; q < 8; q++) split2(fmaxf(v[2 * q], 0.f), fmaxf(v[2 * q + 1], 0.f), ph[q], pl[q]);
                    const int64_t pos = pos0 + p_local;
#pragma unroll
                    for (int part = 0; part < 2; part++) {               // the cell's channels 0-7 and 8-15 may fall into different chunks
                        const int k = cell * 16 + part * 8;
                        const int c = k >= 304 ? 3 : k >= 208 ? 2 : k >= 112 ? 1 : 0;
                        const int64_t off = (pos >> 7) * PD_TILE_B + pd_a_off(c) + umma::op_offset((int)(pos & 127), k - pd_k0(c), pd_kc(c));
                        *reinterpret_cast<uint4 *>(polc_h + off) = make_uint4(ph[4 * part], ph[4 * part + 1], ph[4 * part + 2], ph[4 * part + 3]);
                        *reinterpret_cast<uint4 *>(polc_l + off) = make_uint4(pl[4 * part], pl[4 * part + 1], pl[4 * part + 2], pl[4 * part + 3]);
                    }
                } else {
                    reinterpret_cast<float *>(sctx + C_VALC)[p_local * 25 + cell] = fmaxf(v[0], 0.f);
                }
            }
        }
        store_planes(pw);
        umma::fence_before_sync();
        ctx_barrier();
        if (warp < n_pos) {                                // value head: dense_1 25 -> 32 ReLU, value_head 32 -> 1 tanh, fp32
            const float *valc = reinterpret_cast<const float *>(sctx + C_VALC) + warp * 25;
            float acc = sF[FO_D1B + lane];
            for (int k = 0; k < 25; k++) acc = fmaf(valc[k], sF[FO_D1W + k * 32 + lane], acc);
            float sv = fmaxf(acc, 0.f) * sF[FO_VHW + lane];
#pragma unroll
            for (int off = 16; off; off >>= 1) sv += __shfl_xor_sync(0xFFFFFFFFu, sv, off);
            if (lane == 0) value[pos0 + warp] = tanhf(sv + sF[FO_VHB]);
        }
        ctx_barrier();                                     // the value staging is rewritten by the next tile's heads epilogue
#ifdef CCX_ACC_TIMING
        ACC_TS();
        if (threadIdx.x == 0 && blockIdx.x == 0 && (round == 0 || round == 5)) {
            printf("ACCT round %d:", (int)round);
            for (int i = 1; i < nts; i++) printf(" %d", (int)(ts[i] - ts[i - 1]));
            printf("\n");
        }
#endif
    }
    // every refill that was issued had a consumer that waited for it, so nothing is in flight when the contexts meet here
    umma::fence_before_sync();
    __syncthreads();
    if (threadIdx.x < 32) umma::tmem_free(tmem, tmem_cols(NCTX));
}

// Accurate policy dense: logits = flat(policy conv)[B x 400] * W + b in split precision, 128 positions x 80 outputs per CTA.
// Four K-chunks (112, 96, 96, 96) stream through two shared-memory stages, each holding the chunk's hi and lo halves of the
// activations (written in this layout by k_net_trunk_acc) and of the quarter's weight rows; per chunk the issuing lane fires
// A_hi*W_hi + A_lo*W_hi + A_hi*W_lo and commits to the stage's "consumed" barrier so that the chunk after next can land.
namespace pda {
constexpr int NQ = 80;
constexpr int A_B = 128 * 112 * 2, W_B = NQ * 112 * 2;                 // sized for the largest chunk
constexpr int ST_AH = 0, ST_AL = A_B, ST_WH = 2 * A_B, ST_WL = 2 * A_B + W_B, STAGE_B = 2 * A_B + 2 * W_B;
constexpr int S_TOTAL = 2 * STAGE_B;                                   // 186,368 B
constexpr int OUT_LD = NQ + 1;
static_assert(128 * OUT_LD * 4 <= STAGE_B, "fp32 staging fits in stage 0");
}  // namespace pda

__global__ void __launch_bounds__(128, 1)
k_policy_dense_acc(const uint8_t *__restrict__ wb, const float *__restrict__ bias, const uint8_t *__restrict__ polc_h,
                   const uint8_t *__restrict__ polc_l, int64_t n, float *__restrict__ logits, const int32_t *__restrict__ count)
{
    using namespace pda;
    if (count) n = min(n, (int64_t)*count);        // compacted batch: the row count on the device, capped by the host's capacity
    if ((int64_t)blockIdx.x * 128 >= n) return;
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ uint64_t bar, full[2], empty[2];
    __shared__ uint32_t tmem_slot;
    const int t = threadIdx.x, warp = t >> 5;
    const int quarter = blockIdx.y, half = quarter >> 1, c0 = (quarter & 1) * NQ;
    const int64_t row0 = (int64_t)blockIdx.x * 128;
    const uint32_t sbase = umma::smem_u32(smem);
    if (t == 0) {
        umma::mbar_init(&bar, 1);
#pragma unroll
        for (int q = 0; q < 2; q++) { umma::mbar_init(&full[q], 1); umma::mbar_init(&empty[q], 1); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) umma::tmem_alloc(&tmem_slot, 128);
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = tmem_slot;
    constexpr uint32_t ID = umma::make_idesc(NQ, true);
    if (warp == 0) {
        if (umma::elect_one()) {
            auto load_chunk = [&](int c, int st) {
                const int Kc = acl::pd_kc(c);
                const uint32_t ab = 128 * Kc * 2, wbytes = NQ * Kc * 2;
                const int64_t aoff = (int64_t)blockIdx.x * acl::PD_TILE_B + acl::pd_a_off(c);
                const uint8_t *wh = wb + acl::pd_w_off(half, c) + (c0 / 8) * (Kc / 8) * 128;          // this quarter's 80 rows: a contiguous slice
                const uint8_t *wl = wh + 160 * Kc * 2;
                umma::mbar_expect_tx(&full[st], 2 * ab + 2 * wbytes);
                umma::bulk_g2s(sbase + st * STAGE_B + ST_AH, polc_h + aoff, ab, &full[st]);
                umma::bulk_g2s(sbase + st * STAGE_B + ST_AL, polc_l + aoff, ab, &full[st]);
                umma::bulk_g2s(sbase + st * STAGE_B + ST_WH, wh, wbytes, &full[st]);
                umma::bulk_g2s(sbase + st * STAGE_B + ST_WL, wl, wbytes, &full[st]);
            };
            load_chunk(0, 0);
            load_chunk(1, 1);
#pragma unroll
            for (int c = 0; c < 4; c++) {
                const int st = c & 1, Kc = acl::pd_kc(c);
                umma::mbar_wait(&full[st], (uint32_t)(c >> 1) & 1u);
                const uint32_t sb = sbase + st * STAGE_B;
                const umma::DescBase dAH = umma::desc_base(sb + ST_AH, 128u, (uint32_t)(Kc / 8) * 128u), dAL = umma::desc_base(sb + ST_AL, 128u, (uint32_t)(Kc / 8) * 128u);
                const umma::DescBase dWH = umma::desc_base(sb + ST_WH, 128u, (uint32_t)(Kc / 8) * 128u), dWL = umma::desc_base(sb + ST_WL, 128u, (uint32_t)(Kc / 8) * 128u);
                for (int s = 0; s < Kc / 16; s++) {
                    const uint32_t ko = (uint32_t)(2 * s) * 128u;
                    umma::mma_bf16(tmem, umma::desc_at(dAH, ko), umma::desc_at(dWH, ko), ID, c > 0 || s > 0);
                    umma::mma_bf16(tmem, umma::desc_at(dAL, ko), umma::desc_at(dWH, ko), ID, true);
                    umma::mma_bf16(tmem, umma::desc_at(dAH, ko), umma::desc_at(dWL, ko), ID, true);
                }
                if (c + 2 < 4) {
                    umma::commit(&empty[st]);                              // stage consumed -> the chunk after next may land
                    umma::mbar_wait(&empty[st], 0);
                    load_chunk(c + 2, st);
                }
            }
            umma::commit(&bar);
        }
        __syncwarp();
    }
    umma::mbar_wait(&bar, 0);
    umma::fence_after_sync();
    float *stage = reinterpret_cast<float *>(smem);
#pragma unroll
    for (int c = 0; c < NQ; c += 16) {
        float v[16];
        umma::tmem_ld16(tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)c, v);
#pragma unroll
        for (int j = 0; j < 16; j++) stage[t * OUT_LD + c + j] = v[j];
    }
    umma::fence_before_sync();
    __syncthreads();
    const int col_base = half * 160 + c0;
    // two logits per store: 294 and every column base are even, so a pair never straddles the end of a row and is 8-byte aligned
    // whenever the caller's buffers are (the evaluator's own scratch always is)
    if (((reinterpret_cast<uintptr_t>(logits) | reinterpret_cast<uintptr_t>(bias)) & 7) != 0) {
        for (int i = t; i < 128 * NQ; i += 128) {
            const int r = i / NQ, c = i % NQ, col = col_base + c;
            if (row0 + r < n && col < CCX_NUM_ACTIONS) logits[(row0 + r) * CCX_NUM_ACTIONS + col] = stage[r * OUT_LD + c] + __ldg(bias + col);
        }
    } else
    for (int i = t; i < 128 * (NQ / 2); i += 128) {
        const int r = i / (NQ / 2), c = 2 * (i % (NQ / 2)), col = col_base + c;
        if (row0 + r < n && col < CCX_NUM_ACTIONS) {
            const float2 b2 = __ldg(reinterpret_cast<const float2 *>(bias + col));
            *reinterpret_cast<float2 *>(logits + (row0 + r) * CCX_NUM_ACTIONS + col) = make_float2(stage[r * OUT_LD + c] + b2.x, stage[r * OUT_LD + c + 1] + b2.y);
        }
    }
    if (warp == 0) umma::tmem_free(tmem, 128);
}

struct ccx_net_acc { uint8_t *wb = nullptr; uint8_t *polc = nullptr; int64_t cap = 0; };      // polc: hi tiles then lo tiles

void ccx_net_acc_free(ccx_handle *h)
{
    if (!h->net_acc) return;
    cudaFree(h->net_acc->wb); cudaFree(h->net_acc->polc);
    delete h->net_acc;
    h->net_acc = nullptr;
}

extern "C" {

int ccx_net_acc_blob_bytes(void) { return acl::W_TOTAL; }

int ccx_net_load_acc(ccx_handle *h, const void *blob_host, int64_t blob_bytes)
{
    if (!h || !blob_host || blob_bytes != acl::W_TOTAL) return CCX_ERR_ARG;
    if (!h->net_acc) h->net_acc = new (std::nothrow) ccx_net_acc();
    if (!h->net_acc) return CCX_ERR_NOMEM;
    ccx_net_acc &a = *h->net_acc;
    h->epoch++;
    h->pool_gen++;
    if (!a.wb) CCX_CUDA(h, cudaMalloc(&a.wb, acl::W_TOTAL));
    CCX_CUDA(h, cudaMemcpyAsync(a.wb, blob_host, acl::W_TOTAL, cudaMemcpyHostToDevice, h->stream));
    CCX_CUDA(h, cudaStreamSynchronize(h->stream));
    CCX_CUDA(h, cudaFuncSetAttribute(k_net_trunk_acc, cudaFuncAttributeMaxDynamicSharedMemorySize, acl::S_TOTAL));
#define CCX_ACCM_ATTR(N, S, R) do { CCX_CUDA(h, cudaFuncSetAttribute(k_net_trunk_accm<N, S, R>, cudaFuncAttributeMaxDynamicSharedMemorySize, acm::s_total(N, R))); \
                                     CCX_CUDA(h, cudaFuncSetAttribute(k_net_trunk_accm<N, S, R, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, acm::s_total(N, R))); } while (0)
    CCX_ACCM_ATTR(1, false, false); CCX_ACCM_ATTR(2, false, false); CCX_ACCM_ATTR(3, false, false);
    CCX_ACCM_ATTR(1, true, false); CCX_ACCM_ATTR(2, true, false); CCX_ACCM_ATTR(3, true, false);
    CCX_ACCM_ATTR(1, false, true); CCX_ACCM_ATTR(2, false, true); CCX_ACCM_ATTR(3, false, true);
#undef CCX_ACCM_ATTR
    CCX_CUDA(h, cudaFuncSetAttribute(k_policy_dense_acc, cudaFuncAttributeMaxDynamicSharedMemorySize, pda::S_TOTAL));
    return CCX_OK;
}

int ccx_net_set_acc_contexts(ccx_handle *h, int32_t contexts)
{
    if (!h || contexts < -1 || contexts > 3) return CCX_ERR_ARG;
    if (h->acc_ctx != contexts) h->epoch++;          // a cached round graph holds the old kernel
    h->acc_ctx = contexts;
    return CCX_OK;
}

// needs ccx_net_load (fp32 weights: policy dense), ccx_net_load_tc (fp32 blob: value head) and ccx_net_load_acc
int ccx_net_forward_acc(ccx_handle *h, int64_t n, const uint8_t *planes, float *logits, float *value, const float *w_pold, const float *b_pold)
{
    if (!h || n < 0 || (n && (!planes || !logits || !value || !w_pold || !b_pold))) return CCX_ERR_ARG;
    (void)w_pold;
    return ccx_net_forward_acc_on(h, h->stream, n, 0, n, planes, logits, value, b_pold);
}

}  // extern "C"

// rows [row0, row0 + n) of a batch whose internal policy-conv scratch holds `cap` positions, on an explicit stream (the two
// halves of a split batch are in flight on two streams, ccx_mcts_run_net); planes / logits / value point at the first of the n rows
int ccx_net_forward_acc_on(ccx_handle *h, cudaStream_t stream, int64_t cap, int64_t row0, int64_t n, const uint8_t *planes, float *logits,
                           float *value, const float *b_pold, const int32_t *count)
{
    ccx_net_tc *tc = tc_of(h, false);
    if (!h->net_acc || !h->net_acc->wb || !tc || !tc->fb) return CCX_ERR_STATE;
    ccx_net_acc &a = *h->net_acc;
    if (a.cap < cap) {
        h->epoch++;
        CCX_CUDA(h, cudaDeviceSynchronize());          // another stream may still read the old scratch
        if (a.polc) CCX_CUDA(h, cudaFree(a.polc));
        a.polc = nullptr; a.cap = 0;
        const size_t tile_bytes = (size_t)((cap + 127) / 128) * acl::PD_TILE_B;
        CCX_CUDA(h, cudaMalloc(&a.polc, 2 * tile_bytes));
        CCX_CUDA(h, cudaMemsetAsync(a.polc, 0, 2 * tile_bytes, stream));               // rows past n of the last tile stay finite
        a.cap = cap;
    }
    if (n == 0) return CCX_OK;                         // (a call with n = 0 only reserves the scratch)
    if (row0 % 128) return CCX_ERR_ARG;
    const size_t off = (size_t)(row0 / 128) * acl::PD_TILE_B;
    uint8_t *polc_h = a.polc + off, *polc_l = a.polc + (size_t)((a.cap + 127) / 128) * acl::PD_TILE_B + off;
    int64_t tiles = (n + acl::POS - 1) / acl::POS;
    int acc_ctx = h->acc_ctx;      // -1 = automatic: CCX_ACC_CTX if set, else as many contexts (<= 3) as the batch can keep busy
    bool automatic = false;
    if (acc_ctx < 0) {
        static const int env_ctx = [] { const char *e = getenv("CCX_ACC_CTX"); const int v = e ? atoi(e) : -1; return v < 0 || v > 3 ? -1 : v; }();
        acc_ctx = env_ctx < 0 ? 3 : env_ctx;
        automatic = env_ctx < 0;
    }
    if (acc_ctx == 0) {
        unsigned grid = (unsigned)(tiles < 2 * h->num_sms ? tiles : 2 * h->num_sms);       // two resident CTAs per SM
        k_net_trunk_acc<<<grid, acl::THREADS, acl::S_TOTAL, stream>>>(a.wb, tc->fb, planes, n, polc_h, polc_l, value, count);
    } else {
        unsigned grid = (unsigned)(tiles < h->num_sms ? tiles : h->num_sms);               // one CTA per SM, acc_ctx tiles in flight in each
        static const bool split_a = [] { const char *e = getenv("CCX_ACC_SPLIT"); return e ? atoi(e) != 0 : true; }();   // A/B: 0 = conv A's epilogue in one piece
        // a batch that leaves the higher contexts without a tile runs the smaller instantiation (shorter prologue, no register cap)
        const int nctx = !automatic ? acc_ctx : tiles <= h->num_sms ? 1 : tiles <= 2 * (int64_t)h->num_sms ? 2 : 3;
        // CCX_ACC_ROWS=0: position-major rows with three row-shifted copies of the 3x3 operand (k_net_trunk_acc's layout) for A/B
        static const bool rowmaj = [] { const char *e = getenv("CCX_ACC_ROWS"); return e ? atoi(e) != 0 : true; }();
#define CCX_ACCM_LAUNCH(N, S, R) do { if (count) CCX_ACCM_LAUNCH_C(N, S, R, true); else CCX_ACCM_LAUNCH_C(N, S, R, false); } while (0)
#define CCX_ACCM_LAUNCH_C(N, S, R, C) k_net_trunk_accm<N, S, R, C><<<grid, N * acm::CTX_T, acm::s_total(N, R), stream>>>(a.wb, tc->fb, planes, n, polc_h, polc_l, value, count)
#define CCX_ACCM_PICK(N) do { if (rowmaj) CCX_ACCM_LAUNCH(N, false, true); else if (split_a) CCX_ACCM_LAUNCH(N, true, false); else CCX_ACCM_LAUNCH(N, false, false); } while (0)
        if (nctx == 1) CCX_ACCM_PICK(1);
        else if (nctx == 2) CCX_ACCM_PICK(2);
        else CCX_ACCM_PICK(3);
#undef CCX_ACCM_PICK
#undef CCX_ACCM_LAUNCH
#undef CCX_ACCM_LAUNCH_C
    }
    CCX_LAUNCHED(h);
    k_policy_dense_acc<<<dim3((unsigned)((n + 127) / 128), 4), 128, pda::S_TOTAL, stream>>>(a.wb, b_pold, polc_h, polc_l, n, logits, count);
    CCX_LAUNCHED(h);
    return CCX_OK;
}

