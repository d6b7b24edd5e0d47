// pipe_rates.cu — sustained issue rate of single integer instruction classes (scripts/pipe_rates.py).  Each kernel runs a
// stream of one PTX instruction: eight independent dependency chains per lane, unrolled, so the rate is bound by the pipe
// that executes the instruction and not by its latency.  One block per SM; thread 0 of each block stamps clock64 around the
// stream, between two block barriers.  The SASS opcode each stream compiles to is checked by the script (cuobjdump).
#include <cstdint>
#include <cuda_runtime.h>

#define CHAINS 8
#define UNROLL 16

// op(x, y, z) updates x; y and z are loop-invariant registers, so every chain depends only on itself.  ptxas picks the SASS:
// two adds become one IADD3 and two maxes one VIMNMX3; an add of an immediate alone is folded, so VIADD runs interleaved
// with LOP3 (viadd_lop3), IMAD.IADD with PRMT (vadd: imadiadd_prmt); lop3_imad interleaves the two pipes' main opcodes;
// iadd3_lop3 tells whether IADD3 issues to LOP3's pipe (rate near 0.5 together) or to another one (near 1).
#define OPS(X)                                                                                              \
    X(lop3, "lop3.b32 %0, %0, %1, %2, 0x96;")                                                               \
    X(shf, "shf.l.wrap.b32 %0, %0, %1, %2;")                                                                \
    X(iadd3, "add.u32 %0, %0, %1;\n\tadd.u32 %0, %0, %2;")                                                  \
    X(prmt, "prmt.b32 %0, %0, %1, %2;")                                                                     \
    X(vimnmx, "max.s32 %0, %0, %1;")                                                                        \
    X(imad, "mad.lo.u32 %0, %0, %1, %2;")                                                                   \
    X(flo, "bfind.u32 %0, %0;")                                                                             \
    X(popc, "popc.b32 %0, %0;")                                                                             \
    X(viadd_lop3, "add.u32 %0, %0, 0x1234;\n\txor.b32 %0, %0, %1;")                                          \
    X(imadiadd_prmt, "vadd.u32.u32.u32 %0, %0, %1;")                                                        \
    X(lop3_imad, "lop3.b32 %0, %0, %1, %2, 0x96;\n\tmad.lo.u32 %0, %0, %1, %2;") \
    X(iadd3_lop3, "add.u32 %0, %0, %1;\n\tadd.u32 %0, %0, %2;\n\tlop3.b32 %0, %0, %1, %2, 0x96;")

#define KERNEL(name, insn)                                                                                  \
    __global__ void __launch_bounds__(1024, 1) k_rate_##name(int iters, uint32_t y0, uint32_t z0, uint32_t *out, \
                                                              long long *cycles)                            \
    {                                                                                                       \
        const uint32_t y = y0 ^ threadIdx.x, z = z0 + threadIdx.x;                                          \
        uint32_t x[CHAINS];                                                                                 \
        _Pragma("unroll") for (int j = 0; j < CHAINS; j++) x[j] = threadIdx.x * 7919u + j * 104729u;       \
        __syncthreads();                                                                                    \
        long long t0 = clock64();                                                                           \
        _Pragma("unroll 1") for (int i = 0; i < iters; i++) {                                               \
            _Pragma("unroll") for (int u = 0; u < UNROLL; u++)                                              \
                _Pragma("unroll") for (int j = 0; j < CHAINS; j++) asm volatile(insn : "+r"(x[j]) : "r"(y), "r"(z)); \
        }                                                                                                   \
        __syncthreads();                                                                                    \
        long long t1 = clock64();                                                                           \
        uint32_t s = 0;                                                                                     \
        _Pragma("unroll") for (int j = 0; j < CHAINS; j++) s ^= x[j];                                       \
        out[blockIdx.x * blockDim.x + threadIdx.x] = s;                                                     \
        if (threadIdx.x == 0) cycles[blockIdx.x] = t1 - t0;                                                 \
    }
OPS(KERNEL)

#define NAME(name, insn) #name,
static const char *names[] = {OPS(NAME)};
#define PTR(name, insn) k_rate_##name,
typedef void (*kfn)(int, uint32_t, uint32_t, uint32_t *, long long *);
static const kfn kernels[] = {OPS(PTR)};

extern "C" {

int pr_count() { return (int)(sizeof(names) / sizeof(names[0])); }
const char *pr_name(int k) { return names[k]; }
int pr_per_iter() { return CHAINS * UNROLL; }

// runs stream k on `blocks` blocks of `threads` lanes (one block per SM); cycles[b] = clock64 cycles of block b's stream,
// *ms = CUDA-event time of the launch.  Returns a cudaError_t.
int pr_run(int k, int blocks, int threads, int iters, long long *cycles, float *ms)
{
    uint32_t *d_out = nullptr;
    long long *d_cyc = nullptr;
    cudaEvent_t a, b;
    cudaError_t e = cudaMalloc(&d_out, (size_t)blocks * threads * 4);
    if (e == cudaSuccess) e = cudaMalloc(&d_cyc, (size_t)blocks * 8);
    if (e != cudaSuccess) return (int)e;
    cudaEventCreate(&a);
    cudaEventCreate(&b);
    kernels[k]<<<blocks, threads>>>(iters, 0x9E3779B9u, 0x00000507u, d_out, d_cyc);   // warm-up
    cudaEventRecord(a);
    kernels[k]<<<blocks, threads>>>(iters, 0x9E3779B9u, 0x00000507u, d_out, d_cyc);
    cudaEventRecord(b);
    e = cudaEventSynchronize(b);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaEventElapsedTime(ms, a, b);
    if (e == cudaSuccess) e = cudaMemcpy(cycles, d_cyc, (size_t)blocks * 8, cudaMemcpyDeviceToHost);
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    cudaFree(d_out);
    cudaFree(d_cyc);
    return (int)e;
}

}  // extern "C"
