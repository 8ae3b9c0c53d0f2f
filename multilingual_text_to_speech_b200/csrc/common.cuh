// Shared device/host helpers for the b200tts hot-path library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/b200tts.h"

namespace b200tts {

void set_last_error(const char* fmt, ...);
int check_cuda(cudaError_t e, const char* what, const char* file, int line);

#define B200_CUDA(call)                                                             \
    do {                                                                            \
        int _st = ::b200tts::check_cuda((call), #call, __FILE__, __LINE__);         \
        if (_st != B200TTS_OK) return _st;                                          \
    } while (0)

#define B200_LAUNCH_CHECK() B200_CUDA(cudaGetLastError())

#define B200_REQUIRE(cond, ...)                                                     \
    do {                                                                            \
        if (!(cond)) {                                                              \
            ::b200tts::set_last_error(__VA_ARGS__);                                 \
            return B200TTS_ERR_INVALID;                                             \
        }                                                                           \
    } while (0)

#define B200_TRY(expr)                                                              \
    do {                                                                            \
        int _st = (expr);                                                           \
        if (_st != B200TTS_OK) return _st;                                          \
    } while (0)

// Named kernel timers (b200tts_kernel_timing): when enabled, CUDA events are recorded on the launching stream around the dominant kernels;
// bench.py reads per-name totals after a synchronize.  Disabled (the default) they cost one relaxed load.  A null name times nothing.
void ktimer_start(const char* name, cudaStream_t st);
void ktimer_stop(const char* name, cudaStream_t st);
struct KernelTimer {
    const char* name; cudaStream_t st;
    KernelTimer(const char* n, cudaStream_t s) : name(n), st(s) { if (n) ktimer_start(n, s); }
    ~KernelTimer() { if (name) ktimer_stop(name, st); }
};

// tcgen05 GEMM (gemm_tc.cu): bf16 tensor maps with SWIZZLE_128B.  map3: dims {d0, d1, d2} (d0 contiguous), byte strides of d1 / d2, box
// {b0, b1, b2}; mapN: rank <= 5, rank - 1 byte strides
int tc_make_map3_bf16(void* map, const void* base, int d0, int d1, int d2, size_t stride1, size_t stride2, int b0, int b1, int b2);
int tc_make_mapN_bf16(void* map, const void* base, int rank, const unsigned long long* dims, const unsigned long long* strides, const unsigned* box);

static inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }
static inline size_t align_up_sz(size_t x, size_t a) { return (x + a - 1) / a * a; }

// ---------------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// Block-wide sum / max; `scratch` must hold >= 33 floats; every thread gets the result.
__device__ __forceinline__ float block_sum(float v, float* scratch) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) scratch[warp] = v;
    __syncthreads();
    if (warp == 0) {
        float t = lane < nw ? scratch[lane] : 0.f;
        t = warp_sum(t);
        if (lane == 0) scratch[32] = t;
    }
    __syncthreads();
    return scratch[32];
}
__device__ __forceinline__ float block_max(float v, float* scratch) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    v = warp_max(v);
    __syncthreads();
    if (lane == 0) scratch[warp] = v;
    __syncthreads();
    if (warp == 0) {
        float t = lane < nw ? scratch[lane] : -INFINITY;
        t = warp_max(t);
        if (lane == 0) scratch[32] = t;
    }
    __syncthreads();
    return scratch[32];
}

__device__ __forceinline__ float sigmoidf_acc(float x) { return 1.f / (1.f + expf(-x)); }

// ---------------------------------------------------------------------------------------------
// GEMM (gemm_f32.cu):  C = alpha * op(A) . op(B) + beta * C + bias[n]
//   op(A)(m,k) = transA ? A[k*lda+m] : A[m*lda+k];  op(B)(k,n) = transB ? B[n*ldb+k] : B[k*ldb+n]
//   batch > 1: pointers advance by stride{A,B,C}.  splitk > 1: raw partial sums are written to
//   `partial` as [splitk][batch][M][N] (dense) and, unless `keep_partials`, reduced into C.
// ---------------------------------------------------------------------------------------------
struct GemmDesc {
    const float* A = nullptr;
    const float* B = nullptr;
    float* C = nullptr;
    const float* bias = nullptr;
    int M = 0, N = 0, K = 0;
    int lda = 0, ldb = 0, ldc = 0;
    int transA = 0, transB = 0;
    float alpha = 1.f, beta = 0.f;
    int batch = 1;
    long long strideA = 0, strideB = 0, strideC = 0;
    int a_batch_mod = 0;          // > 0: A advances by strideA * (batch_index % a_batch_mod)
    int splitk = 1;
    float* partial = nullptr;     // required when splitk > 1
    int keep_partials = 0;        // 1: leave the reduction to the consumer kernel (C untouched)
    // optional: op(A) already available as bf16, K contiguous, row stride lda16 elements (16-byte aligned rows): the tcgen05 path
    // reads it through TMA directly (no packing pass); A / lda are then ignored by that path
    const void* A16 = nullptr;
    int lda16 = 0;
    // optional (tcgen05 path, !transB, batch == 1): op(B) = B [K, N] already available as bf16 rows, row stride ldb16 elements (multiple of
    // 64, 16-byte aligned base); the columns up to the next multiple of 64 beyond N must be readable (their products are never stored).
    // Read in place through TMA as an MN-major operand: no packing pass
    const void* B16 = nullptr;
    int ldb16 = 0;
    // optional two-level K (tcgen05 path only; needs !transA && transB): K = kouter * kin, element (row, q * kin + l) of op(A) lives at
    // A[q * kosA + row * lda + l] (op(B) likewise with kosB): sums a product over `kouter` separately stored slabs in ONE GEMM
    int kin = 0;
    long long kosA = 0, kosB = 0;
};

// pack cache of the tcgen05 GEMM (gemm_tc.cu): operands packed inside a begin / end scope are reused by later products of the scope
void tc_pack_cache_begin();
void tc_pack_cache_end();

int gemm_f32(const GemmDesc& d, cudaStream_t stream);
int gemm_bf16(const GemmDesc& d, cudaStream_t stream);
// Precision mode of the library (b200tts_set_precision): 0 = fp32-exact (parity mode), 1 = bf16 tensor-core operands.
int precision_mode();
void set_precision_mode(int mode);
// Dispatch on the precision mode.
int gemm_run(const GemmDesc& d, cudaStream_t stream);
int gemm_run_auto(GemmDesc d, float* scratch, size_t scratch_elems, cudaStream_t stream);
size_t gemm_partial_elems(const GemmDesc& d);
int gemm_f32_auto(GemmDesc d, float* scratch, size_t scratch_elems, cudaStream_t stream);

}  // namespace b200tts
