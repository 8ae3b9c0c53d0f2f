// bf16 tensor-core GEMM (fp32 in / fp32 out, operands rounded to bf16 on the way into shared memory,
// fp32 accumulation) for the perf mode ("bf16 fwd / fp32 master", BASELINE.json configs[1]).
// Same GemmDesc contract as gemm_f32 (transposes, batch strides, a_batch_mod, deterministic split-K).
// 128x128x32 CTA tile, 8 warps (2 x 4), each warp 64x32 through mma.sync.m16n8k16 fed by ldmatrix.
#include <cuda_bf16.h>
#include "common.cuh"
#include "ptx.cuh"

namespace b200tts {

namespace {

constexpr int BM = 128, BN = 128, BK = 32, LDS = BK + 8;   // smem row stride in bf16 (80 B: conflict-free ldmatrix)
constexpr int NT = 256;

struct KernelArgs {
    const float* A; const float* B; float* C; const float* bias; float* partial;
    int M, N, K, lda, ldb, ldc;
    int a_kcontig, b_kcontig, a_vec, b_vec;
    float alpha, beta;
    int batch, splitk, kchunk, a_batch_mod;
    long long strideA, strideB, strideC;
};

using namespace tcx;

// Stage a 128 x 32 operand tile: global fp32 -> registers (16 floats / thread).
//   kcontig: element (r, k) at base[r*ld + k]; else at base[k*ld + r].
__device__ __forceinline__ void tile_load(const float* __restrict__ base, int ld, bool kcontig, bool vec, int row0, int rows_total,
                                          int k0, int k_end, float (&regs)[16]) {
    const int tid = threadIdx.x;
    if (vec) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int v = tid + j * NT;                 // 1024 float4 per tile
            float4 val = make_float4(0.f, 0.f, 0.f, 0.f);
            if (kcontig) {
                const int r = v >> 3, kq = v & 7;       // 8 float4 per row of 32 k
                if (row0 + r < rows_total && k0 + kq * 4 < k_end)
                    val = *reinterpret_cast<const float4*>(base + (size_t)(row0 + r) * ld + k0 + kq * 4);
            } else {
                const int k = v >> 5, r4 = v & 31;      // 32 float4 per k row of 128
                if (k0 + k < k_end && row0 + r4 * 4 < rows_total)
                    val = *reinterpret_cast<const float4*>(base + (size_t)(k0 + k) * ld + row0 + r4 * 4);
            }
            regs[j * 4 + 0] = val.x; regs[j * 4 + 1] = val.y; regs[j * 4 + 2] = val.z; regs[j * 4 + 3] = val.w;
        }
    } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const int idx = tid + j * NT;
            float val = 0.f;
            if (kcontig) {
                const int r = idx >> 5, k = idx & 31;
                if (row0 + r < rows_total && k0 + k < k_end) val = base[(size_t)(row0 + r) * ld + k0 + k];
            } else {
                const int k = idx >> 7, r = idx & 127;
                if (k0 + k < k_end && row0 + r < rows_total) val = base[(size_t)(k0 + k) * ld + row0 + r];
            }
            regs[j] = val;
        }
    }
}

// registers -> shared memory tile sm[row][k] (bf16, k contiguous) regardless of the global orientation
__device__ __forceinline__ void tile_store(__nv_bfloat16* sm, bool kcontig, bool vec, const float (&regs)[16]) {
    const int tid = threadIdx.x;
    if (vec) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int v = tid + j * NT;
            if (kcontig) {
                const int r = v >> 3, kq = v & 7;
                uint2 w;
                w.x = pack2(regs[j * 4 + 0], regs[j * 4 + 1]);
                w.y = pack2(regs[j * 4 + 2], regs[j * 4 + 3]);
                *reinterpret_cast<uint2*>(sm + r * LDS + kq * 4) = w;
            } else {
                const int k = v >> 5, r4 = v & 31;
#pragma unroll
                for (int e = 0; e < 4; ++e) sm[(r4 * 4 + e) * LDS + k] = __float2bfloat16_rn(regs[j * 4 + e]);
            }
        }
    } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const int idx = tid + j * NT;
            if (kcontig) sm[(idx >> 5) * LDS + (idx & 31)] = __float2bfloat16_rn(regs[j]);
            else sm[(idx & 127) * LDS + (idx >> 7)] = __float2bfloat16_rn(regs[j]);
        }
    }
}

__global__ void __launch_bounds__(NT) gemm_bf16_kernel(const KernelArgs p) {
    __shared__ __align__(16) __nv_bfloat16 As[2][BM * LDS];
    __shared__ __align__(16) __nv_bfloat16 Bs[2][BN * LDS];
    const int z = blockIdx.z;
    const int bz = z / p.splitk, ks = z % p.splitk;
    const float* A = p.A + (size_t)(p.a_batch_mod > 0 ? bz % p.a_batch_mod : bz) * p.strideA;
    const float* B = p.B + (size_t)bz * p.strideB;
    const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
    const int k_begin = ks * p.kchunk;
    const int k_end = min(p.K, k_begin + p.kchunk);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wm = (warp >> 2) * 64, wn = (warp & 3) * 32;     // warp tile origin inside the CTA tile

    float acc[4][4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int e = 0; e < 4; ++e) acc[i][j][e] = 0.f;

    float ra[16], rb[16];
    const int ntiles = (k_end > k_begin) ? (k_end - k_begin + BK - 1) / BK : 0;
    if (ntiles > 0) {
        tile_load(A, p.lda, p.a_kcontig, p.a_vec, m0, p.M, k_begin, k_end, ra);
        tile_load(B, p.ldb, p.b_kcontig, p.b_vec, n0, p.N, k_begin, k_end, rb);
        tile_store(As[0], p.a_kcontig, p.a_vec, ra);
        tile_store(Bs[0], p.b_kcontig, p.b_vec, rb);
    }
    __syncthreads();
    for (int t = 0; t < ntiles; ++t) {
        const int cur = t & 1;
        if (t + 1 < ntiles) {
            const int k0 = k_begin + (t + 1) * BK;
            tile_load(A, p.lda, p.a_kcontig, p.a_vec, m0, p.M, k0, k_end, ra);
            tile_load(B, p.ldb, p.b_kcontig, p.b_vec, n0, p.N, k0, k_end, rb);
        }
#pragma unroll
        for (int kk = 0; kk < BK; kk += 16) {
            uint32_t af[4][4], bf[2][4];
#pragma unroll
            for (int i = 0; i < 4; ++i)
                ldmatrix_x4(af[i][0], af[i][1], af[i][2], af[i][3], &As[cur][(wm + i * 16 + (lane & 15)) * LDS + kk + (lane >> 4) * 8]);
#pragma unroll
            for (int j = 0; j < 2; ++j)
                ldmatrix_x4(bf[j][0], bf[j][1], bf[j][2], bf[j][3],
                            &Bs[cur][(wn + j * 16 + (lane & 7) + ((lane >> 4) << 3)) * LDS + kk + ((lane >> 3) & 1) * 8]);
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) mma_bf16(acc[i][j], af[i], bf[j >> 1][(j & 1) * 2], bf[j >> 1][(j & 1) * 2 + 1]);
        }
        if (t + 1 < ntiles) {
            tile_store(As[cur ^ 1], p.a_kcontig, p.a_vec, ra);
            tile_store(Bs[cur ^ 1], p.b_kcontig, p.b_vec, rb);
        }
        __syncthreads();
    }

    // epilogue: accumulator element e of tile (i, j): row = g + 8*(e>>1), col = 2*tq + (e&1)
    float* out;
    size_t ldo;
    const bool raw = p.splitk > 1;
    if (raw) { out = p.partial + ((size_t)ks * p.batch + bz) * (size_t)p.M * p.N; ldo = p.N; }
    else { out = p.C + (size_t)bz * p.strideC; ldo = p.ldc; }
    const int g = lane >> 2, tq = lane & 3;
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int m = m0 + wm + i * 16 + g + 8 * (e >> 1);
                const int n = n0 + wn + j * 8 + 2 * tq + (e & 1);
                if (m < p.M && n < p.N) {
                    float v = acc[i][j][e];
                    if (!raw) {
                        v *= p.alpha;
                        if (p.bias) v += p.bias[n];
                        if (p.beta != 0.f) v += p.beta * out[(size_t)m * ldo + n];
                    }
                    out[(size_t)m * ldo + n] = v;
                }
            }
}

__global__ void splitk_reduce_kernel(const float* __restrict__ partial, float* __restrict__ C, const float* __restrict__ bias, int M,
                                     int N, int ldc, int batch, int splitk, long long strideC, float alpha, float beta) {
    const size_t total = (size_t)batch * M * N;
    for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const int n = idx % N;
        const int m = (idx / N) % M;
        const int b = idx / ((size_t)M * N);
        float s = 0.f;
        for (int k = 0; k < splitk; ++k) s += partial[(size_t)k * total + idx];
        s *= alpha;
        if (bias) s += bias[n];
        float* c = C + (size_t)b * strideC + (size_t)m * ldc + n;
        if (beta != 0.f) s += beta * *c;
        *c = s;
    }
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

}  // namespace

int gemm_tc_try(const GemmDesc& d, cudaStream_t st, bool* handled);

int gemm_bf16(const GemmDesc& d, cudaStream_t stream) {
    if (d.M <= 0 || d.N <= 0 || d.batch <= 0) return B200TTS_OK;
    {   // tcgen05 / TMEM / TMA path for the large contractions (gemm_tc.cu); falls through when not applicable
        bool handled = false;
        B200_TRY(gemm_tc_try(d, stream, &handled));
        if (handled) return B200TTS_OK;
    }
    B200_REQUIRE(d.A && d.B && (d.C || (d.splitk > 1 && d.keep_partials)), "gemm_bf16: null operand");
    B200_REQUIRE(d.splitk >= 1 && (d.splitk == 1 || d.partial), "gemm_bf16: split-K needs a partial workspace");
    KernelArgs p;
    p.A = d.A; p.B = d.B; p.C = d.C; p.bias = d.bias; p.partial = d.partial;
    p.M = d.M; p.N = d.N; p.K = d.K; p.lda = d.lda; p.ldb = d.ldb; p.ldc = d.ldc;
    p.a_kcontig = !d.transA; p.b_kcontig = d.transB;
    p.alpha = d.alpha; p.beta = d.beta; p.batch = d.batch; p.splitk = d.splitk;
    p.strideA = d.strideA; p.strideB = d.strideB; p.strideC = d.strideC; p.a_batch_mod = d.a_batch_mod;
    int kchunk = cdiv(d.K > 0 ? d.K : 1, d.splitk);
    p.kchunk = cdiv(kchunk, BK) * BK;
    auto vec_ok = [&](const float* ptr, int ld, long long stride, bool kcontig, int rows) {
        if (!aligned16(ptr) || (ld & 3) || (stride & 3)) return false;
        return kcontig ? ((d.K & 3) == 0) : ((rows & 3) == 0);
    };
    p.a_vec = vec_ok(d.A, d.lda, d.strideA, p.a_kcontig, d.M);
    p.b_vec = vec_ok(d.B, d.ldb, d.strideB, p.b_kcontig, d.N);
    dim3 grid(cdiv(d.N, BN), cdiv(d.M, BM), d.batch * d.splitk);
    gemm_bf16_kernel<<<grid, NT, 0, stream>>>(p);
    B200_LAUNCH_CHECK();
    if (d.splitk > 1 && !d.keep_partials) {
        const size_t total = (size_t)d.batch * d.M * d.N;
        int blocks = (int)((total + 255) / 256);
        if (blocks > 148 * 8) blocks = 148 * 8;
        splitk_reduce_kernel<<<blocks, 256, 0, stream>>>(d.partial, d.C, d.bias, d.M, d.N, d.ldc, d.batch, d.splitk, d.strideC,
                                                          d.alpha, d.beta);
        B200_LAUNCH_CHECK();
    }
    return B200TTS_OK;
}

}  // namespace b200tts
