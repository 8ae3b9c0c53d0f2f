// tcgen05 / TMEM / TMA bf16 GEMM for the time-batched contractions of the perf mode (sm_100a only).
//
//   C[M, N] (fp32) = alpha * A[M, K] . B[N, K]^T + beta * C + bias[n]
//
// Operands are first packed to bf16, K-major (pack kernels below: fp32 -> bf16, transposing when the source is
// M/N-contiguous), then one warp-specialised kernel per 128 x 128 output tile:
//   warp 4 (one lane)  : TMA producer  -- cp.async.bulk.tensor (128B swizzle) into a 4-stage shared-memory ring,
//                        mbarrier expect_tx / complete_tx
//   warp 5 (one lane)  : MMA issuer    -- tcgen05.mma.cta_group::1.kind::f16, M = 128, N = 128, K = 16 per instruction,
//                        accumulator in TMEM (128 lanes x 128 columns fp32); tcgen05.commit frees ring slots
//   warps 0-3          : epilogue      -- tcgen05.ld (32 lanes x 32 columns per instruction) -> staged through the (now idle)
//                        operand ring so that every global store is a full 512-byte row segment -> alpha/beta/bias -> global
// Two CTAs are co-resident per SM (3 x 32 KB ring each, 128 TMEM columns each): one tile's epilogue overlaps the other's main loop.
// Every mbarrier wait carries a clock64 watchdog that traps instead of hanging the device.
#include <cuda.h>
#include <cuda_bf16.h>
#include "common.cuh"
#include "ptx.cuh"

namespace b200tts {

namespace {

constexpr int TBM = 128, TBN = 128, TBK = 64;
constexpr int STAGES = 3;
constexpr int STAGE_BYTES = (TBM + TBN) * TBK * 2;          // 32 KB
constexpr int TC_THREADS = 192;
constexpr int TMEM_COLS = 128;
constexpr int STG_LD = TBN + 4;                             // fp32 row stride of the epilogue staging tile (16-byte aligned, conflict-free)
static_assert(4 * 32 * STG_LD * 4 <= STAGES * STAGE_BYTES, "epilogue staging must fit in the operand ring");

using namespace tcx;

struct TcArgs {
    float* C; const float* bias;
    int M, N, K, ldc;
    float alpha, beta;
    int batch, a_batch_mod;
    long long strideC;
    // implicit 1-D convolution (conv_cb > 0): k-block kb = (tap t = kb / conv_cb, channel block cb = kb % conv_cb); the B tile is
    // rows [n0 + t * conv_dil - conv_pad, + 128) x channels [g * conv_cin + 64 cb, + 64) of sample bz / conv_G in the position-major
    // bf16 copy of the input (TMA zero-fills the rows outside [0, L))
    int conv_cb, conv_dil, conv_pad, conv_G, conv_cin;
    // split-K (batch == 1 only): blockIdx.z = split; each split multiplies k-blocks [z * kper, (z + 1) * kper) and stores its raw fp32
    // tile into partial[z][M][N]; a fixed-order reduction kernel applies alpha / beta / bias afterwards
    int ksplit, kper;
    float* partial;
    // MN-major operands (batch == 1): the bf16 source is [K rows][MN columns] row-major (the natural layout of op(A) = A^T / op(B) = B of a
    // weight-gradient product), fetched as two 64-column chunks of 64 k-rows per stage (3-D map {64, K, MN / 64}, box {64, 64, 2}) and
    // described to the tensor core as MN-major SWIZZLE_128B tiles: no transposing pack
    int a_mn, b_mn;
};

__global__ void __launch_bounds__(TC_THREADS, 2)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const TcArgs p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    // 1024-byte aligned ring (128B swizzle atoms are 1024 B)
    uint8_t* ring = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    __shared__ uint64_t full_bar[STAGES], empty_bar[STAGES], tmem_full_bar;
    __shared__ uint32_t tmem_base_smem;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m0 = blockIdx.y * TBM, n0 = blockIdx.x * TBN;
    const int bz = p.ksplit > 1 ? 0 : blockIdx.z;
    const int az = p.a_batch_mod > 0 ? bz % p.a_batch_mod : bz;
    const int nk_all = (p.K + TBK - 1) / TBK;
    const int kb_lo = p.ksplit > 1 ? blockIdx.z * p.kper : 0;
    const int nk = p.ksplit > 1 ? min(p.kper, nk_all - kb_lo) : nk_all;       // k-blocks of this CTA: [kb_lo, kb_lo + nk)

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        mbar_init(&tmem_full_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 5) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_smem)), "r"(TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = tmem_base_smem;

    if (warp == 4) {
        if (lane == 0) {
            for (int kb = 0; kb < nk; ++kb) {
                const int s = kb % STAGES;
                const uint32_t ph = (kb / STAGES) & 1;
                mbar_wait(&empty_bar[s], ph ^ 1);
                mbar_expect_tx(&full_bar[s], STAGE_BYTES);
                uint8_t* sa = ring + (size_t)s * STAGE_BYTES;
                if (p.a_mn) tma_load_3d(sa, &tmA, &full_bar[s], 0, (kb_lo + kb) * TBK, m0 >> 6);
                else tma_load_3d(sa, &tmA, &full_bar[s], (kb_lo + kb) * TBK, m0, az);
                if (p.b_mn) {
                    tma_load_3d(sa + TBM * TBK * 2, &tmB, &full_bar[s], 0, (kb_lo + kb) * TBK, n0 >> 6);
                } else if (p.conv_cb > 0) {
                    const int t = (kb_lo + kb) / p.conv_cb, cb = (kb_lo + kb) % p.conv_cb;
                    tma_load_3d(sa + TBM * TBK * 2, &tmB, &full_bar[s], (bz % p.conv_G) * p.conv_cin + cb * TBK, n0 + t * p.conv_dil - p.conv_pad,
                                bz / p.conv_G);
                } else {
                    tma_load_3d(sa + TBM * TBK * 2, &tmB, &full_bar[s], (kb_lo + kb) * TBK, n0, bz);
                }
            }
        }
    } else if (warp == 5) {
        if (lane == 0) {
            // instruction descriptor (cute::UMMA::InstrDescriptor): D = F32, A = B = BF16, both K-major, N >> 3, M >> 4
            const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(TBN >> 3) << 17) | ((uint32_t)(TBM >> 4) << 24) |
                                   (p.a_mn ? (1u << 15) : 0u) | (p.b_mn ? (1u << 16) : 0u);      // bits 15 / 16: A / B MN-major
            const uint64_t a_step = p.a_mn ? (2048 >> 4) : 2, b_step = p.b_mn ? (2048 >> 4) : 2;   // address-field advance per K = 16
            for (int kb = 0; kb < nk; ++kb) {
                const int s = kb % STAGES;
                const uint32_t ph = (kb / STAGES) & 1;
                mbar_wait(&full_bar[s], ph);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t a_addr = smem_u32(ring + (size_t)s * STAGE_BYTES);
                const uint64_t adesc = p.a_mn ? make_sw128_mn_desc(a_addr) : make_sw128_desc(a_addr);
                const uint64_t bdesc = p.b_mn ? make_sw128_mn_desc(a_addr + TBM * TBK * 2) : make_sw128_desc(a_addr + TBM * TBK * 2);
#pragma unroll
                for (int k = 0; k < TBK / 16; ++k)        // K-major: advance 16 bf16 = 32 B inside the swizzle atom (+2); MN-major: 16 rows
                    umma_bf16(tmem_base, adesc + a_step * k, bdesc + b_step * k, idesc, (kb | k) != 0);
                umma_commit(&empty_bar[s]);               // implicit tcgen05.fence::before_thread_sync
            }
            umma_commit(&tmem_full_bar);
        }
    } else {
        // epilogue: warp w owns TMEM lanes [32w, 32w + 32) = rows m0 + 32w + lane.  tmem_full implies every MMA (and therefore
        // every TMA load) of this tile has completed, so the operand ring is free to stage the fp32 tile.
        mbar_wait(&tmem_full_bar, 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        float* stg = reinterpret_cast<float*>(ring) + (size_t)warp * 32 * STG_LD;
#pragma unroll 1
        for (int c = 0; c < TBN / 32; ++c) {
            uint32_t r[32];
            tmem_ld32(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(c * 32), r);
            float4* dst = reinterpret_cast<float4*>(stg + (size_t)lane * STG_LD + c * 32);
#pragma unroll
            for (int j = 0; j < 8; ++j)
                dst[j] = make_float4(__uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1]), __uint_as_float(r[4 * j + 2]),
                                     __uint_as_float(r[4 * j + 3]));
        }
        __syncwarp();
        const bool part = p.ksplit > 1;
        float* cbase = part ? p.partial + (size_t)blockIdx.z * p.M * p.N : p.C + (size_t)bz * p.strideC;
        const int ldc = part ? p.N : p.ldc;
        const float alpha = part ? 1.f : p.alpha, beta = part ? 0.f : p.beta;
        const float* bias = part ? nullptr : p.bias;
        const int rows = min(32, p.M - (m0 + warp * 32));
        const int n = n0 + 4 * lane;
        const bool vec = ((ldc & 3) == 0) && ((reinterpret_cast<uintptr_t>(cbase) & 15) == 0) && (n0 + TBN <= p.N);   // warp-uniform
        if (vec) {
            float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
            if (bias) bv = make_float4(bias[n], bias[n + 1], bias[n + 2], bias[n + 3]);
#pragma unroll 4
            for (int rr = 0; rr < rows; ++rr) {
                const float4 a = *reinterpret_cast<const float4*>(stg + (size_t)rr * STG_LD + 4 * lane);
                float4* cp = reinterpret_cast<float4*>(cbase + (size_t)(m0 + warp * 32 + rr) * ldc + n);
                float4 v = make_float4(fmaf(alpha, a.x, bv.x), fmaf(alpha, a.y, bv.y), fmaf(alpha, a.z, bv.z), fmaf(alpha, a.w, bv.w));
                if (beta != 0.f) {
                    const float4 o = *cp;
                    v.x = fmaf(beta, o.x, v.x); v.y = fmaf(beta, o.y, v.y); v.z = fmaf(beta, o.z, v.z); v.w = fmaf(beta, o.w, v.w);
                }
                *cp = v;
            }
        } else {
            for (int rr = 0; rr < rows; ++rr) {
                float* crow = cbase + (size_t)(m0 + warp * 32 + rr) * ldc;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int nn = n0 + j * 32 + lane;
                    if (nn < p.N) {
                        float v = alpha * stg[(size_t)rr * STG_LD + j * 32 + lane];
                        if (bias) v += bias[nn];
                        if (beta != 0.f) v += beta * crow[nn];
                        crow[nn] = v;
                    }
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 5) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS));
    }
}

// ------------------------------------------------------------------------------------------------
// operand packing: fp32 (either orientation) -> bf16 [batch][rows][Kp], K contiguous, Kp % 8 == 0
// ------------------------------------------------------------------------------------------------
// Thread = 8 consecutive k of one row -> ONE 16-byte store (Kp % 8 == 0); rows ride on blockIdx.y: no per-element 64-bit division.
__global__ void pack_kcontig_kernel(__nv_bfloat16* __restrict__ dst, const float* __restrict__ src, int ld, long long bstride, int rows,
                                    int K, int Kp, int kin, long long kos) {
    const float* s = src + (size_t)blockIdx.z * bstride;
    __nv_bfloat16* d = dst + (size_t)blockIdx.z * rows * Kp;
    const bool vec = kin == 0 && (ld & 3) == 0 && (bstride & 3) == 0 && (reinterpret_cast<uintptr_t>(src) & 15) == 0;
    for (int r = blockIdx.y; r < rows; r += gridDim.y) {
        const float* srow = s + (size_t)r * ld;
        __nv_bfloat16* drow = d + (size_t)r * Kp;
        for (int k = (blockIdx.x * blockDim.x + threadIdx.x) * 8; k < Kp; k += gridDim.x * blockDim.x * 8) {
            float v[8];
            if (vec && k + 7 < K) {
                const float4 a = *reinterpret_cast<const float4*>(srow + k), b = *reinterpret_cast<const float4*>(srow + k + 4);
                v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
            } else {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int kk = k + j;
                    v[j] = 0.f;
                    if (kk < K) {
                        if (kin > 0) { const unsigned q = (unsigned)kk / (unsigned)kin; v[j] = srow[(size_t)q * kos + (kk - (int)q * kin)]; }   // slab q = k / kin
                        else v[j] = srow[kk];
                    }
                }
            }
            *reinterpret_cast<uint4*>(drow + k) = make_uint4(pack2(v[0], v[1]), pack2(v[2], v[3]), pack2(v[4], v[5]), pack2(v[6], v[7]));
        }
    }
}
// source element (r, k) at src[k*ld + r]: 32 (r) x 64 (k) tile transpose through shared memory; reads are 128-byte rows along r,
// writes are 128-byte rows along k (one bf16 pair per thread).  grid = (ceil(rows / 32), ceil(Kp / 64), batch), block = (32, 8).
__global__ void pack_transpose_kernel(__nv_bfloat16* __restrict__ dst, const float* __restrict__ src, int ld, long long bstride, int rows,
                                      int K, int Kp) {
    __shared__ float tile[64][33];
    const float* s = src + (size_t)blockIdx.z * bstride;
    __nv_bfloat16* d = dst + (size_t)blockIdx.z * rows * Kp;
    const int r0 = blockIdx.x * 32, k0 = blockIdx.y * 64;
    for (int j = threadIdx.y; j < 64; j += blockDim.y) {
        const int k = k0 + j, r = r0 + threadIdx.x;
        tile[j][threadIdx.x] = (k < K && r < rows) ? s[(size_t)k * ld + r] : 0.f;
    }
    __syncthreads();
    for (int j = threadIdx.y; j < 32; j += blockDim.y) {
        const int r = r0 + j, k = k0 + 2 * threadIdx.x;
        if (r < rows && k < Kp)        // Kp is even: the pair (k, k + 1) is inside the padded row
            *reinterpret_cast<uint32_t*>(d + (size_t)r * Kp + k) = pack2(tile[2 * threadIdx.x][j], tile[2 * threadIdx.x + 1][j]);
    }
}

// C = alpha * sum_z partial[z] + beta * C + bias   (fixed order over the splits: deterministic)
__global__ void tc_splitk_reduce_kernel(const float* __restrict__ partial, float* __restrict__ C, const float* __restrict__ bias, int M, int N,
                                        int ldc, int ksplit, float alpha, float beta) {
    const size_t total = (size_t)M * N;
    for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const int n = idx % N;
        const size_t m = idx / N;
        float s = 0.f;
        for (int z = 0; z < ksplit; ++z) s += partial[(size_t)z * total + idx];
        s *= alpha;
        if (bias) s += bias[n];
        float* c = C + m * ldc + n;
        if (beta != 0.f) s += beta * *c;
        *c = s;
    }
}

// Convolution weights W[g][co][ci][t] (fp32) -> bf16 A operands with K ordered (tap, channel):
//   forward : dst[g][co][t * Cin + ci]            (rows = output channels)
//   backward: dst[g][ci][t * Cout + co]           (rows = input channels: the input-gradient convolution)
__global__ void pack_conv_weight_kernel(__nv_bfloat16* __restrict__ dst, const float* __restrict__ w, int G, int Cout, int Cin, int k, int bwd,
                                        int colsP) {
    // block (x, row, g): one destination row [t][col] of k * colsP elements (columns >= cols are zero padding: channel counts that are no
    // multiple of the 64-wide k-block); 32-bit index arithmetic only
    const int rows = bwd ? Cin : Cout, cols = bwd ? Cout : Cin;
    const int row = blockIdx.y, g = blockIdx.z;
    __nv_bfloat16* drow = dst + ((size_t)g * rows + row) * (size_t)(k * colsP);
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < k * colsP; j += gridDim.x * blockDim.x) {
        const int t = j / colsP, col = j - t * colsP;
        const int co = bwd ? col : row, ci = bwd ? row : col;
        drow[j] = __float2bfloat16_rn(col < cols ? w[(((size_t)g * Cout + co) * Cin + ci) * k + t] : 0.f);
    }
}

// B operand of a convolution's weight gradient, straight from the block input (no materialised im2col):
//   dst[g][ci * k + t][q * L + l] = x[q][g * Cin + ci][l + t * dil - pad]   (zero outside [0, L)), bf16, K = NB * L contiguous (padded to Kp)
__global__ void pack_im2col_kcontig_kernel(__nv_bfloat16* __restrict__ dst, const float* __restrict__ x, int NB, int G, int Cin, int L, int k,
                                           int dil, int pad, int Kp) {
    const int R = Cin * k, g = blockIdx.z;
    __nv_bfloat16* d = dst + (size_t)g * R * Kp;
    for (int r = blockIdx.y; r < R; r += gridDim.y) {
        const int ci = r / k, t = r % k, shift = t * dil - pad;
        const float* xrow = x + ((size_t)g * Cin + ci) * L;             // + q * G * Cin * L per sample row
        __nv_bfloat16* drow = d + (size_t)r * Kp;
        for (int kk0 = (blockIdx.x * blockDim.x + threadIdx.x) * 8; kk0 < Kp; kk0 += gridDim.x * blockDim.x * 8) {
            float v[8];
            unsigned q = (unsigned)kk0 / (unsigned)L;
            int l = kk0 - (int)q * L;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int ls = l + shift;
                v[j] = (kk0 + j < NB * L && ls >= 0 && ls < L) ? xrow[(size_t)q * G * Cin * L + ls] : 0.f;
                if (++l == L) { l = 0; ++q; }
            }
            *reinterpret_cast<uint4*>(drow + kk0) = make_uint4(pack2(v[0], v[1]), pack2(v[2], v[3]), pack2(v[4], v[5]), pack2(v[6], v[7]));
        }
    }
}

// ------------------------------------------------------------------------------------------------
// host
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(ptr);
        else
            cudaGetLastError();
    }
    return fn;
}

int make_map(CUtensorMap* map, const __nv_bfloat16* base, int rows, int K, int Kp, int batch, int box_rows) {
    EncodeTiledFn fn = encode_fn();
    B200_REQUIRE(fn != nullptr, "gemm_tc: cuTensorMapEncodeTiled is unavailable");
    const cuuint64_t dims[3] = {(cuuint64_t)K, (cuuint64_t)rows, (cuuint64_t)batch};
    const cuuint64_t strides[2] = {(cuuint64_t)Kp * 2, (cuuint64_t)rows * Kp * 2};
    const cuuint32_t box[3] = {(cuuint32_t)TBK, (cuuint32_t)box_rows, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    const CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<__nv_bfloat16*>(base), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    B200_REQUIRE(r == CUDA_SUCCESS, "gemm_tc: cuTensorMapEncodeTiled failed with %d (rows=%d K=%d Kp=%d batch=%d)", (int)r, rows, K, Kp, batch);
    return B200TTS_OK;
}

struct Scratch { unsigned char* ptr = nullptr; size_t bytes = 0; };
Scratch g_scratch;

// Pack cache: inside a begin / end scope (one backward pass over buffers that do not change) a packed operand is kept in the scratch
// and reused by every later product that reads the same source view (e.g. the transposed gate gradients feed three weight-gradient
// GEMMs).  Outside a scope every call packs into the start of the scratch.
struct PackKey {
    const void* src; int ld, rows, K, Kp, kcontig, nb, kin; long long bstride, kos;
    bool operator==(const PackKey& o) const {
        return src == o.src && ld == o.ld && rows == o.rows && K == o.K && Kp == o.Kp && kcontig == o.kcontig && nb == o.nb && kin == o.kin &&
               bstride == o.bstride && kos == o.kos;
    }
};
struct PackEntry { PackKey key; __nv_bfloat16* dst; };
constexpr int MAX_CACHE = 32;
PackEntry g_cache[MAX_CACHE];
int g_ncache = 0;
bool g_cache_on = false;
size_t g_cache_off = 0;
int g_tc_enabled = 1;

}  // namespace

// 3-D bf16 tensor map {K, rows, batch} with a {64, box_rows, 1} box and SWIZZLE_128B (shared with the persistent loop kernels)
int tc_make_map_bf16(void* map, const void* base, int rows, int K, int Kp, int batch, int box_rows) {
    return make_map(static_cast<CUtensorMap*>(map), static_cast<const __nv_bfloat16*>(base), rows, K, Kp, batch, box_rows);
}

int tc_make_map3_bf16(void* map, const void* base, int d0, int d1, int d2, size_t stride1, size_t stride2, int b0, int b1, int b2) {
    EncodeTiledFn fn = encode_fn();
    B200_REQUIRE(fn != nullptr, "tc_make_map3: cuTensorMapEncodeTiled is unavailable");
    const cuuint64_t dims[3] = {(cuuint64_t)d0, (cuuint64_t)d1, (cuuint64_t)d2};
    const cuuint64_t strides[2] = {(cuuint64_t)stride1, (cuuint64_t)stride2};
    const cuuint32_t box[3] = {(cuuint32_t)b0, (cuuint32_t)b1, (cuuint32_t)b2};
    const cuuint32_t estr[3] = {1, 1, 1};
    const CUresult r = fn(static_cast<CUtensorMap*>(map), CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    B200_REQUIRE(r == CUDA_SUCCESS, "tc_make_map3: cuTensorMapEncodeTiled failed with %d (dims %d %d %d, strides %zu %zu, box %d %d %d)", (int)r,
                 d0, d1, d2, stride1, stride2, b0, b1, b2);
    return B200TTS_OK;
}

// rank-N (<= 5) bf16 tensor map, SWIZZLE_128B; dims / box: `rank` entries (innermost first), strides: rank - 1 byte strides
int tc_make_mapN_bf16(void* map, const void* base, int rank, const unsigned long long* dims, const unsigned long long* strides, const unsigned* box) {
    EncodeTiledFn fn = encode_fn();
    B200_REQUIRE(fn != nullptr, "tc_make_mapN: cuTensorMapEncodeTiled is unavailable");
    B200_REQUIRE(rank >= 1 && rank <= 5, "tc_make_mapN: rank %d", rank);
    cuuint64_t d[5], s[4];
    cuuint32_t b[5], e[5];
    for (int i = 0; i < rank; ++i) { d[i] = dims[i]; b[i] = box[i]; e[i] = 1; }
    for (int i = 0; i + 1 < rank; ++i) s[i] = strides[i];
    const CUresult r = fn(static_cast<CUtensorMap*>(map), CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), d, s, b, e,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    B200_REQUIRE(r == CUDA_SUCCESS, "tc_make_mapN: cuTensorMapEncodeTiled failed with %d (rank %d)", (int)r, rank);
    return B200TTS_OK;
}

void set_tc_scratch(void* ptr, size_t bytes) { g_scratch.ptr = static_cast<unsigned char*>(ptr); g_scratch.bytes = bytes; g_ncache = 0; g_cache_off = 0; }
void tc_pack_cache_begin() { g_cache_on = true; g_ncache = 0; g_cache_off = 0; }
void tc_pack_cache_end() { g_cache_on = false; g_ncache = 0; g_cache_off = 0; }
void set_tc_enabled(int on) { g_tc_enabled = on; }
int tc_enabled() { return g_tc_enabled; }

// Returns B200TTS_OK and sets *handled = true when the tcgen05 path ran; *handled = false -> caller uses the mma.sync path.
// Split-K decision shared by the dense and the convolution weight-gradient products: with fewer output tiles than CTA slots (2 per SM)
// and a long K, K is cut into `splits` ranges of `kper` k-blocks; the partial tiles live at the END of the scratch, clear of the
// packed (and cached) operands that occupy its first `used` bytes.  Leaves a.ksplit = 1 when it does not pay or does not fit.
static void pick_ksplit(TcArgs& a, int M, int N, int K, size_t used) {
    const int tiles = cdiv(N, TBN) * cdiv(M, TBM), nk = cdiv(K, TBK);
    if (tiles > 148 || nk < 64) return;
    int want = 296 / tiles;
    if (want > nk / 16) want = nk / 16;
    if (want > 32) want = 32;
    if (want < 2) return;
    const int kper = cdiv(nk, want), splits = cdiv(nk, kper);
    const size_t pbytes = (size_t)splits * M * N * 4;
    if (splits >= 2 && used + pbytes + 1024 <= g_scratch.bytes) {
        a.ksplit = splits; a.kper = kper;
        a.partial = reinterpret_cast<float*>(g_scratch.ptr + ((g_scratch.bytes - pbytes) & ~(size_t)1023));
    }
}

int gemm_tc_try(const GemmDesc& d, cudaStream_t st, bool* handled) {
    *handled = false;
    if (!g_tc_enabled || g_scratch.ptr == nullptr) return B200TTS_OK;
    if (d.splitk != 1 || d.keep_partials) return B200TTS_OK;
    if (d.kin > 0 && (d.transA || !d.transB || d.K % d.kin != 0 || d.A16)) return B200TTS_OK;      // two-level K: K-contiguous operands only
    if (d.M < 64 || d.N < 64 || d.K < 32) return B200TTS_OK;                 // tiny problems: not worth packing
    if ((long long)d.M * d.N * d.K * d.batch < (1ll << 24)) return B200TTS_OK;
    const int Kp = (d.K + 7) / 8 * 8;
    const int abatch = d.a_batch_mod > 0 ? d.a_batch_mod : d.batch;
    const bool a16ok = d.A16 != nullptr && d.batch == 1 && (d.lda16 % 8) == 0 && (reinterpret_cast<uintptr_t>(d.A16) & 15) == 0;
    // A16 with transA: the bf16 matrix is [K, M] row-major (e.g. the gate-gradient history of the reverse loops) = an MN-major operand in place
    const bool a_mn_ready = a16ok && d.transA && d.kin == 0 && (d.lda16 % 64) == 0 && !getenv("B200TTS_NO_MN_MAJOR");
    const bool a_ready = (a16ok && !d.transA) || a_mn_ready;
    // MN-major operands (op(A) = A^T with A [K, M], op(B) = B [K, N]: weight gradients): the bf16 copy keeps the source's row-major
    // [K][MN] layout (a plain row conversion, no transpose; MN padded to 64) and is keyed exactly like the K-contiguous copy another product
    // makes of the same matrix, so e.g. the gate gradients are converted ONCE for their dX (K-major use) and dW (MN-major use) products
    const bool a_mn = d.transA && !a_ready && d.batch == 1 && d.kin == 0 && !getenv("B200TTS_NO_MN_MAJOR");
    const bool b_mn = !d.transB && d.batch == 1 && d.kin == 0 && !getenv("B200TTS_NO_MN_MAJOR");
    const bool b_ready = b_mn && d.B16 != nullptr && (d.ldb16 % 64) == 0 && (reinterpret_cast<uintptr_t>(d.B16) & 15) == 0;
    const int Mp64 = (d.M + 63) / 64 * 64, Np64 = (d.N + 63) / 64 * 64;
    const size_t a_bytes = a_ready ? 0 : a_mn ? ((size_t)d.K * Mp64 * 2 + 1023) / 1024 * 1024 : ((size_t)abatch * d.M * Kp * 2 + 1023) / 1024 * 1024;
    const size_t b_bytes = b_ready ? 0 : b_mn ? ((size_t)d.K * Np64 * 2 + 1023) / 1024 * 1024 : ((size_t)d.batch * d.N * Kp * 2 + 1023) / 1024 * 1024;
    if ((reinterpret_cast<uintptr_t>(g_scratch.ptr) & 1023) != 0) return B200TTS_OK;
    const PackKey ka = a_mn ? PackKey{d.A, d.lda, d.K, d.M, Mp64, 1, 1, 0, 0, 0} : PackKey{d.A, d.lda, d.M, d.K, Kp, !d.transA, abatch, d.kin, d.strideA, d.kosA};
    const PackKey kb = b_mn ? PackKey{d.B, d.ldb, d.K, d.N, Np64, 1, 1, 0, 0, 0} : PackKey{d.B, d.ldb, d.N, d.K, Kp, d.transB != 0, d.batch, d.kin, d.strideB, d.kosB};
    auto cached = [&](const PackKey& k) -> __nv_bfloat16* {
        if (!g_cache_on) return nullptr;
        for (int e = 0; e < g_ncache; ++e)
            if (g_cache[e].key == k) return g_cache[e].dst;
        return nullptr;
    };
    __nv_bfloat16* pa = a_ready ? nullptr : cached(ka);
    __nv_bfloat16* pb = b_ready ? nullptr : cached(kb);
    const bool pack_a = !a_ready && pa == nullptr, pack_b = !b_ready && pb == nullptr;
    {   // place what has to be packed now: behind the cached operands (kept, when a scope is open and there is room for more)
        size_t off = g_cache_on ? g_cache_off : 0;
        const size_t need = (pack_a ? a_bytes : 0) + (pack_b ? b_bytes : 0);
        if (off + need > g_scratch.bytes) return B200TTS_OK;
        if (pack_a) { pa = reinterpret_cast<__nv_bfloat16*>(g_scratch.ptr + off); off += a_bytes; }
        if (pack_b) { pb = reinterpret_cast<__nv_bfloat16*>(g_scratch.ptr + off); off += b_bytes; }
        // keep them only if the largest operand of this backward pass would still fit behind (otherwise the region is reused as scratch)
        if (g_cache_on && g_ncache + 2 <= MAX_CACHE && off + (g_scratch.bytes >> 2) <= g_scratch.bytes) {
            if (pack_a) g_cache[g_ncache++] = PackEntry{ka, pa};
            if (pack_b) g_cache[g_ncache++] = PackEntry{kb, pb};
            g_cache_off = off;
        }
    }

    auto pack = [&](__nv_bfloat16* dst, const float* src, int ld, long long bstride, int rows, bool kcontig, int nb, long long kos) -> int {
        if (kcontig) {
            const int gx = Kp > 32768 ? 16 : cdiv(Kp, 2048);
            pack_kcontig_kernel<<<dim3(gx, rows < 32768 ? rows : 32768, nb), 256, 0, st>>>(dst, src, ld, bstride, rows, d.K, Kp, d.kin, kos);
        } else {
            dim3 grid(cdiv(rows, 32), cdiv(Kp, 64), nb), block(32, 8);
            pack_transpose_kernel<<<grid, block, 0, st>>>(dst, src, ld, bstride, rows, d.K, Kp);
        }
        B200_LAUNCH_CHECK();
        return B200TTS_OK;
    };
    // row conversion of an MN-major source: `rows` = K lines of `cols` = M (or N) values, zero-padded to `colsP`
    auto pack_rows = [&](__nv_bfloat16* dst, const float* src, int ld, int rows, int cols, int colsP) -> int {
        const int gx = colsP > 32768 ? 16 : cdiv(colsP, 2048);
        pack_kcontig_kernel<<<dim3(gx, rows < 32768 ? rows : 32768, 1), 256, 0, st>>>(dst, src, ld, 0, rows, cols, colsP, 0, 0);
        B200_LAUNCH_CHECK();
        return B200TTS_OK;
    };
    if (pack_a) B200_TRY(a_mn ? pack_rows(pa, d.A, d.lda, d.K, d.M, Mp64) : pack(pa, d.A, d.lda, d.strideA, d.M, !d.transA, abatch, d.kosA));
    if (pack_b) B200_TRY(b_mn ? pack_rows(pb, d.B, d.ldb, d.K, d.N, Np64) : pack(pb, d.B, d.ldb, d.strideB, d.N, d.transB != 0, d.batch, d.kosB));

    CUtensorMap tmA, tmB;
    if (a_mn_ready) B200_TRY(tc_make_map3_bf16(&tmA, d.A16, 64, d.K, Mp64 / 64, (size_t)d.lda16 * 2, 128, 64, 64, 2));
    else if (a_ready) B200_TRY(make_map(&tmA, static_cast<const __nv_bfloat16*>(d.A16), d.M, d.K, d.lda16, 1, TBM));
    else if (a_mn) B200_TRY(tc_make_map3_bf16(&tmA, pa, 64, d.K, Mp64 / 64, (size_t)Mp64 * 2, 128, 64, 64, 2));
    else B200_TRY(make_map(&tmA, pa, d.M, d.K, Kp, abatch, TBM));
    if (b_ready) B200_TRY(tc_make_map3_bf16(&tmB, d.B16, 64, d.K, Np64 / 64, (size_t)d.ldb16 * 2, 128, 64, 64, 2));
    else if (b_mn) B200_TRY(tc_make_map3_bf16(&tmB, pb, 64, d.K, Np64 / 64, (size_t)Np64 * 2, 128, 64, 64, 2));
    else B200_TRY(make_map(&tmB, pb, d.N, d.K, Kp, d.batch, TBN));
    TcArgs a;
    a.C = d.C; a.bias = d.bias; a.M = d.M; a.N = d.N; a.K = d.K; a.ldc = d.ldc; a.alpha = d.alpha; a.beta = d.beta;
    a.batch = d.batch; a.a_batch_mod = d.a_batch_mod; a.strideC = d.strideC;
    a.conv_cb = 0; a.conv_dil = 0; a.conv_pad = 0; a.conv_G = 1; a.conv_cin = 0;
    a.ksplit = 1; a.kper = 0; a.partial = nullptr; a.a_mn = (a_mn || a_mn_ready) ? 1 : 0; a.b_mn = b_mn ? 1 : 0;
    // few output tiles and a long K (weight gradients over all (step, utterance) rows): split K over the idle SMs
    if (d.batch == 1)
        pick_ksplit(a, d.M, d.N, d.K, (g_cache_on ? g_cache_off : 0) + (pack_a ? a_bytes : 0) + (pack_b ? b_bytes : 0));
    const size_t smem = (size_t)STAGES * STAGE_BYTES + 1024;
    static bool configured = false;
    if (!configured) {
        B200_CUDA(cudaFuncSetAttribute(gemm_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured = true;
    }
    dim3 grid(cdiv(d.N, TBN), cdiv(d.M, TBM), a.ksplit > 1 ? a.ksplit : d.batch);
    {
        KernelTimer kt("gemm_tc_kernel", st);
        gemm_tc_kernel<<<grid, TC_THREADS, smem, st>>>(tmA, tmB, a);
    }
    B200_LAUNCH_CHECK();
    if (a.ksplit > 1) {
        const size_t total = (size_t)d.M * d.N;
        int blocks = (int)((total + 255) / 256);
        if (blocks > 148 * 8) blocks = 148 * 8;
        tc_splitk_reduce_kernel<<<blocks, 256, 0, st>>>(a.partial, d.C, d.bias, d.M, d.N, d.ldc, a.ksplit, d.alpha, d.beta);
        B200_LAUNCH_CHECK();
    }
    *handled = true;
    return B200TTS_OK;
}


// Implicit 1-D convolution on the tcgen05 GEMM (no im2col):  out[row, g][m, l] (+)= sum_{t, c} Wp[g][m][t * Cred + c] . in[row][g * Cred + c][l + t * dil - pad]
//   forward        : Wp = weights packed (co, t, ci), in = x,        Cred = Cin,  rows m = Cout, dil/pad as given
//   input gradient : Wp = weights packed (ci, t, co), in = d conv,   Cred = Cout, rows m = Cin,  dil -> -dil, pad -> -pad
// `in` is [NB, G * Cred, L] fp32; its position-major bf16 copy [NB][L][G * Cred] is made here (one transposing pass, 1x the activation).
// out is [NB * G][Mrows][L] fp32 with row stride L.  Declines (handled = false) when the shape does not fit the tiling.
int gemm_tc_conv(const float* weight, const float* in, float* out, int NB, int G, int Cout, int Cin, int L, int k, int dil, int pad, int bwd,
                 float beta, cudaStream_t st, bool* handled) {
    *handled = false;
    const int Cred = bwd ? Cout : Cin, Mrows = bwd ? Cin : Cout;
    if (!g_tc_enabled || g_scratch.ptr == nullptr || g_cache_on) return B200TTS_OK;
    // reduction channels are processed in 64-wide k-blocks; an ungrouped convolution with another channel count (the 80 mel channels of the
    // postnet's first / last layer) is zero-padded to the next multiple in the bf16 operand copies
    const int CredP = (Cred + TBK - 1) / TBK * TBK;
    if ((CredP != Cred && G != 1) || Mrows < 64 || L < 64 || k < 1) return B200TTS_OK;
    if ((reinterpret_cast<uintptr_t>(g_scratch.ptr) & 1023) != 0) return B200TTS_OK;
    const int K = k * CredP, Ctot = G * CredP;
    const size_t a_bytes = ((size_t)G * Mrows * K * 2 + 1023) / 1024 * 1024;
    const size_t b_bytes = ((size_t)NB * L * Ctot * 2 + 1023) / 1024 * 1024;
    if (a_bytes + b_bytes > g_scratch.bytes) return B200TTS_OK;
    __nv_bfloat16* pa = reinterpret_cast<__nv_bfloat16*>(g_scratch.ptr);
    __nv_bfloat16* pb = reinterpret_cast<__nv_bfloat16*>(g_scratch.ptr + a_bytes);
    {
        const int prow = bwd ? Cin : Cout;
        pack_conv_weight_kernel<<<dim3(cdiv((long long)k * CredP, 256 * 4), prow, G), 256, 0, st>>>(pa, weight, G, Cout, Cin, k, bwd, CredP);
        B200_LAUNCH_CHECK();
        // position-major copy: element (row = l, k = channel) of sample n at in[n][channel][l]; channels >= G * Cred are zero padding
        dim3 grid(cdiv(L, 32), cdiv(Ctot, 64), NB), block(32, 8);
        pack_transpose_kernel<<<grid, block, 0, st>>>(pb, in, L, (long long)G * Cred * L, L, G * Cred, Ctot);
        B200_LAUNCH_CHECK();
    }
    CUtensorMap tmA, tmB;
    B200_TRY(make_map(&tmA, pa, Mrows, K, K, G, TBM));
    B200_TRY(make_map(&tmB, pb, L, Ctot, Ctot, NB, TBN));
    TcArgs a;
    a.C = out; a.bias = nullptr; a.M = Mrows; a.N = L; a.K = K; a.ldc = L; a.alpha = 1.f; a.beta = beta;
    a.batch = NB * G; a.a_batch_mod = G; a.strideC = (long long)Mrows * L;
    a.conv_cb = CredP / TBK; a.conv_dil = bwd ? -dil : dil; a.conv_pad = bwd ? -pad : pad; a.conv_G = G; a.conv_cin = CredP;
    a.ksplit = 1; a.kper = 0; a.partial = nullptr; a.a_mn = 0; a.b_mn = 0;
    const size_t smem = (size_t)STAGES * STAGE_BYTES + 1024;
    B200_CUDA(cudaFuncSetAttribute(gemm_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid(cdiv(L, TBN), cdiv(Mrows, TBM), NB * G);
    {
        KernelTimer kt("gemm_tc_kernel", st);
        gemm_tc_kernel<<<grid, TC_THREADS, smem, st>>>(tmA, tmB, a);
    }
    B200_LAUNCH_CHECK();
    *handled = true;
    return B200TTS_OK;
}


// Weight gradient of a 1-D convolution in ONE batched tcgen05 GEMM:  dW[g][co][ci * k + t] += sum_{q, l} dz[q][g, co][l] . x[q][g, ci][l + t dil - pad].
// A = dz packed with a two-level K (sample row, position); B = the shifted input packed straight from x (pack_im2col_kcontig_kernel).
int gemm_tc_conv_dw(const float* dz, const float* x, float* dweight, int NB, int G, int Cout, int Cin, int L, int k, int dil, int pad,
                    cudaStream_t st, bool* handled) {
    *handled = false;
    if (!g_tc_enabled || g_scratch.ptr == nullptr || g_cache_on) return B200TTS_OK;
    const int R = Cin * k, K = NB * L, Kp = (K + 7) / 8 * 8;
    if (Cout < 64 || R < 64 || K < 64) return B200TTS_OK;
    if ((reinterpret_cast<uintptr_t>(g_scratch.ptr) & 1023) != 0) return B200TTS_OK;
    const size_t a_bytes = ((size_t)G * Cout * Kp * 2 + 1023) / 1024 * 1024;
    const size_t b_bytes = ((size_t)G * R * Kp * 2 + 1023) / 1024 * 1024;
    if (a_bytes + b_bytes > g_scratch.bytes) return B200TTS_OK;
    __nv_bfloat16* pa = reinterpret_cast<__nv_bfloat16*>(g_scratch.ptr);
    __nv_bfloat16* pb = reinterpret_cast<__nv_bfloat16*>(g_scratch.ptr + a_bytes);
    {
        pack_kcontig_kernel<<<dim3(Kp > 32768 ? 16 : cdiv(Kp, 2048), Cout, G), 256, 0, st>>>(pa, dz, L, (long long)Cout * L, Cout, K, Kp, L,
                                                                                             (long long)G * Cout * L);
        B200_LAUNCH_CHECK();
        pack_im2col_kcontig_kernel<<<dim3(Kp > 32768 ? 16 : cdiv(Kp, 2048), R, G), 256, 0, st>>>(pb, x, NB, G, Cin, L, k, dil, pad, Kp);
        B200_LAUNCH_CHECK();
    }
    CUtensorMap tmA, tmB;
    B200_TRY(make_map(&tmA, pa, Cout, K, Kp, G, TBM));
    B200_TRY(make_map(&tmB, pb, R, K, Kp, G, TBN));
    TcArgs a;
    a.C = dweight; a.bias = nullptr; a.M = Cout; a.N = R; a.K = K; a.ldc = R; a.alpha = 1.f; a.beta = 1.f;
    a.batch = G; a.a_batch_mod = 0; a.strideC = (long long)Cout * R;
    a.conv_cb = 0; a.conv_dil = 0; a.conv_pad = 0; a.conv_G = 1; a.conv_cin = 0;
    a.ksplit = 1; a.kper = 0; a.partial = nullptr; a.a_mn = 0; a.b_mn = 0;
    if (G == 1) pick_ksplit(a, Cout, R, K, a_bytes + b_bytes);      // postnet convolutions: 16 .. 80 tiles over K = NB * L
    const size_t smem = (size_t)STAGES * STAGE_BYTES + 1024;
    B200_CUDA(cudaFuncSetAttribute(gemm_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid(cdiv(R, TBN), cdiv(Cout, TBM), a.ksplit > 1 ? a.ksplit : G);
    {
        KernelTimer kt("gemm_tc_kernel", st);
        gemm_tc_kernel<<<grid, TC_THREADS, smem, st>>>(tmA, tmB, a);
    }
    B200_LAUNCH_CHECK();
    if (a.ksplit > 1) {
        const size_t total = (size_t)Cout * R;
        int blocks = (int)((total + 255) / 256);
        if (blocks > 148 * 8) blocks = 148 * 8;
        tc_splitk_reduce_kernel<<<blocks, 256, 0, st>>>(a.partial, dweight, nullptr, Cout, R, R, a.ksplit, 1.f, 1.f);
        B200_LAUNCH_CHECK();
    }
    *handled = true;
    return B200TTS_OK;
}

}  // namespace b200tts
