// Persistent generator-LSTM BACKWARD loop of the bf16 perf mode on TMA + tcgen05 + TMEM (sm_100a).
//
// Reverse step i needs  d h_{i-1}[b, n] = sum_r dgates_i[b, r] . W_hh[r, n]  (r over the 4D gate rows): the transpose of the forward
// product.  CTA (gate g, n-block nb, batch half bh) keeps W_hh^T[n-block (64 outputs), gate g (D rows of K)] in shared memory as
// K-major SWIZZLE_128B tiles (A operand, M = 64); per step ONE TMA box brings the bf16 gate gradients [32 utterances x D] of its
// gate (B operand, N = 32); D / 16 tcgen05 MMAs accumulate in TMEM; the epilogue stores the fp32 partial [gate][b][n] that the next
// step's cell backward sums over the 4 gates (fixed order, no atomics).  Per step:
//   P1  cell backward of this CTA's 16 hidden units x 32 utterances (operands prefetched during the previous product)
//   --  grid barrier (gate gradients of all units visible)
//   P2  TMA + tcgen05 product, TMEM -> partial store
//   --  grid barrier.
// Warp roles as in decoder_persist_tc.cu: warps 0-7 compute, warp 8 = TMA producer, warp 9 = MMA issuer (one elected lane each).
// Reference semantics: autograd replay of modules/layers.py:18-47 (train.py:83).
#include <cuda.h>
#include <cuda_bf16.h>
#include "decoder_internal.cuh"
#include "persist.cuh"

namespace b200tts {

namespace {

constexpr int NCW = 8;
constexpr int CT = 32 * NCW;
constexpr int PT = CT + 64;
constexpr int UNITS = 16;               // hidden units of the cell backward per CTA
constexpr int ROWS = 64;                // outputs (n) per CTA = MMA M
constexpr int BT = 32;                  // utterances per CTA = MMA N
constexpr int KB = 64;
constexpr int WTILE = ROWS * KB * 2;
constexpr int ATILE = BT * KB * 2;
constexpr int TMEM_COLS = 32;
constexpr int NG = 4;                   // gates = K blocks of the product

struct TcBwdArgs {
    int B, T, D, NNB, NBH;                    // NNB = D / 64 n-blocks
    const float* W; int ldw;                  // fp32 [4D, ldw]: dgates . W
    const float* gates; const float* cstate; const float* dh_static;
    const uint8_t* mask_h; const uint8_t* mask_c;
    int kind, training; float rate_h, rate_c;
    float* dgates;                            // [T, B, 4D] out (fp32)
    __nv_bfloat16* dgb;                       // [B, 4D] staging (bf16), TMA source -- or a [T, B, 4D] history (dgb_step = B * 4D, dgb_rows = B)
    long long dgb_step; int dgb_rows;
    float* part;                              // [NG, B, D] partial products of the previous reverse step
    unsigned* barrier; int* abort_flag;
    long long* prof;
};

using namespace tcx;

__global__ void __launch_bounds__(PT, 1) lstm_bwd_loop_tc_kernel(const __grid_constant__ CUtensorMap tmG, const TcBwdArgs p) {
    extern __shared__ __align__(1024) unsigned char smem_raw0[];
    unsigned char* smem_raw = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw0) + 1023) & ~(uintptr_t)1023);
    __shared__ uint64_t full_bar, accum_bar;
    __shared__ uint32_t tmem_base_s;
    __shared__ int s_ok;

    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const int cta = blockIdx.x;
    const int gsel = cta % NG, nb = (cta / NG) % p.NNB, bh = cta / (NG * p.NNB);
    const int B = p.B, D = p.D, NNB = p.NNB;
    const int b0 = bh * BT, n0 = nb * ROWS;
    const int u0 = (gsel * NNB + nb) * UNITS;                 // hidden units whose cell backward this CTA owns
    // batch halves are independent (cell backward and product of a CTA serve the same 32 utterances): one barrier counter per half
    // (per-batch-half barrier counters were measured SLOWER than one grid-wide counter: +0.9 ms on the attention loop; the cost of a
    // barrier is its latency chain -- store acks, atomic round trip, poll -- not the number of arrivals: tools/microbench/barrier_latency.cu)
    const unsigned nblocks = gridDim.x;
    unsigned* const bar_counter = p.barrier;
    const bool compute = warp < NCW, is_producer = warp == NCW, is_mma = warp == NCW + 1;

    unsigned char* sW = smem_raw;                              // [NNB][64 rows (n)][128 B] swizzled: W^T[n0 + r, gate gsel, k]
    unsigned char* ring = smem_raw + (size_t)NNB * WTILE;      // [NNB][32 rows (b)][128 B] swizzled (one TMA box)

    // ---- one-time: resident transposed weight block, fp32 -> bf16, canonical K-major SWIZZLE_128B layout (n fastest: coalesced reads) ----
    for (int idx = tid; idx < ROWS * D; idx += PT) {
        const int k = idx / ROWS, r = idx % ROWS;
        const float w = (n0 + r < D) ? p.W[(size_t)(gsel * D + k) * p.ldw + n0 + r] : 0.f;
        const int kb = k / KB, kc = k % KB, chunk = kc >> 3, e = kc & 7;
        *reinterpret_cast<__nv_bfloat16*>(sW + (size_t)kb * WTILE + r * 128 + ((chunk ^ (r & 7)) << 4) + e * 2) = __float2bfloat16_rn(w);
    }
    if (tid == 0) {
        mbar_init(&full_bar, 1); mbar_init(&accum_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == NCW + 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "n"(TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    proxy_fence_shared();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;
    const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BT >> 3) << 17) | ((uint32_t)(ROWS >> 4) << 24);

    const float inv_h = 1.f / (1.f - p.rate_h), inv_c = 1.f / (1.f - p.rate_c);
    // cell-backward operands of this thread's two (b, u) pairs, fetched one step ahead (during the previous product)
    float gi_[2], gf_[2], gg_[2], go_[2], cp_[2], dhs_[2];
    uint8_t mh_[2], mc_[2];
    float dc_reg[2] = {0.f, 0.f}, dhz_reg[2] = {0.f, 0.f};
    auto prefetch = [&](int step) {
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int idx = tid + e * CT;
            const int bl = idx / UNITS, uu = idx % UNITS, b = b0 + bl, u = u0 + uu;
            gi_[e] = gf_[e] = gg_[e] = go_[e] = cp_[e] = dhs_[e] = 0.f; mh_[e] = 1; mc_[e] = 1;
            if (b < B && u < D) {
                const size_t g0 = ((size_t)step * B + b) * 4 * D + u, mi = ((size_t)step * B + b) * D + u;
                gi_[e] = p.gates[g0]; gf_[e] = p.gates[g0 + D]; gg_[e] = p.gates[g0 + 2 * D]; go_[e] = p.gates[g0 + 3 * D];
                cp_[e] = p.cstate[mi];
                dhs_[e] = p.dh_static[mi];
                if (p.training && p.mask_h) mh_[e] = p.mask_h[mi];
                if (p.training && p.mask_c) mc_[e] = p.mask_c[mi];
            }
        }
    };
    auto prefetch_l2 = [&](int step) {
        if (step < 0) return;
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int idx = tid + e * CT;
            const int bl = idx / UNITS, uu = idx % UNITS, b = b0 + bl, u = u0 + uu;
            if (b < B && u < D && (uu & 7) == 0) {
                const size_t g0 = ((size_t)step * B + b) * 4 * D + u, mi = ((size_t)step * B + b) * D + u;
                l2_prefetch(p.gates + g0); l2_prefetch(p.gates + g0 + D); l2_prefetch(p.gates + g0 + 2 * D); l2_prefetch(p.gates + g0 + 3 * D);
                l2_prefetch(p.cstate + mi); l2_prefetch(p.dh_static + mi);
                if (uu == 0 && p.training && p.mask_h) l2_prefetch(p.mask_h + mi);
                if (uu == 0 && p.training && p.mask_c) l2_prefetch(p.mask_c + mi);
            }
        }
    };
    if (compute) { prefetch(p.T - 1); prefetch_l2(p.T - 2); }

    unsigned target = 0;
    uint32_t it = 0;                         // products done (mbarrier phase)
    PROF_DECL

    for (int i = p.T - 1; i >= 0; --i) {
        const bool last = (i == p.T - 1);
        // ---------------- P1: LSTM cell backward (2 (b, u) pairs per compute thread) ----------------
        if (compute) {
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int idx = tid + e * CT;
                const int bl = idx / UNITS, uu = idx % UNITS, b = b0 + bl, u = u0 + uu;
                if (b < B && u < D) {
                    const size_t g0 = ((size_t)i * B + b) * 4 * D + u;
                    float dh = dhs_[e];
                    float dc_in = 0.f;
                    if (!last) {
                        float r4[NG];
#pragma unroll
                        for (int k2 = 0; k2 < NG; ++k2) r4[k2] = __ldcg(p.part + ((size_t)k2 * B + b) * D + u);
                        dh += ((r4[0] + r4[1]) + (r4[2] + r4[3])) + dhz_reg[e];
                        dc_in = dc_reg[e];
                    }
                    const float gi = gi_[e], gf = gf_[e], gg = gg_[e], go = go_[e], cp = cp_[e];
                    const float tc = tanh_exp(gf * cp + gi * gg);
                    float dhn, dcn, dc_prev_direct = 0.f, dh_prev_direct = 0.f;
                    if (p.kind == B200TTS_CELL_ZONEOUT) {
                        float kh, kc;
                        if (p.training) {
                            kh = (1.f - p.rate_h) * (p.mask_h ? (float)mh_[e] * inv_h : 1.f);
                            kc = (1.f - p.rate_c) * (p.mask_c ? (float)mc_[e] * inv_c : 1.f);
                        } else { kh = 1.f - p.rate_h; kc = 1.f - p.rate_c; }
                        dhn = dh * kh; dh_prev_direct = dh - dhn;
                        dcn = dc_in * kc + dhn * go * (1.f - tc * tc);
                        dc_prev_direct = dc_in - dc_in * kc;
                    } else {
                        dhn = (p.training && p.mask_h) ? dh * (float)mh_[e] * inv_h : dh;
                        dcn = dc_in + dhn * go * (1.f - tc * tc);
                    }
                    const float di = dcn * gg * gi * (1.f - gi), df = dcn * cp * gf * (1.f - gf);
                    const float dg = dcn * gi * (1.f - gg * gg), dO = dhn * tc * go * (1.f - go);
                    p.dgates[g0] = di; p.dgates[g0 + D] = df; p.dgates[g0 + 2 * D] = dg; p.dgates[g0 + 3 * D] = dO;
                    __nv_bfloat16* db = p.dgb + (size_t)i * p.dgb_step + (size_t)b * 4 * D + u;
                    db[0] = __float2bfloat16_rn(di); db[D] = __float2bfloat16_rn(df);
                    db[2 * D] = __float2bfloat16_rn(dg); db[3 * D] = __float2bfloat16_rn(dO);
                    dc_reg[e] = dcn * gf + dc_prev_direct;
                    dhz_reg[e] = dh_prev_direct;
                }
            }
        }
        PROF_MARK(0);
        if (!grid_barrier<true>(bar_counter, target, nblocks, p.abort_flag, &s_ok)) break;
        PROF_MARK(1);
        if (i == 0) break;

        // ---------------- P2: partial[gate] = dgates[:, gate block] . W[gate block, n-block]  (TMA + tcgen05) ----------------
        if (is_producer) {
            proxy_fence_global();
            if (elect_one()) {
                mbar_expect_tx(&full_bar, (uint32_t)NNB * ATILE);
                tma_load_3d(ring, &tmG, &full_bar, 0, i * p.dgb_rows + b0, gsel * NNB);
            }
            __syncwarp();
        }
        if (is_mma) {
            mbar_wait(&full_bar, it & 1);
            tc_fence_after();
            if (elect_one()) {
                for (int c = 0; c < NNB; ++c) {
                    const uint64_t adesc = make_sw128_desc(smem_u32(sW + (size_t)c * WTILE));
                    const uint64_t bdesc = make_sw128_desc(smem_u32(ring + (size_t)c * ATILE));
#pragma unroll
                    for (int k = 0; k < KB / 16; ++k) umma_bf16(tmem_base, adesc + 2 * k, bdesc + 2 * k, idesc, (c == 0 && k == 0) ? 0u : 1u);
                }
                umma_commit(&accum_bar);
            }
            __syncwarp();
        }
        if (compute) {
            prefetch(i - 1);                 // operands of the next cell backward: their latency hides behind the product
            prefetch_l2(i - 2);
            mbar_wait(&accum_bar, it & 1);
            tc_fence_after();
            PROF_MARK(2);
            const int q = warp & 3, c0 = (warp >> 2) * 16;
            uint32_t r[16];
            tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c0, r);
            if (lane < 16) {
                const int n = n0 + q * 16 + lane;
#pragma unroll
                for (int j = 0; j < 16; ++j)
                    if (b0 + c0 + j < B && n < D) p.part[((size_t)gsel * B + b0 + c0 + j) * D + n] = __uint_as_float(r[j]);
            }
            tc_fence_before();
        }
        ++it;
        PROF_MARK(3);
        if (!grid_barrier<true>(bar_counter, target, nblocks, p.abort_flag, &s_ok)) break;
        PROF_MARK(4);
    }
    PROF_FLUSH;
    tc_fence_before();
    __syncthreads();
    if (warp == NCW + 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS));
    }
}

size_t bwd_tc_smem_bytes(int D) { return 1024 + (size_t)(D / KB) * (WTILE + ATILE); }

}  // namespace

bool tc_persist_gen_bwd_supported(const b200tts_decoder_shape& s) {
    if (s.D % KB != 0 || s.D % (NG * (s.D / KB) * UNITS) != 0) return false;       // 4 x D/64 CTAs per batch half x 16 units = D
    const int NBH = (s.B + BT - 1) / BT;
    if (NG * (s.D / KB) * NBH > 148) return false;
    return bwd_tc_smem_bytes(s.D) <= 227 * 1024 - 1088;
}

// dgates for all T steps of the generator LSTM (tcgen05 variant); `extra` = persist_bwd_gen_extra_bytes scratch (same layout as the
// mma.sync variant: dgb [B, 4D] bf16, then the partial buffer (4 of its 8 slabs are used), then barrier + profile counters).
int tc_persist_gen_bwd_loop(const b200tts_decoder_shape& s, const b200tts_decoder_params& w, const b200tts_decoder_inputs& in,
                            const DecoderLayout& fl, const float* fws, const float* dh_static, float* dgates, unsigned char* extra,
                            cudaStream_t st, void* dgb_hist) {
    const int B = s.B, D = s.D;
    TcBwdArgs a{};
    a.B = B; a.T = s.T; a.D = D; a.NNB = D / KB; a.NBH = (B + BT - 1) / BT;
    a.W = w.gen_w_hh; a.ldw = D;
    a.gates = fws + fl.gg; a.cstate = fws + fl.cg; a.dh_static = dh_static;
    a.mask_h = in.mask_gen_h; a.mask_c = in.mask_gen_c; a.kind = s.cell_kind; a.training = s.training; a.rate_h = s.rate_h; a.rate_c = s.rate_c;
    a.dgates = dgates;
    size_t off = 0;
    a.dgb = dgb_hist ? static_cast<__nv_bfloat16*>(dgb_hist) : reinterpret_cast<__nv_bfloat16*>(extra + off);
    a.dgb_step = dgb_hist ? (long long)B * 4 * D : 0; a.dgb_rows = dgb_hist ? B : 0;
    off += ((size_t)B * 4 * D * 2 + 255) / 256 * 256;
    a.part = reinterpret_cast<float*>(extra + off); off += ((size_t)8 * B * D * 4 + 255) / 256 * 256;
    B200_TRY(reset_grid_barrier(extra + off, a, st));
    CUtensorMap tm;        // {64 columns, B rows, 4D/64 k-blocks}: k-block stride 128 B, row stride 4D * 2 B
    B200_TRY(tc_make_map3_bf16(&tm, a.dgb, KB, dgb_hist ? s.T * B : B, 4 * D / KB, (size_t)4 * D * 2, 128, KB, BT, a.NNB));
    const size_t smem = bwd_tc_smem_bytes(D);
    void* params[] = {&tm, &a};
    B200_TRY(launch_persistent((void*)lstm_bwd_loop_tc_kernel, NG * a.NNB * a.NBH, PT, smem, params, st, "tcgen05 persistent backward",
                               "lstm_bwd_loop_tc_kernel"));
    return B200TTS_OK;
}

}  // namespace b200tts
