// Persistent recurrent kernels of the bf16 perf mode (backward): reverse-time LSTM loops.
//
// Per reverse step the recurrence needs  d x_{i-1} = dgates_i . W   (K = 4D gate rows -> N output columns), the
// transpose of the forward product.  2-D weight-stationary partition: CTA (kb, nb, bh) keeps the bf16 block
// W[K-block kb (4 x UK gate rows), N-block nb] in shared memory for the whole sequence, owns a batch half, and
//   P1  runs the LSTM-cell backward for a 1/NB share of its K-block's hidden units (dgates -> fp32 for the dW GEMMs,
//       bf16 for the tensor cores),
//   --  grid barrier
//   P2  streams the bf16 dgates of its K-block (32 x 4UK) and multiplies (warps split N; ldmatrix.trans B fragments)
//       writing an fp32 partial [32 x UN] that the next step's P1 sums over the KB K-blocks (deterministic order),
//   --  grid barrier.
// Reference semantics: autograd replay of modules/layers.py:18-47 (train.py:83).
#include <stdlib.h>
#include <cuda_bf16.h>
#include "decoder_internal.cuh"
#include "persist.cuh"

namespace b200tts {

namespace {

constexpr int PT = 256;
constexpr int BT = 32;
constexpr int KB = 8;            // K-blocks (over hidden units)
constexpr int NBK = 8;           // N-blocks (over output columns)

struct BwdLoopArgs {
    int B, T, D, NOUT, UK, UN, NBH;        // NOUT output columns (D for the generator loop), UN = ceil(NOUT / NBK / 8) * 8
    const float* W; int ldw;               // fp32 [4D, ldw]: dgates . W
    const float* gates;                    // [T, B, 4D] activated gates (forward)
    const float* cstate;                   // [T+1, B, D]
    const float* dh_static;                // [T, B, D]
    const uint8_t* mask_h; const uint8_t* mask_c;
    int kind, training; float rate_h, rate_c;
    float* dgates;                         // [T, B, 4D] out (fp32)
    __nv_bfloat16* dgb;                    // [B, 4D] staging (bf16)
    float* part;                           // [KB, B, NOUT] partial products of the previous reverse step
    int hcol;                              // column of d h inside the NOUT outputs (0 for the generator loop)
    unsigned* barrier; int* abort_flag;
    long long* prof;
};

using namespace tcx;

// Generator-LSTM reverse loop (no attention): NOUT = D.
__global__ void __launch_bounds__(PT, 1) lstm_bwd_loop_kernel(const BwdLoopArgs p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int s_ok;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int cta = blockIdx.x;
    const int kb = cta % KB, nb = (cta / KB) % NBK, bh = cta / (KB * NBK);
    const int B = p.B, D = p.D, UK = p.UK, UN = p.UN, KROWS = 4 * UK;
    const int WLD = UN + 8, ALD = KROWS + 8;
    const int b0 = bh * BT, n0 = nb * UN;
    __nv_bfloat16* Ws = reinterpret_cast<__nv_bfloat16*>(smem_raw);                 // [KROWS][WLD]  (k rows, n contiguous)
    __nv_bfloat16* As = Ws + (size_t)KROWS * WLD;                                    // [BT][ALD]
    const unsigned nblocks = gridDim.x;

    // resident weight block: row r = g*UK + uk  <->  gate row g*D + kb*UK + uk ; column n <-> output n0 + n
    for (int idx = tid; idx < KROWS * UN; idx += PT) {
        const int r = idx / UN, n = idx % UN;
        const int g = r / UK, uk = r % UK;
        float w = 0.f;
        if (n0 + n < p.NOUT) w = p.W[(size_t)(g * D + kb * UK + uk) * p.ldw + n0 + n];
        Ws[r * WLD + n] = __float2bfloat16_rn(w);
    }
    __syncthreads();

    // P1 ownership: hidden units [kb*UK + nb*UP, +UP) with UP = UK / NBK, for the 32 utterances of this batch half
    const int UP = UK / NBK;
    const float inv_h = 1.f / (1.f - p.rate_h), inv_c = 1.f / (1.f - p.rate_c);
    constexpr int MAXE = 4;                       // (b, u) pairs per thread: BT * UP / PT  (UP <= 32)
    float dc_reg[MAXE], dhz_reg[MAXE];
#pragma unroll
    for (int e = 0; e < MAXE; ++e) { dc_reg[e] = 0.f; dhz_reg[e] = 0.f; }
    unsigned target = 0;
    PROF_DECL

    for (int i = p.T - 1; i >= 0; --i) {
        const bool last = (i == p.T - 1);
        // ---------------- P1: LSTM cell backward ----------------
#pragma unroll
        for (int e = 0; e < MAXE; ++e) {
            const int idx = tid + e * PT;
            if (idx < BT * UP) {
                const int bl = idx / UP, up = idx % UP, b = b0 + bl, u = kb * UK + nb * UP + up;
                if (b < B) {
                    const size_t bu = (size_t)b * D + u, g0 = ((size_t)i * B + b) * 4 * D + u;
                    float dh = p.dh_static[(size_t)i * B * D + bu];
                    float dc_in = 0.f;
                    if (!last) {
                        float rec = 0.f;
                        for (int k2 = 0; k2 < KB; ++k2) rec += __ldcg(p.part + ((size_t)k2 * B + b) * p.NOUT + p.hcol + u);
                        dh += rec + dhz_reg[e];
                        dc_in = dc_reg[e];
                    }
                    const float gi = p.gates[g0], gf = p.gates[g0 + D], gg = p.gates[g0 + 2 * D], go = p.gates[g0 + 3 * D];
                    const float cp = p.cstate[(size_t)i * B * D + bu];
                    const float tc = tanhf(gf * cp + gi * gg);
                    const size_t mi = (size_t)i * B * D + bu;
                    float dhn, dcn, dc_prev_direct = 0.f, dh_prev_direct = 0.f;
                    if (p.kind == B200TTS_CELL_ZONEOUT) {
                        float kh, kc;
                        if (p.training) {
                            kh = (1.f - p.rate_h) * (p.mask_h ? (float)p.mask_h[mi] * inv_h : 1.f);
                            kc = (1.f - p.rate_c) * (p.mask_c ? (float)p.mask_c[mi] * inv_c : 1.f);
                        } else { kh = 1.f - p.rate_h; kc = 1.f - p.rate_c; }
                        dhn = dh * kh; dh_prev_direct = dh - dhn;
                        dcn = dc_in * kc + dhn * go * (1.f - tc * tc);
                        dc_prev_direct = dc_in - dc_in * kc;
                    } else {
                        dhn = (p.training && p.mask_h) ? dh * (float)p.mask_h[mi] * inv_h : dh;
                        dcn = dc_in + dhn * go * (1.f - tc * tc);
                    }
                    const float di = dcn * gg * gi * (1.f - gi), df = dcn * cp * gf * (1.f - gf);
                    const float dg = dcn * gi * (1.f - gg * gg), dO = dhn * tc * go * (1.f - go);
                    p.dgates[g0] = di; p.dgates[g0 + D] = df; p.dgates[g0 + 2 * D] = dg; p.dgates[g0 + 3 * D] = dO;
                    __nv_bfloat16* db = p.dgb + (size_t)b * 4 * D + u;
                    db[0] = __float2bfloat16_rn(di); db[D] = __float2bfloat16_rn(df);
                    db[2 * D] = __float2bfloat16_rn(dg); db[3 * D] = __float2bfloat16_rn(dO);
                    dc_reg[e] = dcn * gf + dc_prev_direct;
                    dhz_reg[e] = dh_prev_direct;
                }
            }
        }
        PROF_MARK(0);
        if (!grid_barrier<false>(p.barrier, target, nblocks, p.abort_flag, &s_ok)) return;
        PROF_MARK(1);
        if (i == 0) break;

        // ---------------- P2: partial[kb] = dgates[:, K-block kb] . W[K-block kb, N-block nb] ----------------
        {
            const int segs = UK / 8;                       // 16-byte segments per gate block per row
            for (int idx = tid; idx < BT * 4 * segs; idx += PT) {
                const int r = idx / (4 * segs), rem = idx % (4 * segs), g = rem / segs, sg = rem % segs;
                __nv_bfloat16* d = As + r * ALD + g * UK + sg * 8;
                if (b0 + r < B) cp_async16(d, p.dgb + (size_t)(b0 + r) * 4 * D + g * D + kb * UK + sg * 8);
                else *reinterpret_cast<uint4*>(d) = make_uint4(0u, 0u, 0u, 0u);
            }
            cp_async_commit_wait();
            __syncthreads();
            // warps split N: warp w owns n-tile pairs {w, w+8, ...} (16 columns each)
            const int npairs = UN / 16;
            for (int np = warp; np < npairs; np += 8) {
                float acc[2][2][4];
#pragma unroll
                for (int mt = 0; mt < 2; ++mt)
#pragma unroll
                    for (int nt = 0; nt < 2; ++nt)
#pragma unroll
                        for (int e = 0; e < 4; ++e) acc[mt][nt][e] = 0.f;
                for (int kk = 0; kk < KROWS; kk += 16) {
                    uint32_t af[2][4], bf[4];
#pragma unroll
                    for (int mt = 0; mt < 2; ++mt)
                        ldmatrix_x4(af[mt][0], af[mt][1], af[mt][2], af[mt][3], As + (mt * 16 + (lane & 15)) * ALD + kk + (lane >> 4) * 8);
                    ldmatrix_x4_trans(bf[0], bf[1], bf[2], bf[3],
                                      Ws + (size_t)(kk + (lane & 7) + ((lane >> 3) & 1) * 8) * WLD + np * 16 + (lane >> 4) * 8);
#pragma unroll
                    for (int mt = 0; mt < 2; ++mt) {
                        mma_bf16(acc[mt][0], af[mt], bf[0], bf[1]);
                        mma_bf16(acc[mt][1], af[mt], bf[2], bf[3]);
                    }
                }
                const int g = lane >> 2, tq = lane & 3;
#pragma unroll
                for (int mt = 0; mt < 2; ++mt)
#pragma unroll
                    for (int nt = 0; nt < 2; ++nt)
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const int b = b0 + mt * 16 + g + 8 * (e >> 1);
                            const int n = n0 + np * 16 + nt * 8 + 2 * tq + (e & 1);
                            if (b < B && n < p.NOUT) p.part[((size_t)kb * B + b) * p.NOUT + n] = acc[mt][nt][e];
                        }
            }
        }
        if (!grid_barrier<false>(p.barrier, target, nblocks, p.abort_flag, &s_ok)) return;
    }
}


// =================================================================================================
// Attention-LSTM + attention reverse loop
// =================================================================================================
constexpr int KBA = 8;            // K-blocks of the attention-loop product (over hidden units)
constexpr int NBA = 9;            // N-blocks over the M + D output columns  -> 8 x 9 x 2 = 144 CTAs
constexpr int GLD = 33;           // row stride of the G tile buffer (floats)
// tcgen05 variant of the product: CTA (kb, nb) of 8 x 18 keeps W^T[n-block of 80 outputs, K-slice kb] as K-major SWIZZLE_128B tiles (UMMA B
// operand, N = 80); the whole batch (<= 64 utterances, TMA zero-fills the rest) is the A operand (M = 64), ONE 5-D TMA box per step
constexpr int NBT = 18;           // n-blocks of the tcgen05 variant  -> 8 x 18 = 144 CTAs (72 pairs)
constexpr int TUN = 80;           // outputs per n-block (UMMA N); TUN_WIDE when M + D > NBT * TUN (memory dim 512)
constexpr int TUN_WIDE = 96;
constexpr int TMEM_COLS_ATT = 128;

struct AttBwdArgs {
    int B, T, D, M, L, A, KC, NOUT, UK, UN, NBH, MT;      // NOUT = M + D, MT = ceil(L / 16)
    const float* W; int ldw;                              // wcat_att fp32 [4D, M + D]
    const float* gates; const float* cstate;              // forward saves
    const float* dh_static;                               // [T, B, D]   (from the generator input projection)
    const float* dctx_static;                             // [T, B, M]
    const uint8_t* mask_h; const uint8_t* mask_c;
    int kind, training; float rate_h, rate_c;
    float* dgates; __nv_bfloat16* dgb; float* part;       // as in BwdLoopArgs; part [KBA, B, NOUT]
    long long dgb_step;                                   // bf16 gate gradients: 0 = [B, 4D] staging reused every step, B * 4D = [T, B, 4D] history
    int dgb_rows;                                         // rows of one step inside the TMA source (0 for the staging, B for the history)
    // attention
    const float* q; const float* cum; const float* align; long long align_bstride;
    const float* dalign; long long dalign_bstride;        // may be null
    const float* bias; const float* v; const float* Wq;   // [A], [A], [A, D]
    const __nv_bfloat16* WcB;                             // [A][40]   Wcomb[a][k], k contiguous (k >= KC zero)
    const __nv_bfloat16* WcB2;                            // [32][A+8] Wcomb^T[k][a], a contiguous
    const __nv_bfloat16* memTf;                           // [B][MT][32 lanes][64] fragment-major memory projection
    const __nv_bfloat16* memb; int ldm;                   // [B, L, ldm]
    const uint4* memFb; int M16;                          // [B][MT][M16][32] A fragments (rows = positions, k = memory dims), bf16
    const int* lengths;
    int dqp_after_g;                                      // 1: dq partials live after the G tile buffer, 0: alias the scratch head
    float* dctx_tot;                                      // [T, B, M] out
    float* dq;                                            // [T, B, A] out
    float* de;                                            // [T, B, L] out (softmax-backward energies, consumed by the post pass)
    unsigned* barrier; int* abort_flag;
    long long* prof;
};

// Build the Toeplitz pair arrays of the zero-padded cumulative weights: Ph[x] = (hi[x], hi[x+1]), Pl likewise, where
// cumpad[j] = cum[j - half] and cum = hi + lo with hi, lo in bf16 (16 mantissa bits in total).
__device__ __forceinline__ void build_pairs(uint32_t* Ph, uint32_t* Pl, const float* cum, int L, int half, int n, int tid, int nthreads) {
    for (int x = tid; x < n; x += nthreads) {
        float c0 = 0.f, c1 = 0.f;
        const int l0 = x - half, l1 = x + 1 - half;
        if (l0 >= 0 && l0 < L) c0 = __ldcg(cum + l0);
        if (l1 >= 0 && l1 < L) c1 = __ldcg(cum + l1);
        const __nv_bfloat16 h0 = __float2bfloat16_rn(c0), h1 = __float2bfloat16_rn(c1);
        const float r0 = c0 - __bfloat162float(h0), r1 = c1 - __bfloat162float(h1);
        __nv_bfloat162 hp; hp.x = h0; hp.y = h1;
        Ph[x] = *reinterpret_cast<uint32_t*>(&hp);
        Pl[x] = pack2(r0, r1);
    }
}

// UNC: outputs per n-block of the tcgen05 product (UMMA N), compile-time (80, or 96 for memory dim 512); 0 for the mma.sync variant
template <bool TC, int UNC>
__global__ void __launch_bounds__(PT, 1) att_bwd_loop_kernel(const __grid_constant__ CUtensorMap tmG, const AttBwdArgs p) {
    extern __shared__ __align__(1024) unsigned char smem_raw0[];
    unsigned char* smem_raw = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw0) + 1023) & ~(uintptr_t)1023);
    __shared__ uint64_t full_bar, accum_bar, xb1, xb2;      // xb1 / xb2: arrival of the peer's softmax dot / query-gradient partial + G halo tile
    __shared__ uint32_t tmem_base_s;
    __shared__ int s_ok;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int cta = blockIdx.x;
    const int kb = cta % KBA, nb = TC ? cta / KBA : (cta / KBA) % NBA, bh = TC ? 0 : cta / (KBA * NBA);
    const int B = p.B, D = p.D, UK = p.UK, UN = p.UN, KROWS = 4 * UK, M = p.M, L = p.L, A = p.A;
    const int WLD = UN + 8, ALD = KROWS + 8;
    const int b0 = bh * BT, n0 = nb * UN;
    const int NKT = KROWS / 64;                                                      // TC: k-block tiles of the K-slice
    // mma.sync: Ws [KROWS][WLD] bf16, As [BT][ALD] bf16.  tcgen05: sW [NKT][UN rows][128 B] swizzled, slot [NKT][64 rows][128 B] (one TMA box).
    // The activation stage `As` doubles as the attention scratch / query-gradient staging in both variants.
    __nv_bfloat16* Ws = reinterpret_cast<__nv_bfloat16*>(smem_raw);
    unsigned char* sW = smem_raw;
    __nv_bfloat16* As = TC ? reinterpret_cast<__nv_bfloat16*>(smem_raw + (size_t)NKT * UN * 128) : Ws + (size_t)KROWS * WLD;
    unsigned char* extra = TC ? reinterpret_cast<unsigned char*>(As) + (size_t)NKT * 8192 : reinterpret_cast<unsigned char*>(As + (size_t)BT * ALD);
    __nv_bfloat16* sWcB = reinterpret_cast<__nv_bfloat16*>(extra);                   // [A][40]
    __nv_bfloat16* sWcB2 = sWcB + (size_t)A * 40;                                    // [32][A+8]
    float* dcum = reinterpret_cast<float*>(sWcB2 + (size_t)32 * (A + 8));            // [L16 + 32] persistent d cum
    float* wq8 = dcum + (p.MT * 16 + 32);                                            // [A][8 + 1] query weights of this CTA's 8 units
    const unsigned nblocks = gridDim.x;
    const int L16 = p.MT * 16;

    for (int idx = tid; idx < KROWS * UN; idx += PT) {
        const int r = idx / UN, n = idx % UN;
        const int g = r / UK, uk = r % UK;
        float w = 0.f;
        if (n0 + n < p.NOUT) w = p.W[(size_t)(g * D + kb * UK + uk) * p.ldw + n0 + n];
        if (TC) {       // W^T[n][k] of k-block tile c = r / 64 (same order as the TMA box: gate-major, then 64-row halves), SWIZZLE_128B
            const int c = r >> 6, kc = r & 63;
            *reinterpret_cast<__nv_bfloat16*>(sW + (size_t)c * UN * 128 + n * 128 + ((((kc >> 3) ^ (n & 7))) << 4) + (kc & 7) * 2) = __float2bfloat16_rn(w);
        } else {
            Ws[r * WLD + n] = __float2bfloat16_rn(w);
        }
    }
    for (int idx = tid; idx < A * 40; idx += PT) sWcB[idx] = p.WcB[idx];
    for (int idx = tid; idx < 32 * (A + 8); idx += PT) sWcB2[idx] = p.WcB2[idx];
    for (int idx = tid; idx < L16 + 32; idx += PT) dcum[idx] = 0.f;
    // cell-backward ownership: CTA c < D/8 owns hidden units [8c, 8c+8) for every utterance
    const int UOWN = 8;
    const bool owner = cta * UOWN < D;
    const int uo0 = cta * UOWN;
    if (owner)
        for (int idx = tid; idx < A * UOWN; idx += PT) wq8[(idx / UOWN) * (UOWN + 1) + idx % UOWN] = p.Wq[(size_t)(idx / UOWN) * D + uo0 + idx % UOWN];
    uint32_t tmem_base = 0, prod_it = 0;
    if (tid == 0) { tcx::mbar_init(&xb1, 1); tcx::mbar_init(&xb2, 1); tcx::mbar_init_fence(); }
    if (TC) {
        if (tid == 0) { tcx::mbar_init(&full_bar, 1); tcx::mbar_init(&accum_bar, 1); tcx::mbar_init_fence(); }
        if (warp == 1) tcx::tmem_alloc<TMEM_COLS_ATT>(&tmem_base_s);
        tcx::proxy_fence_shared();           // the weight tiles were written through the generic proxy; tcgen05.mma reads them through the async proxy
        tcx::tc_fence_before();
    }
    __syncthreads();
    cluster_arrive(); cluster_wait();      // one-time: the peer's exchange mbarriers are initialised before the first remote st.async targets them
    if (TC) { tcx::tc_fence_after(); tmem_base = tmem_base_s; }
    const uint32_t idesc = tcx::make_idesc_bf16(64, UNC);

    const float inv_h = 1.f / (1.f - p.rate_h), inv_c = 1.f / (1.f - p.rate_c);
    constexpr int MAXE = 3;               // (b, u) pairs per thread: B * 8 / 256 <= 3 for B <= 64... (B <= 96)
    float dc_reg[MAXE], dhz_reg[MAXE];
#pragma unroll
    for (int e = 0; e < MAXE; ++e) { dc_reg[e] = 0.f; dhz_reg[e] = 0.f; }
    unsigned target = 0;

    // attention scratch (aliases As): floats
    float* scr = reinterpret_cast<float*>(As);
    float* s_dctx = scr;                                  // [M (+3)]
    float* s_w = s_dctx + ((M + 3) & ~3);                 // [L16]
    float* s_de = s_w + L16;                              // [L16]
    float* s_qb = s_de + L16;                             // [A]
    float* s_vv = s_qb + A;                               // [A]
    uint32_t* s_Ph = reinterpret_cast<uint32_t*>(s_vv + A);   // [L16 + 48]
    uint32_t* s_Pl = s_Ph + (L16 + 48);
    float* s_red = reinterpret_cast<float*>(s_Pl + (L16 + 48));   // [64]
    // attention backward runs on CTA PAIRS (cluster of 2): rank hf = cta & 1 owns the position tiles [t_lo, t_hi) of utterance cta >> 1
    const int hf = cta & 1, HT0 = (p.MT + 1) / 2;
    const int t_lo = hf ? HT0 : 0, t_hi = hf ? p.MT : HT0;
    const int g_lo = hf ? (HT0 - 1) * 16 : 0;             // first G row held locally: the own tiles plus ONE halo tile of the peer
    float* s_G = s_red + 64;                              // [(HT0 + 1) * 16][GLD], row l stored at l - g_lo
    float* s_dqp = s_G + (size_t)(HT0 + 1) * 16 * GLD;    // [8][A] per-warp query-gradient partials
    float* s_dqx = s_dqp + 8 * A;                         // [A]  the peer's partial (written through distributed shared memory)
    float* s_dotx = s_dqx + A;                            // [4]  the peer's partial softmax dot
    float* s_stage = s_dotx + 4;                          // [L16] d cum staging
    uint2* s_bf = reinterpret_cast<uint2*>(s_stage + L16); // [M16][32] B fragments (hi / lo split of d ctx) of the dw product, shared by all warps
    PROF_DECL

    const int pc = cta >> 1;
    // cell-backward operands of this thread's (b, u) pairs (owner CTAs): fetched a whole reverse step ahead, at the end of the previous
    // cell phase, so that their DRAM latency never sits on the critical path
    float gi_[MAXE], gf_[MAXE], gg_[MAXE], go_[MAXE], cp_[MAXE], dhs_[MAXE];
    uint8_t mh_[MAXE], mc_[MAXE];
    auto pb_prefetch = [&](int step) {
#pragma unroll
        for (int e = 0; e < MAXE; ++e) {
            const int idx = tid + e * PT;
            gi_[e] = gf_[e] = gg_[e] = go_[e] = cp_[e] = dhs_[e] = 0.f; mh_[e] = 1; mc_[e] = 1;
            if (owner && idx < B * UOWN && step >= 0) {
                const int b = idx / UOWN, u = uo0 + idx % UOWN;
                const size_t bu = (size_t)b * D + u, g0 = ((size_t)step * B + b) * 4 * D + u, mi = (size_t)step * B * D + bu;
                gi_[e] = p.gates[g0]; gf_[e] = p.gates[g0 + D]; gg_[e] = p.gates[g0 + 2 * D]; go_[e] = p.gates[g0 + 3 * D];
                cp_[e] = p.cstate[mi];
                dhs_[e] = p.dh_static[mi];
                if (p.training && p.mask_h) mh_[e] = p.mask_h[mi];
                if (p.training && p.mask_c) mc_[e] = p.mask_c[mi];
            }
        }
    };
    pb_prefetch(p.T - 1);
    int pa_len = 0;
    if (pc < B) { const int l0 = p.lengths[pc]; pa_len = l0 < 0 ? 0 : (l0 > L ? L : l0); }
    for (int i = p.T - 1; i >= 0; --i) {
        const bool last = (i == p.T - 1);
        // =========================== PA: attention backward of utterance `pc` on the CTA pair (2 pc, 2 pc + 1) ===========================
        if (pc < B) {
            const int b = pc, half = (p.KC - 1) / 2;
            if (i > 0) {       // DRAM -> L2 one step ahead: the rows of step i-1 this phase starts with (alignment, query, cumulative weights, d ctx)
                const size_t r1 = (size_t)(i - 1) * B + b;
                const char* rows[5] = {reinterpret_cast<const char*>(p.align + (size_t)b * p.align_bstride + (size_t)(i - 1) * L),
                                       reinterpret_cast<const char*>(p.q + r1 * A), reinterpret_cast<const char*>(p.cum + r1 * L),
                                       reinterpret_cast<const char*>(p.dctx_static + r1 * M),
                                       p.dalign ? reinterpret_cast<const char*>(p.dalign + (size_t)b * p.dalign_bstride + (size_t)(i - 1) * L) : nullptr};
                const int bytes[5] = {L * 4, A * 4, L * 4, M * 4, L * 4};
                const int which = tid >> 4, line = tid & 15;           // up to 16 lines of 128 B per row
                if (which < 5 && rows[which] && line * 128 < bytes[which] + 127) l2_prefetch(rows[which] + line * 128);
            }
            const int len = pa_len;                        // loaded once, before the loop
            const int mtiles = (len + 15) / 16;
            constexpr int KT = 6;                          // k-tiles (16 memory dims) per register batch of the dw product
            {   // Staging of the step's operands.  EVERY global load of the phase is issued before the first dependent instruction: ONE L2
                // round trip instead of five serial ones (partial d ctx sums, alignment row, query, cumulative weights, d alignment);
                // two register slots per thread cover M <= 2 PT and L16 + 48 <= 2 PT (checked on the host)
                const size_t row = (size_t)i * B + b;
                const float* cum = p.cum + row * L;
                float r_g[2], r_p[2][KBA], r_w[2], r_da[2], r_c0[2], r_c1[2], r_q = 0.f, bias_r = 0.f, v_r = 0.f;
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int m = tid + e * PT;            // memory dim / text position / Toeplitz index of this slot
                    r_g[e] = 0.f; r_w[e] = 0.f; r_da[e] = 0.f; r_c0[e] = 0.f; r_c1[e] = 0.f;
#pragma unroll
                    for (int k2 = 0; k2 < KBA; ++k2) r_p[e][k2] = 0.f;
                    if (m < M) {
                        r_g[e] = p.dctx_static[row * M + m];
                        if (!last) {
#pragma unroll
                            for (int k2 = 0; k2 < KBA; ++k2) r_p[e][k2] = __ldcg(p.part + ((size_t)k2 * B + b) * p.NOUT + m);
                        }
                    }
                    if (m < L) {
                        r_w[e] = p.align[(size_t)b * p.align_bstride + (size_t)i * L + m];
                        if (p.dalign && m < len) r_da[e] = p.dalign[(size_t)b * p.dalign_bstride + (size_t)i * L + m];
                    }
                    if (m < L16 + 48) {
                        const int l0 = m - half, l1 = l0 + 1;
                        if (l0 >= 0 && l0 < L) r_c0[e] = __ldcg(cum + l0);
                        if (l1 >= 0 && l1 < L) r_c1[e] = __ldcg(cum + l1);
                    }
                }
                if (tid < A) { r_q = p.q[row * A + tid]; bias_r = p.bias[tid]; v_r = p.v[tid]; }
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int m = tid + e * PT;
                    if (m < M) {
                        float g = r_g[e];
#pragma unroll
                        for (int k2 = 0; k2 < KBA; ++k2) g += r_p[e][k2];
                        s_dctx[m] = g;
                        if (hf == 0) p.dctx_tot[row * M + m] = g;
                    }
                    if (m < L16) { s_w[m] = r_w[e]; s_de[m] = r_da[e]; }      // s_de starts as d alignment (or 0); the dw epilogue adds to it
                    if (m < L16 + 48) {
                        const __nv_bfloat16 h0 = __float2bfloat16_rn(r_c0[e]), h1 = __float2bfloat16_rn(r_c1[e]);
                        __nv_bfloat162 hp; hp.x = h0; hp.y = h1;
                        s_Ph[m] = *reinterpret_cast<uint32_t*>(&hp);
                        s_Pl[m] = pack2(r_c0[e] - __bfloat162float(h0), r_c1[e] - __bfloat162float(h1));
                    }
                }
                if (tid < A) { s_qb[tid] = r_q + bias_r; s_vv[tid] = v_r; }
            }
            __syncthreads();
            // B fragments of the dw product: lanes g = 0 hold hi(dctx), g = 1 hold lo(dctx), other columns zero.  They depend on the k-tile only,
            // so the CTA builds the M16 fragments ONCE (every warp used to rebuild all of them: ~40 instructions per fragment and warp)
            for (int idx = tid; idx < p.M16 * 32; idx += PT) {
                const int kt = idx >> 5, gg = (idx >> 2) & 7, tt = idx & 3;
                const int m0 = kt * 16 + 2 * tt;
                uint2 f = make_uint2(0u, 0u);
                if (gg < 2) {
                    const float w0 = m0 < M ? s_dctx[m0] : 0.f, w1 = m0 + 1 < M ? s_dctx[m0 + 1] : 0.f;
                    const float w2 = m0 + 8 < M ? s_dctx[m0 + 8] : 0.f, w3 = m0 + 9 < M ? s_dctx[m0 + 9] : 0.f;
                    const float h0 = __bfloat162float(__float2bfloat16_rn(w0)), h1 = __bfloat162float(__float2bfloat16_rn(w1));
                    const float h2 = __bfloat162float(__float2bfloat16_rn(w2)), h3 = __bfloat162float(__float2bfloat16_rn(w3));
                    f = gg == 0 ? make_uint2(pack2(h0, h1), pack2(h2, h3)) : make_uint2(pack2(w0 - h0, w1 - h1), pack2(w2 - h2, w3 - h3));
                }
                s_bf[idx] = f;
            }
            __syncthreads();
            // dw[l] = dalign + dcum + <dctx, memory[l]> on the tensor cores: A = fragment-major memory (one 16-byte load per lane per
            // MMA), B = (hi(dctx), lo(dctx)) in columns 0 / 1; warp owns position tiles {warp, warp + 8}
            {
                const int g = lane >> 2, tq = lane & 3;
                for (int lt = t_lo + warp; lt < t_hi; lt += 8) {
                    float dacc[4] = {0.f, 0.f, 0.f, 0.f}, dacc2[4] = {0.f, 0.f, 0.f, 0.f};
                    if (lt * 16 < len) {
                        const uint4* fr = p.memFb + (((size_t)b * p.MT + lt) * p.M16) * 32 + lane;
                        for (int kt0 = 0; kt0 < p.M16; kt0 += KT) {
                            uint4 av[KT];
#pragma unroll
                            for (int j = 0; j < KT; ++j)
                                if (kt0 + j < p.M16) av[j] = __ldg(fr + (size_t)(kt0 + j) * 32);
                            uint32_t bfr[KT][2];
#pragma unroll
                            for (int j = 0; j < KT; ++j) {
                                bfr[j][0] = 0u; bfr[j][1] = 0u;
                                if (kt0 + j < p.M16) { const uint2 f = s_bf[(kt0 + j) * 32 + lane]; bfr[j][0] = f.x; bfr[j][1] = f.y; }
                            }
#pragma unroll
                            for (int j = 0; j < KT; j += 2) {        // two independent accumulation chains
                                if (kt0 + j < p.M16) {
                                    const uint32_t af[4] = {av[j].x, av[j].y, av[j].z, av[j].w};
                                    mma_bf16(dacc, af, bfr[j][0], bfr[j][1]);
                                }
                                if (kt0 + j + 1 < p.M16) {
                                    const uint32_t af[4] = {av[j + 1].x, av[j + 1].y, av[j + 1].z, av[j + 1].w};
                                    mma_bf16(dacc2, af, bfr[j + 1][0], bfr[j + 1][1]);
                                }
                            }
                        }
                    }
#pragma unroll
                    for (int q4 = 0; q4 < 4; ++q4) dacc[q4] += dacc2[q4];
                    if (tq == 0) {
#pragma unroll
                        for (int rr = 0; rr < 2; ++rr) {
                            const int l = lt * 16 + g + 8 * rr;
                            float gv = 0.f;
                            if (l < len) gv = (rr ? dacc[2] + dacc[3] : dacc[0] + dacc[1]) + (last ? 0.f : dcum[l]) + s_de[l];   // s_de[l]: d alignment
                            s_de[l] = gv;
                        }
                    }
                }
            }
            __syncthreads();
            // softmax backward: dot = sum_l w[l] dw[l] over ALL positions = own partial + the peer's (exchanged through DSMEM)
            float pdot = 0.f;
            for (int l = t_lo * 16 + tid; l < t_hi * 16 && l < len; l += PT) pdot = fmaf(s_w[l], s_de[l], pdot);
            pdot = block_sum(pdot, s_red);
            if (tid == 0) { tcx::mbar_expect_tx(&xb1, 4); st_async_peer_f32(s_dotx, &xb1, (uint32_t)(hf ^ 1), pdot); }
            tcx::mbar_wait(&xb1, (uint32_t)(p.T - 1 - i) & 1);
            const float dot = pdot + s_dotx[0];           // a + b == b + a: both ranks get the same value
            for (int l = t_lo * 16 + tid; l < t_hi * 16; l += PT) {
                const float d = l < len ? s_w[l] * (s_de[l] - dot) : 0.f;
                s_de[l] = d;
                if (l < L) p.de[((size_t)i * B + b) * L + l] = d;
            }
            __syncthreads();
            PROF_MARK(0);
            // energies backward on the tensor cores; warp owns position tiles {warp, warp + 8}
            float dqacc[16][2];
#pragma unroll
            for (int nt = 0; nt < 16; ++nt) { dqacc[nt][0] = 0.f; dqacc[nt][1] = 0.f; }
            const int g = lane >> 2, tq = lane & 3;
            for (int mt = t_lo + warp; mt < t_hi && mt < mtiles; mt += 8) {
                const int l0 = mt * 16;
                float sacc[16][4];
#pragma unroll
                for (int nt = 0; nt < 16; ++nt)
#pragma unroll
                    for (int e = 0; e < 4; ++e) sacc[nt][e] = 0.f;
#pragma unroll
                for (int ks = 0; ks < 2; ++ks) {
                    const int x = l0 + ks * 16 + g + 2 * tq;       // cumpad index of (row g, col 2t) of this k-step
                    uint32_t ah[4], al[4];
                    ah[0] = s_Ph[x]; ah[1] = s_Ph[x + 8]; ah[2] = s_Ph[x + 8]; ah[3] = s_Ph[x + 16];
                    al[0] = s_Pl[x]; al[1] = s_Pl[x + 8]; al[2] = s_Pl[x + 8]; al[3] = s_Pl[x + 16];
#pragma unroll
                    for (int np = 0; np < 8; ++np) {
                        uint32_t bf[4];
                        ldmatrix_x4(bf[0], bf[1], bf[2], bf[3], sWcB + (size_t)(np * 16 + (lane & 7) + ((lane >> 4) << 3)) * 40 + ks * 16 + ((lane >> 3) & 1) * 8);
                        mma_bf16(sacc[2 * np], ah, bf[0], bf[1]);
                        mma_bf16(sacc[2 * np], al, bf[0], bf[1]);
                        mma_bf16(sacc[2 * np + 1], ah, bf[2], bf[3]);
                        mma_bf16(sacc[2 * np + 1], al, bf[2], bf[3]);
                    }
                }
                // ds = de[l] * v[a] * (1 - tanh^2(S + q + bias + memT)); fragment-major memory projection: 64 bf16 per lane
                const uint4* mf = reinterpret_cast<const uint4*>(p.memTf + (((size_t)b * p.MT + mt) * 32 + lane) * 64);
                const float de0 = s_de[l0 + g], de1 = s_de[l0 + g + 8];
                uint32_t dsA[16][2];
#pragma unroll
                for (int c4 = 0; c4 < 8; ++c4) {
                    const uint4 raw = mf[c4];                      // n-tiles 2*c4, 2*c4+1; 4 values each
                    const uint32_t words[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
                    for (int hf = 0; hf < 2; ++hf) {
                        const int nt = 2 * c4 + hf;
                        const float2 m01 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&words[2 * hf]));
                        const float2 m23 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&words[2 * hf + 1]));
                        const int a0 = nt * 8 + 2 * tq;
                        const float t0 = tanh_fast(sacc[nt][0] + s_qb[a0] + m01.x), t1 = tanh_fast(sacc[nt][1] + s_qb[a0 + 1] + m01.y);
                        const float t2 = tanh_fast(sacc[nt][2] + s_qb[a0] + m23.x), t3 = tanh_fast(sacc[nt][3] + s_qb[a0 + 1] + m23.y);
                        const float d0 = de0 * s_vv[a0] * (1.f - t0 * t0), d1 = de0 * s_vv[a0 + 1] * (1.f - t1 * t1);
                        const float d2 = de1 * s_vv[a0] * (1.f - t2 * t2), d3 = de1 * s_vv[a0 + 1] * (1.f - t3 * t3);
                        dqacc[nt][0] += d0 + d2; dqacc[nt][1] += d1 + d3;
                        dsA[nt][0] = pack2(d0, d1); dsA[nt][1] = pack2(d2, d3);
                    }
                }
                // G[l, tap] = sum_a ds[l, a] * Wcomb[a, tap]   (C fragments of ds reused as A fragments)
                float gacc[4][4];
#pragma unroll
                for (int nt = 0; nt < 4; ++nt)
#pragma unroll
                    for (int e = 0; e < 4; ++e) gacc[nt][e] = 0.f;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const uint32_t af[4] = {dsA[2 * j][0], dsA[2 * j][1], dsA[2 * j + 1][0], dsA[2 * j + 1][1]};
#pragma unroll
                    for (int np = 0; np < 2; ++np) {
                        uint32_t bf[4];
                        ldmatrix_x4(bf[0], bf[1], bf[2], bf[3], sWcB2 + (size_t)(np * 16 + (lane & 7) + ((lane >> 4) << 3)) * (A + 8) + j * 16 + ((lane >> 3) & 1) * 8);
                        mma_bf16(gacc[2 * np], af, bf[0], bf[1]);
                        mma_bf16(gacc[2 * np + 1], af, bf[2], bf[3]);
                    }
                }
#pragma unroll
                for (int nt = 0; nt < 4; ++nt)
#pragma unroll
                    for (int e = 0; e < 4; ++e) s_G[(l0 - g_lo + g + 8 * (e >> 1)) * GLD + nt * 8 + 2 * tq + (e & 1)] = gacc[nt][e];
            }
            // dq[a] = sum_l ds[l, a]: reduce over the 8 row lanes, then over warps
            __syncthreads();                               // every warp is done with s_de / s_qb / s_vv / Ph / Pl
#pragma unroll
            for (int nt = 0; nt < 16; ++nt)
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    float v = dqacc[nt][c];
                    v += __shfl_xor_sync(0xffffffffu, v, 4);
                    v += __shfl_xor_sync(0xffffffffu, v, 8);
                    v += __shfl_xor_sync(0xffffffffu, v, 16);
                    if (g == 0) s_dqp[warp * A + nt * 8 + 2 * tq + c] = v;
                }
            __syncthreads();
            float pdq = 0.f;                                // this rank's partial of dq[a] (a = tid < A)
            if (tid < A) {
#pragma unroll
                for (int w8 = 0; w8 < 8; ++w8) pdq += s_dqp[w8 * A + tid];
                st_async_peer_f32(s_dqx + tid, &xb2, (uint32_t)(hf ^ 1), pdq);
            }
            {   // the boundary tile of G goes to the peer's halo rows (rank 0 sends its last tile, rank 1 its first)
                const int ht = hf ? HT0 : HT0 - 1;             // tile sent
                const int peer_g_lo = hf ? 0 : (HT0 - 1) * 16;
                if (ht >= t_lo && ht < t_hi)
                    for (int idx = tid; idx < 16 * GLD; idx += PT) {
                        const int l = ht * 16 + idx / GLD, k = idx % GLD;
                        st_async_peer_f32(s_G + (size_t)(l - peer_g_lo) * GLD + k, &xb2, (uint32_t)(hf ^ 1), s_G[(size_t)(l - g_lo) * GLD + k]);
                    }
                // what the PEER sends here: its A query-gradient partials, and its boundary tile if it has one (rank 0 always does; rank 1 only
                // when it owns tiles at all)
                const bool peer_sends_tile = hf ? true : (HT0 < p.MT);
                if (tid == 0) tcx::mbar_expect_tx(&xb2, (uint32_t)(A * 4 + (peer_sends_tile ? 16 * GLD * 4 : 0)));
            }
            tcx::mbar_wait(&xb2, (uint32_t)(p.T - 1 - i) & 1);
            if (hf == 0 && tid < A) p.dq[((size_t)i * B + b) * A + tid] = pdq + s_dqx[tid];
            // d cum_{i-1}[j] = d cum_i[j] + sum_k G[j + half - k, k] for the own positions (their G rows: own tiles + the halo tile)
            for (int j = t_lo * 16 + tid; j < t_hi * 16 && j < L; j += PT) {
                float acc = last ? 0.f : dcum[j];
#pragma unroll 4
                for (int k = 0; k < p.KC; ++k) {
                    const int l = j + half - k;
                    if (l >= 0 && l < mtiles * 16) acc += s_G[(size_t)(l - g_lo) * GLD + k];
                }
                s_stage[j] = acc;                           // staged: dcum is still being read by other threads
            }
            __syncthreads();
            for (int j = t_lo * 16 + tid; j < t_hi * 16 && j < L; j += PT) dcum[j] = s_stage[j];
        }
        PROF_MARK(1);
        if (!grid_barrier<false>(p.barrier, target, nblocks, p.abort_flag, &s_ok)) break;
        PROF_MARK(2);

        // =========================== PB: attention-LSTM cell backward ===========================
        if (owner) {
            // recurrent partial sums of this thread's (b, u) pairs (written by the product of the previous reverse step)
            // ... requested together with the query gradients of ALL utterances (staged below): one L2 round trip for both.  (The loop
            // this replaces issued load -> dependent shared-memory store per iteration: eight serial round trips per step.)
            float rec_[MAXE];
            float r8[MAXE][KBA];
#pragma unroll
            for (int e = 0; e < MAXE; ++e) {
                const int idx = tid + e * PT;
#pragma unroll
                for (int k2 = 0; k2 < KBA; ++k2) r8[e][k2] = 0.f;
                if (idx < B * UOWN && !last) {
                    const int b = idx / UOWN, u = uo0 + idx % UOWN;
#pragma unroll
                    for (int k2 = 0; k2 < KBA; ++k2) r8[e][k2] = __ldcg(p.part + ((size_t)k2 * B + b) * p.NOUT + M + u);
                }
            }
            // d h (query part) = dq[b, :] . Wq[:, u] on the tensor cores: A = dq rows staged in shared memory (bf16 hi + lo),
            // B = this CTA's 8 columns of Wq (bf16 hi + lo, register resident); hi.hi + lo.hi + hi.lo = fp32-equivalent
            // (As is idle between PA and P2: [B][A] query gradients, row b rotated by 8 (b & 7) floats against bank conflicts, then [64][8] products)
            float* s_dq = reinterpret_cast<float*>(As);
            float* s_dhq = s_dq + (size_t)B * A;
            {
                constexpr int NQ = 8;                     // float4 per thread: B * A / 4 <= NQ * PT  (A = 128, B <= 64: checked on the host)
                const float4* dq4 = reinterpret_cast<const float4*>(p.dq + (size_t)i * B * A);      // [B][A] block of this step, contiguous
                float4 qv[NQ];
#pragma unroll
                for (int j = 0; j < NQ; ++j) {
                    const int idx = tid + j * PT;
                    if (idx < B * 32) qv[j] = __ldcg(dq4 + idx);         // A == 128 (host check): 32 float4 per utterance
                }
#pragma unroll
                for (int e = 0; e < MAXE; ++e) {
                    float rs = 0.f;
#pragma unroll
                    for (int k2 = 0; k2 < KBA; ++k2) rs += r8[e][k2];
                    rec_[e] = rs;
                }
#pragma unroll
                for (int j = 0; j < NQ; ++j) {
                    const int idx = tid + j * PT;
                    if (idx < B * 32) {
                        const int b = idx >> 5, c4 = idx & 31;
                        *reinterpret_cast<float4*>(s_dq + b * A + ((c4 * 4 + 8 * (b & 7)) & (A - 1))) = qv[j];
                    }
                }
                __syncthreads();
                const int g = lane >> 2, tq = lane & 3, mt = warp & 3, kh = warp >> 2;      // warp = (16-utterance tile, half of the A range)
                float acc[4] = {0.f, 0.f, 0.f, 0.f};
                const int ksteps = A / 32;                                // k-steps of 16 per half
#pragma unroll 4
                for (int ks = 0; ks < ksteps; ++ks) {
                    const int a0 = (kh * ksteps + ks) * 16;
                    uint32_t ah[4], al[4];
#pragma unroll
                    for (int r4 = 0; r4 < 4; ++r4) {
                        const int br = mt * 16 + g + 8 * (r4 & 1);       // rows >= B read stale shared memory: their products are never used
                        const float2 x = *reinterpret_cast<const float2*>(s_dq + br * A + ((a0 + 2 * tq + 8 * (r4 >> 1) + 8 * (br & 7)) & (A - 1)));
                        const __nv_bfloat16 h0 = __float2bfloat16_rn(x.x), h1 = __float2bfloat16_rn(x.y);
                        __nv_bfloat162 hp; hp.x = h0; hp.y = h1;
                        ah[r4] = *reinterpret_cast<uint32_t*>(&hp);
                        al[r4] = pack2(x.x - __bfloat162float(h0), x.y - __bfloat162float(h1));
                    }
                    uint32_t bh[2], bl[2];
#pragma unroll
                    for (int r2 = 0; r2 < 2; ++r2) {
                        const int a = a0 + 2 * tq + 8 * r2;
                        const float x0 = wq8[a * (UOWN + 1) + g], x1 = wq8[(a + 1) * (UOWN + 1) + g];
                        const __nv_bfloat16 h0 = __float2bfloat16_rn(x0), h1 = __float2bfloat16_rn(x1);
                        __nv_bfloat162 hp; hp.x = h0; hp.y = h1;
                        bh[r2] = *reinterpret_cast<uint32_t*>(&hp);
                        bl[r2] = pack2(x0 - __bfloat162float(h0), x1 - __bfloat162float(h1));
                    }
                    mma_bf16(acc, ah, bh[0], bh[1]);
                    mma_bf16(acc, al, bh[0], bh[1]);
                    mma_bf16(acc, ah, bl[0], bl[1]);
                }
                __syncthreads();                                       // every warp is done reading s_dq (s_dhq may overlap its unused tail rows)
                float* d0 = s_dhq + (mt * 16 + g) * UOWN + 2 * tq;
                float* d1 = s_dhq + (mt * 16 + g + 8) * UOWN + 2 * tq;
                if (kh == 0) { d0[0] = acc[0]; d0[1] = acc[1]; d1[0] = acc[2]; d1[1] = acc[3]; }
                __syncthreads();
                if (kh == 1) { d0[0] += acc[0]; d0[1] += acc[1]; d1[0] += acc[2]; d1[1] += acc[3]; }
                __syncthreads();
            }
#pragma unroll
            for (int e = 0; e < MAXE; ++e) {
                const int idx = tid + e * PT;
                if (idx < B * UOWN) {
                    const int b = idx / UOWN, uu = idx % UOWN, u = uo0 + uu;
                    const size_t bu = (size_t)b * D + u, g0 = ((size_t)i * B + b) * 4 * D + u;
                    float dh = dhs_[e] + s_dhq[b * UOWN + uu];
                    float dc_in = 0.f;
                    if (!last) {
                        dh += rec_[e] + dhz_reg[e];
                        dc_in = dc_reg[e];
                    }
                    const float gi = gi_[e], gf = gf_[e], gg = gg_[e], go = go_[e];
                    const float cp = cp_[e];
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
                    if (i > 1 && (uu & 7) == 0) {      // DRAM -> L2 two steps ahead (the register prefetch below runs one step ahead)
                        const size_t g1 = g0 - (size_t)2 * B * 4 * D, m1 = (size_t)(i - 2) * B * D + bu;
                        l2_prefetch(p.gates + g1); l2_prefetch(p.gates + g1 + D); l2_prefetch(p.gates + g1 + 2 * D); l2_prefetch(p.gates + g1 + 3 * D);
                        l2_prefetch(p.cstate + m1); l2_prefetch(p.dh_static + m1);
                        if (p.training && p.mask_h) l2_prefetch(p.mask_h + m1);
                        if (p.training && p.mask_c) l2_prefetch(p.mask_c + m1);
                    }
                }
            }
        }
        PROF_MARK(3);
        // the operands of the next cell backward are fetched between this CTA's arrival and its wait (the compiler parks them in local
        // memory, i.e. the thread waits for the loads right there: under the barrier that wait is free)
        if (!grid_barrier<TC>(p.barrier, target, nblocks, p.abort_flag, &s_ok, [&]() { pb_prefetch(i - 1); })) break;
        PROF_MARK(4);
        if (i == 0) break;

        // =========================== P2: [d ctx | d h](i-1) partial = dgates_i[:, kb] . W[kb, nb] ===========================
        if (TC) {
            // TMA: the bf16 gate gradients of the K-slice, all utterances (rows >= B zero-filled), as NKT swizzled [64 x 64] tiles in ONE box;
            // tcgen05: D[b, n] (TMEM, 64 lanes x 80 columns) = sum over the tiles; warp 0 issues (elected lane), everybody drains TMEM
            if (warp == 0) {
                if (tcx::elect_one()) {
                    tcx::proxy_fence_shared();       // the slot was last touched through the generic proxy (attention scratch, dq staging)
                    tcx::proxy_fence_global();
                    tcx::mbar_expect_tx(&full_bar, (uint32_t)NKT * 8192);
                    tcx::tma_load_5d(As, &tmG, &full_bar, 0, i * p.dgb_rows, 0, kb, 0);
                }
                __syncwarp();
                tcx::mbar_wait(&full_bar, prod_it & 1);
                tcx::tc_fence_after();
                if (tcx::elect_one()) {
                    for (int c = 0; c < NKT; ++c) {
                        const uint64_t adesc = tcx::make_sw128_desc(tcx::smem_u32(reinterpret_cast<unsigned char*>(As) + (size_t)c * 8192));
                        const uint64_t bdesc = tcx::make_sw128_desc(tcx::smem_u32(sW + (size_t)c * UN * 128));
#pragma unroll
                        for (int k = 0; k < 4; ++k) tcx::umma_bf16(tmem_base, adesc + 2 * k, bdesc + 2 * k, idesc, (c == 0 && k == 0) ? 0u : 1u);
                    }
                    tcx::umma_commit(&accum_bar);
                }
                __syncwarp();
            }
            tcx::mbar_wait(&accum_bar, prod_it & 1);
            tcx::tc_fence_after();
            ++prod_it;
            {   // M = 64 accumulator layout: utterance b sits in TMEM lane (b / 16) * 32 + b % 16; warp = (quadrant, half of the UN = 80 / 96 columns)
                constexpr int hc = UNC / 2, NJ = hc / 8;
                const int q = warp & 3, ch = warp >> 2;
                uint32_t r[NJ > 0 ? NJ : 1][8];
#pragma unroll
                for (int j = 0; j < NJ; ++j) tcx::tmem_ld8(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(ch * hc + j * 8), r[j]);
                tcx::tmem_ld_wait();
                const int b = q * 16 + lane;
                if (lane < 16 && b < B) {
                    float* dst = p.part + ((size_t)kb * B + b) * p.NOUT + n0 + ch * hc;
#pragma unroll
                    for (int j = 0; j < NJ; ++j)
#pragma unroll
                        for (int h4 = 0; h4 < 2; ++h4)
                            if (n0 + ch * hc + j * 8 + h4 * 4 < p.NOUT)         // NOUT % 4 == 0 (checked on the host)
                                *reinterpret_cast<float4*>(dst + j * 8 + h4 * 4) =
                                    make_float4(__uint_as_float(r[j][h4 * 4]), __uint_as_float(r[j][h4 * 4 + 1]), __uint_as_float(r[j][h4 * 4 + 2]),
                                                __uint_as_float(r[j][h4 * 4 + 3]));
                }
                tcx::tc_fence_before();
            }
        } else {
            const int segs = UK / 8;
            for (int idx = tid; idx < BT * 4 * segs; idx += PT) {
                const int r = idx / (4 * segs), rem = idx % (4 * segs), g = rem / segs, sg = rem % segs;
                __nv_bfloat16* d = As + r * ALD + g * UK + sg * 8;
                if (b0 + r < B) cp_async16(d, p.dgb + (size_t)i * p.dgb_step + (size_t)(b0 + r) * 4 * D + g * D + kb * UK + sg * 8);
                else *reinterpret_cast<uint4*>(d) = make_uint4(0u, 0u, 0u, 0u);
            }
            cp_async_commit_wait();
            __syncthreads();
            const int npairs = UN / 16;
            for (int np = warp; np < npairs; np += 8) {
                float acc[2][2][4];
#pragma unroll
                for (int mt = 0; mt < 2; ++mt)
#pragma unroll
                    for (int nt = 0; nt < 2; ++nt)
#pragma unroll
                        for (int e = 0; e < 4; ++e) acc[mt][nt][e] = 0.f;
                for (int kk = 0; kk < KROWS; kk += 16) {
                    uint32_t af[2][4], bf[4];
#pragma unroll
                    for (int mt = 0; mt < 2; ++mt)
                        ldmatrix_x4(af[mt][0], af[mt][1], af[mt][2], af[mt][3], As + (mt * 16 + (lane & 15)) * ALD + kk + (lane >> 4) * 8);
                    ldmatrix_x4_trans(bf[0], bf[1], bf[2], bf[3],
                                      Ws + (size_t)(kk + (lane & 7) + ((lane >> 3) & 1) * 8) * WLD + np * 16 + (lane >> 4) * 8);
#pragma unroll
                    for (int mt = 0; mt < 2; ++mt) {
                        mma_bf16(acc[mt][0], af[mt], bf[0], bf[1]);
                        mma_bf16(acc[mt][1], af[mt], bf[2], bf[3]);
                    }
                }
                const int g = lane >> 2, tq = lane & 3;
#pragma unroll
                for (int mt = 0; mt < 2; ++mt)
#pragma unroll
                    for (int nt = 0; nt < 2; ++nt)
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const int b = b0 + mt * 16 + g + 8 * (e >> 1);
                            const int n = n0 + np * 16 + nt * 8 + 2 * tq + (e & 1);
                            if (b < B && n < p.NOUT) p.part[((size_t)kb * B + b) * p.NOUT + n] = acc[mt][nt][e];
                        }
            }
        }
        PROF_MARK(5);
        if (!grid_barrier<false>(p.barrier, target, nblocks, p.abort_flag, &s_ok)) break;
        PROF_MARK(6);
    }
    PROF_FLUSH;
    if (TC) {
        tcx::tc_fence_before();
        __syncthreads();
        if (warp == 1) tcx::tmem_dealloc<TMEM_COLS_ATT>(tmem_base);
    }
}

// -------------------------------------------------------------------------------------------------
// Post pass (fully parallel): accumulate what the recurrence does not need -- d memT, d Wcomb, d v.
// CTA = (utterance b, position tile mt); warp w owns the attention dims [16w, 16w+16); loops over all T steps
// recomputing S^T = Wcomb . T^T on the tensor cores from the saved query / cumulative weights / de.
// -------------------------------------------------------------------------------------------------
struct AttPostArgs {
    int B, T, L, A, KC, MT;
    const float* q; const float* cum; const float* de; const float* bias; const float* v;
    const __nv_bfloat16* WcB;          // [A][40]
    const float* memT;                 // [B, L, A] fp32
    const int* lengths;
    float* dmemT;                      // [B, L, A] out (each element written exactly once)
    float* dWcomb_part;                // [B*MT][A][32]
    float* dv_part;                    // [B*MT][A]
};

__global__ void __launch_bounds__(PT, 3) att_post_kernel(const AttPostArgs p) {
    constexpr int NS = 4;                               // decoder steps per block barrier
    __shared__ uint32_t Ph[2][NS][64], Pl[2][NS][64];
    __shared__ float s_de[2][NS][16], s_q[2][NS][128];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = blockIdx.x / p.MT, mt = blockIdx.x % p.MT;
    const int L = p.L, A = p.A, half = (p.KC - 1) / 2, l0 = mt * 16;
    const int g = lane >> 2, tq = lane & 3;
    int len = p.lengths[b];
    len = len < 0 ? 0 : (len > L ? L : len);
    const int a_base = warp * 16;                       // requires A <= 128 (8 warps x 16)
    const bool active = a_base < A && l0 < len;
    // A fragments of Wcomb (rows a, cols k): constant over the whole loop
    uint32_t wa[2][4];
#pragma unroll
    for (int ks = 0; ks < 2; ++ks) {
        const __nv_bfloat16* base = p.WcB + (size_t)(a_base + g) * 40 + ks * 16 + 2 * tq;
        wa[ks][0] = *reinterpret_cast<const uint32_t*>(base);
        wa[ks][1] = *reinterpret_cast<const uint32_t*>(base + 8 * 40);
        wa[ks][2] = *reinterpret_cast<const uint32_t*>(base + 8);
        wa[ks][3] = *reinterpret_cast<const uint32_t*>(base + 8 * 40 + 8);
    }
    // memT values of this thread's S^T fragment: rows a = a_base + g (+8), cols l = l0 + nt*8 + 2t (+1)
    float mT[2][4];
#pragma unroll
    for (int nt = 0; nt < 2; ++nt)
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int a = a_base + g + 8 * (e >> 1), l = l0 + nt * 8 + 2 * tq + (e & 1);
            // rounded through bf16 exactly like the operand the forward / in-loop kernels consumed
            mT[nt][e] = (a < A && l < L) ? __bfloat162float(__float2bfloat16_rn(p.memT[((size_t)b * L + l) * A + a])) : 0.f;
        }
    const float bias0 = a_base + g < A ? p.bias[a_base + g] : 0.f, bias1 = a_base + g + 8 < A ? p.bias[a_base + g + 8] : 0.f;
    const float v0 = a_base + g < A ? p.v[a_base + g] : 0.f, v1 = a_base + g + 8 < A ? p.v[a_base + g + 8] : 0.f;
    float dmacc[2][4], dwacc[4][4], dvacc[2] = {0.f, 0.f};
#pragma unroll
    for (int nt = 0; nt < 2; ++nt)
#pragma unroll
        for (int e = 0; e < 4; ++e) dmacc[nt][e] = 0.f;
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
#pragma unroll
        for (int e = 0; e < 4; ++e) dwacc[nt][e] = 0.f;

    // The T steps are independent here (only the accumulators chain), so they are processed in chunks of NS with ONE block barrier per
    // chunk: the operands of the next chunk (cumulative-weight window, de, query of NS steps) are loaded into registers before the MMAs
    // of the current chunk and stored to the other shared-memory buffer after them, i.e. their DRAM / L2 latency hides behind compute.
    float r0[NS], r1[NS];
    auto load = [&](int i0) {
#pragma unroll
        for (int s2 = 0; s2 < NS; ++s2) {
            const int i = i0 + s2;
            r0[s2] = 0.f; r1[s2] = 0.f;
            if (i >= p.T) continue;
            if (tid < 64) {                    // window of cumpad needed by this tile: x in [l0, l0 + 16 + 32)
                const float* cum = p.cum + ((size_t)i * p.B + b) * L;
                const int la = l0 + tid - half, lb = la + 1;
                if (la >= 0 && la < L) r0[s2] = __ldg(cum + la);
                if (lb >= 0 && lb < L) r1[s2] = __ldg(cum + lb);
            } else if (tid < 80) {
                const int l = l0 + tid - 64;
                if (l < L) r0[s2] = __ldg(p.de + ((size_t)i * p.B + b) * L + l);
            } else if (tid >= 128 && tid < 128 + A) {
                r0[s2] = __ldg(p.q + ((size_t)i * p.B + b) * A + tid - 128);
            }
        }
    };
    auto store = [&](int buf) {
#pragma unroll
        for (int s2 = 0; s2 < NS; ++s2) {
            if (tid < 64) {
                const __nv_bfloat16 h0 = __float2bfloat16_rn(r0[s2]), h1 = __float2bfloat16_rn(r1[s2]);
                __nv_bfloat162 hp; hp.x = h0; hp.y = h1;
                Ph[buf][s2][tid] = *reinterpret_cast<uint32_t*>(&hp);
                Pl[buf][s2][tid] = pack2(r0[s2] - __bfloat162float(h0), r1[s2] - __bfloat162float(h1));
            } else if (tid < 80) {
                s_de[buf][s2][tid - 64] = r0[s2];
            } else if (tid >= 128 && tid < 128 + A) {
                s_q[buf][s2][tid - 128] = r0[s2];
            }
        }
    };
    if (l0 < len) { load(0); store(0); }
    __syncthreads();
    for (int i0 = 0; i0 < p.T && l0 < len; i0 += NS) {
        const int buf = (i0 / NS) & 1;
        const bool more = i0 + NS < p.T;
        if (more) load(i0 + NS);
        if (active) {
#pragma unroll
            for (int s2 = 0; s2 < NS; ++s2) {
                if (i0 + s2 >= p.T) break;
                // S^T[a, l] = sum_k Wcomb[a, k] * cumpad[l + k]
                float sacc[2][4];
#pragma unroll
                for (int nt = 0; nt < 2; ++nt)
#pragma unroll
                    for (int e = 0; e < 4; ++e) sacc[nt][e] = 0.f;
#pragma unroll
                for (int ks = 0; ks < 2; ++ks)
#pragma unroll
                    for (int nt = 0; nt < 2; ++nt) {
                        // B fragment (k rows, l cols): (k = ks*16 + 2t (+1) (+8), l = nt*8 + g) -> cumpad[l + k]
                        const int x = nt * 8 + g + ks * 16 + 2 * tq;
                        mma_bf16(sacc[nt], wa[ks], Ph[buf][s2][x], Ph[buf][s2][x + 8]);
                        mma_bf16(sacc[nt], wa[ks], Pl[buf][s2][x], Pl[buf][s2][x + 8]);
                    }
                const float q0 = s_q[buf][s2][a_base + g] + bias0, q1 = s_q[buf][s2][a_base + g + 8] + bias1;
                uint32_t dsA[2][2];
#pragma unroll
                for (int nt = 0; nt < 2; ++nt) {
                    const float dea = s_de[buf][s2][nt * 8 + 2 * tq], deb = s_de[buf][s2][nt * 8 + 2 * tq + 1];
                    const float t0 = tanh_fast(sacc[nt][0] + q0 + mT[nt][0]), t1 = tanh_fast(sacc[nt][1] + q0 + mT[nt][1]);
                    const float t2 = tanh_fast(sacc[nt][2] + q1 + mT[nt][2]), t3 = tanh_fast(sacc[nt][3] + q1 + mT[nt][3]);
                    const float d0 = dea * v0 * (1.f - t0 * t0), d1 = deb * v0 * (1.f - t1 * t1);
                    const float d2 = dea * v1 * (1.f - t2 * t2), d3 = deb * v1 * (1.f - t3 * t3);
                    dmacc[nt][0] += d0; dmacc[nt][1] += d1; dmacc[nt][2] += d2; dmacc[nt][3] += d3;
                    dvacc[0] += dea * t0 + deb * t1; dvacc[1] += dea * t2 + deb * t3;
                    dsA[nt][0] = pack2(d0, d1); dsA[nt][1] = pack2(d2, d3);
                }
                // d Wcomb[a, k] += sum_l ds^T[a, l] * cumpad[l + k]   (A = ds^T chained; B fragment (l rows, k cols) = cumpad[l + k])
                const uint32_t af[4] = {dsA[0][0], dsA[0][1], dsA[1][0], dsA[1][1]};
#pragma unroll
                for (int nt = 0; nt < 4; ++nt) {
                    const int x = 2 * tq + nt * 8 + g;                  // l = 2t (+1) (+8), k = nt*8 + g
                    mma_bf16(dwacc[nt], af, Ph[buf][s2][x], Ph[buf][s2][x + 8]);
                }
            }
        }
        if (more) store(buf ^ 1);
        __syncthreads();
    }
    if (a_base < A) {
#pragma unroll
        for (int nt = 0; nt < 2; ++nt)
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int a = a_base + g + 8 * (e >> 1), l = l0 + nt * 8 + 2 * tq + (e & 1);
                if (a < A && l < L) p.dmemT[((size_t)b * L + l) * A + a] = dmacc[nt][e];
            }
#pragma unroll
        for (int nt = 0; nt < 4; ++nt)
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int a = a_base + g + 8 * (e >> 1), k = nt * 8 + 2 * tq + (e & 1);
                if (a < A) p.dWcomb_part[((size_t)blockIdx.x * A + a) * 32 + k] = dwacc[nt][e];
            }
        float d0 = dvacc[0], d1 = dvacc[1];
        d0 += __shfl_xor_sync(0xffffffffu, d0, 1); d0 += __shfl_xor_sync(0xffffffffu, d0, 2);
        d1 += __shfl_xor_sync(0xffffffffu, d1, 1); d1 += __shfl_xor_sync(0xffffffffu, d1, 2);
        if (tq == 0) {
            if (a_base + g < A) p.dv_part[(size_t)blockIdx.x * A + a_base + g] = d0;
            if (a_base + g + 8 < A) p.dv_part[(size_t)blockIdx.x * A + a_base + g + 8] = d1;
        }
    }
}

// prep: bf16 copies of Wcomb in the two operand layouts, fragment-major memT
__global__ void att_bwd_prep_kernel(__nv_bfloat16* __restrict__ WcB, __nv_bfloat16* __restrict__ WcB2, __nv_bfloat16* __restrict__ memTf,
                                    const float* __restrict__ WcombT, const float* __restrict__ memT, int B, int L, int A, int KC, int MT) {
    const size_t n1 = (size_t)A * 40, n2 = (size_t)32 * (A + 8), n3 = (size_t)B * MT * 32 * 64;
    for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < n1 + n2 + n3; idx += (size_t)gridDim.x * blockDim.x) {
        if (idx < n1) {
            const int a = idx / 40, k = idx % 40;
            WcB[idx] = __float2bfloat16_rn(k < KC ? WcombT[(size_t)k * A + a] : 0.f);
        } else if (idx < n1 + n2) {
            const size_t j = idx - n1;
            const int k = j / (A + 8), a = j % (A + 8);
            WcB2[j] = __float2bfloat16_rn((k < KC && a < A) ? WcombT[(size_t)k * A + a] : 0.f);
        } else {
            const size_t j = idx - n1 - n2;
            const int v = j % 64, lane = (j / 64) % 32, mt = (j / (64 * 32)) % MT, b = j / ((size_t)64 * 32 * MT);
            const int nt = v / 4, e = v % 4, g = lane >> 2, tq = lane & 3;
            const int l = mt * 16 + g + 8 * (e >> 1), a = nt * 8 + 2 * tq + (e & 1);
            memTf[j] = __float2bfloat16_rn((l < L && a < A) ? memT[((size_t)b * L + l) * A + a] : 0.f);
        }
    }
}

// stage 1: dW[a, k] = sum over the nparts partial blocks (one thread per element, grid over the A * 32 + A outputs; fixed order)
__global__ void att_bwd_reduce_parts_kernel(float* __restrict__ dWsum, float* __restrict__ dvsum, const float* __restrict__ dWcomb_part,
                                            const float* __restrict__ dv_part, int nparts, int A) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx < A * 32) {
        float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
        int p2 = 0;
        for (; p2 + 3 < nparts; p2 += 4) {
            s0 += dWcomb_part[(size_t)p2 * A * 32 + idx]; s1 += dWcomb_part[(size_t)(p2 + 1) * A * 32 + idx];
            s2 += dWcomb_part[(size_t)(p2 + 2) * A * 32 + idx]; s3 += dWcomb_part[(size_t)(p2 + 3) * A * 32 + idx];
        }
        for (; p2 < nparts; ++p2) s0 += dWcomb_part[(size_t)p2 * A * 32 + idx];
        dWsum[idx] = (s0 + s1) + (s2 + s3);
    } else if (idx < A * 32 + A) {
        const int a = idx - A * 32;
        float sv = 0.f;
        for (int p2 = 0; p2 < nparts; ++p2) sv += dv_part[(size_t)p2 * A + a];
        dvsum[a] = sv;
    }
}
// stage 2: dWloc[a, c] += sum_k dWcomb[a, k] * Wc[c, k];  dWc[c, k] += sum_a Wloc[a, c] * dWcomb[a, k];  dv += dvsum
__global__ void att_bwd_finish_kernel(float* __restrict__ dWloc, float* __restrict__ dWc, float* __restrict__ dv,
                                      const float* __restrict__ dWsum, const float* __restrict__ dvsum,
                                      const float* __restrict__ Wloc, const float* __restrict__ Wc, int A, int C, int KC) {
    extern __shared__ float dW[];        // [A][32] reduced dWcomb
    for (int idx = threadIdx.x; idx < A * 32; idx += blockDim.x) dW[idx] = dWsum[idx];
    for (int a = threadIdx.x; a < A; a += blockDim.x) dv[a] += dvsum[a];
    __syncthreads();
    for (int idx = threadIdx.x; idx < A * C; idx += blockDim.x) {
        const int a = idx / C, c = idx % C;
        float s = 0.f;
        for (int k = 0; k < KC; ++k) s = fmaf(dW[a * 32 + k], Wc[c * KC + k], s);
        dWloc[idx] += s;
    }
    for (int idx = threadIdx.x; idx < C * KC; idx += blockDim.x) {
        const int c = idx / KC, k = idx % KC;
        float s = 0.f;
        for (int a = 0; a < A; ++a) s = fmaf(Wloc[a * C + c], dW[a * 32 + k], s);
        dWc[idx] += s;
    }
}

}  // namespace

bool persist_bwd_supported(const b200tts_decoder_shape& s) {
    if (s.D % (KB * 16) != 0 || s.B > 2 * BT) return false;
    const int UK = s.D / KB;
    if (UK / NBK > 32 || (UK % NBK) != 0) return false;
    return true;
}

// -------------------------------------------------------------------------------------------------
// attention loop, host side
// -------------------------------------------------------------------------------------------------
AttBwdExtra att_bwd_extra(const b200tts_decoder_shape& s) {
    AttBwdExtra x;
    size_t off = 0;
    auto take = [&](size_t n) { size_t o = off; off = (off + n + 255) / 256 * 256; return o; };
    x.MT = (s.L + 15) / 16;
    x.dgb = take((size_t)s.B * 4 * s.D * 2);
    x.part = take((size_t)KBA * s.B * (s.M + s.D) * 4);
    x.wcb = take((size_t)s.A * 40 * 2);
    x.wcb2 = take((size_t)32 * (s.A + 8) * 2);
    x.memTf = take((size_t)s.B * x.MT * 32 * 64 * 2);
    x.de = take((size_t)s.T * s.B * s.L * 4);
    x.dwpart = take((size_t)s.B * x.MT * s.A * 32 * 4);
    x.dvpart = take((size_t)s.B * x.MT * s.A * 4);
    x.barrier = take(256 + 148 * 8 * 8);
    x.total = off;
    return x;
}

// Geometry of the two product variants of the attention reverse loop.
struct AttBwdGeom {
    bool tc; int UK, UN, NBH, grid; size_t region, smem;      // region = bytes of the activation stage (= attention scratch capacity)
};
static AttBwdGeom att_bwd_geom(const b200tts_decoder_shape& s, bool tc) {
    AttBwdGeom g{};
    g.tc = tc;
    g.UK = s.D / KBA;
    const int L16 = (s.L + 15) / 16 * 16;
    const size_t extras = (size_t)s.A * 40 * 2 + (size_t)32 * (s.A + 8) * 2 + (size_t)(L16 + 32) * 4 + (size_t)s.A * 9 * 4;
    if (tc) {
        g.UN = (s.M + s.D <= NBT * TUN) ? TUN : TUN_WIDE; g.NBH = 1; g.grid = KBA * NBT;
        const int NKT = 4 * g.UK / 64;
        g.region = (size_t)NKT * 8192;
        g.smem = 1024 + (size_t)NKT * g.UN * 128 + g.region + extras;
    } else {
        g.UN = (cdiv(s.M + s.D, NBA) + 15) / 16 * 16; g.NBH = (s.B + BT - 1) / BT; g.grid = KBA * NBA * g.NBH;
        g.region = (size_t)BT * (4 * g.UK + 8) * 2;
        g.smem = 1024 + (size_t)4 * g.UK * (g.UN + 8) * 2 + g.region + extras;
    }
    return g;
}

static bool att_bwd_variant_ok(const b200tts_decoder_shape& s, const AttBwdGeom& g) {
    if (s.A != 128 || s.K > 32 || s.B * 8 > 3 * PT || s.D % KBA != 0) return false;
    if (s.M > 2 * PT || (s.L + 15) / 16 * 16 + 48 > 2 * PT || s.B * (s.A / 4) > 8 * PT) return false;      // register-slot staging of the attention backward
    if (s.D / 8 > g.grid) return false;                       // cell-backward ownership: 8 hidden units per CTA
    if (g.grid / 2 < s.B || g.grid > 148) return false;       // one CTA pair per utterance, all CTAs co-resident
    if (g.tc) {
        if (g.UK % 64 != 0 || s.B > 64 || s.M + s.D > NBT * g.UN || (s.M + s.D) % 4 != 0) return false;
    } else {
        if (!persist_bwd_supported(s) || s.B > 2 * BT) return false;
    }
    const int MT = (s.L + 15) / 16, L16 = MT * 16, HT0 = (MT + 1) / 2;
    // attention-backward scratch of one CTA of the pair (aliases the activation stage)
    const size_t fl = (size_t)((s.M + 3) & ~3) + 3 * (size_t)L16 + 2 * s.A + 2 * (size_t)(L16 + 48) + 64 + (size_t)(HT0 + 1) * 16 * GLD +
                      8 * (size_t)s.A + s.A + 4 + (size_t)((s.M + 15) / 16) * 32 * 2;
    if (fl * 4 > g.region) return false;
    // the cell-backward phase stages the query gradients [B][A] fp32 + [64][8] products in the (then idle) activation stage
    if ((size_t)s.B * s.A * 4 + 64 * 8 * 4 > g.region) return false;
    return g.smem <= 227 * 1024;
}

static bool att_bwd_pick(const b200tts_decoder_shape& s, AttBwdGeom* out) {
    for (int tc = 1; tc >= 0; --tc) {
        if (tc && getenv("B200TTS_ATT_BWD_MMA_SYNC")) continue;      // A/B switch: force the mma.sync product
        const AttBwdGeom g = att_bwd_geom(s, tc != 0);
        if (att_bwd_variant_ok(s, g)) { if (out) *out = g; return true; }
    }
    return false;
}

bool persist_att_bwd_supported(const b200tts_decoder_shape& s) { return att_bwd_pick(s, nullptr); }
bool persist_att_bwd_tc(const b200tts_decoder_shape& s) { AttBwdGeom g{}; return att_bwd_pick(s, &g) && g.tc; }

int persist_att_bwd_loop(const b200tts_decoder_shape& s, const b200tts_decoder_params& w, const b200tts_decoder_inputs& in,
                         const DecoderLayout& fl, const float* fws, const PersistLayout& pl, const unsigned char* pws,
                         const float* align, const float* dalign, const float* dh_static, const float* dctx_static, float* dgates,
                         float* dq, float* dctx_tot, float* dmemT, unsigned char* extra, const b200tts_decoder_params& dw,
                         cudaStream_t st, void* dgb_hist) {
    const AttBwdExtra x = att_bwd_extra(s);
    const int B = s.B, D = s.D, M = s.M, T = s.T, L = s.L, A = s.A;
    AttBwdArgs a{};
    AttBwdGeom geo{};
    B200_REQUIRE(att_bwd_pick(s, &geo), "persistent attention backward: shape not supported");
    a.B = B; a.T = T; a.D = D; a.M = M; a.L = L; a.A = A; a.KC = s.K; a.NOUT = M + D; a.UK = geo.UK;
    a.UN = geo.UN; a.NBH = geo.NBH; a.MT = x.MT;
    a.W = fws + fl.wcat_att; a.ldw = M + D;
    a.gates = fws + fl.ga; a.cstate = fws + fl.ca; a.dh_static = dh_static; a.dctx_static = dctx_static;
    a.mask_h = in.mask_att_h; a.mask_c = in.mask_att_c; a.kind = s.cell_kind; a.training = s.training; a.rate_h = s.rate_h; a.rate_c = s.rate_c;
    a.dgates = dgates;
    // bf16 gate gradients: a [T, B, 4D] history when the caller wants to feed the time-batched products from it (no conversion pass),
    // else a [B, 4D] staging reused every step
    a.dgb = dgb_hist ? static_cast<__nv_bfloat16*>(dgb_hist) : reinterpret_cast<__nv_bfloat16*>(extra + x.dgb);
    a.dgb_step = dgb_hist ? (long long)B * 4 * D : 0; a.dgb_rows = dgb_hist ? B : 0;
    a.part = reinterpret_cast<float*>(extra + x.part);
    a.q = fws + fl.q; a.cum = fws + fl.cum; a.align = align; a.align_bstride = (long long)T * L;
    a.dalign = dalign; a.dalign_bstride = (long long)T * L;
    a.bias = w.attn_bias; a.v = w.attn_energy; a.Wq = w.attn_query;
    __nv_bfloat16* wcb = reinterpret_cast<__nv_bfloat16*>(extra + x.wcb);
    __nv_bfloat16* wcb2 = reinterpret_cast<__nv_bfloat16*>(extra + x.wcb2);
    __nv_bfloat16* memTf = reinterpret_cast<__nv_bfloat16*>(extra + x.memTf);
    a.WcB = wcb; a.WcB2 = wcb2; a.memTf = memTf;
    a.memb = reinterpret_cast<const __nv_bfloat16*>(pws + pl.memb); a.ldm = pl.ldm;
    a.memFb = reinterpret_cast<const uint4*>(pws + pl.memFb); a.M16 = pl.M16;
    a.dqp_after_g = 1;
    a.lengths = in.text_lengths; a.dctx_tot = dctx_tot; a.dq = dq; a.de = reinterpret_cast<float*>(extra + x.de);
    const float* wcombT = reinterpret_cast<const float*>(pws + pl.wcombT);
    B200_TRY(reset_grid_barrier(extra + x.barrier, a, st));
    att_bwd_prep_kernel<<<148 * 4, 256, 0, st>>>(wcb, wcb2, memTf, wcombT, fws + fl.memT, B, L, A, s.K, x.MT);
    B200_LAUNCH_CHECK();
    void* fn = geo.tc ? (geo.UN == TUN ? (void*)att_bwd_loop_kernel<true, TUN> : (void*)att_bwd_loop_kernel<true, TUN_WIDE>)
                      : (void*)att_bwd_loop_kernel<false, 0>;
    const int grid = geo.grid;
    B200_REQUIRE(grid % 2 == 0 && grid / 2 >= B, "persistent attention backward: %d CTAs cannot be paired", grid);
    CUtensorMap tm;
    memset(&tm, 0, sizeof(tm));
    if (geo.tc) {
        // bf16 gate gradients dgb [B, 4D] as {64 k, B rows, UK/64 halves, KBA k-slices, 4 gates}: element (b, g, kb, h, c) at
        // b * 4D + g * D + kb * UK + h * 64 + c; one box = {64, 64 rows, UK/64, 1, 4} = the whole K-slice of a CTA
        const unsigned long long dims[5] = {64ull, (unsigned long long)(dgb_hist ? (size_t)T * B : (size_t)B), (unsigned long long)(geo.UK / 64), (unsigned long long)KBA, 4ull};
        const unsigned long long strides[4] = {(unsigned long long)4 * D * 2, 128ull, (unsigned long long)geo.UK * 2, (unsigned long long)D * 2};
        const unsigned box[5] = {64u, 64u, (unsigned)(geo.UK / 64), 1u, 4u};
        B200_TRY(tc_make_mapN_bf16(&tm, a.dgb, 5, dims, strides, box));
    }
    void* params[] = {&tm, &a};
    // the attention backward of an utterance runs on a CTA pair
    B200_TRY(launch_persistent(fn, grid, PT, geo.smem, params, st, "persistent attention backward", "att_bwd_loop_kernel", 2, true));
    // parallel post pass
    AttPostArgs pp{};
    pp.B = B; pp.T = T; pp.L = L; pp.A = A; pp.KC = s.K; pp.MT = x.MT;
    pp.q = a.q; pp.cum = a.cum; pp.de = a.de; pp.bias = w.attn_bias; pp.v = w.attn_energy; pp.WcB = wcb; pp.memT = fws + fl.memT;
    pp.lengths = in.text_lengths; pp.dmemT = dmemT;
    pp.dWcomb_part = reinterpret_cast<float*>(extra + x.dwpart); pp.dv_part = reinterpret_cast<float*>(extra + x.dvpart);
    B200_CUDA(cudaMemsetAsync(dmemT, 0, (size_t)B * L * A * 4, st));
    B200_CUDA(cudaMemsetAsync(pp.dWcomb_part, 0, (size_t)B * x.MT * A * 32 * 4, st));
    B200_CUDA(cudaMemsetAsync(pp.dv_part, 0, (size_t)B * x.MT * A * 4, st));
    {
        KernelTimer kt("att_post_kernel", st);
        att_post_kernel<<<B * x.MT, PT, 0, st>>>(pp);
    }
    B200_LAUNCH_CHECK();
    // the de buffer is dead after the post pass: its head holds the reduced partials
    float* dWsum = a.de;
    float* dvsum = dWsum + (size_t)A * 32;
    att_bwd_reduce_parts_kernel<<<cdiv(A * 32 + A, 128), 128, 0, st>>>(dWsum, dvsum, pp.dWcomb_part, pp.dv_part, B * x.MT, A);
    B200_LAUNCH_CHECK();
    att_bwd_finish_kernel<<<1, 512, (size_t)A * 32 * 4, st>>>(dw.attn_location, dw.attn_loc_features, dw.attn_energy, dWsum, dvsum,
                                                             w.attn_location, w.attn_loc_features, A, s.C, s.K);
    B200_LAUNCH_CHECK();
    return B200TTS_OK;
}

size_t persist_bwd_gen_extra_bytes(const b200tts_decoder_shape& s) {
    // dgb [B, 4D] bf16 + part [KB, B, D] fp32 + barrier
    return ((size_t)s.B * 4 * s.D * 2 + 255) / 256 * 256 + ((size_t)KB * s.B * s.D * 4 + 255) / 256 * 256 + 256 + 148 * 8 * 8;
}

// dgates for all T steps of the generator LSTM.  `extra` = persist_bwd_gen_extra_bytes scratch.
int persist_gen_bwd_loop(const b200tts_decoder_shape& s, const b200tts_decoder_params& w, const b200tts_decoder_inputs& in,
                         const DecoderLayout& fl, const float* fws, const float* dh_static, float* dgates, unsigned char* extra,
                         cudaStream_t st) {
    const int B = s.B, D = s.D;
    BwdLoopArgs a{};
    a.B = B; a.T = s.T; a.D = D; a.NOUT = D; a.UK = D / KB; a.UN = (cdiv(D, NBK) + 15) / 16 * 16; a.NBH = (B + BT - 1) / BT;
    a.W = w.gen_w_hh; a.ldw = D;
    a.gates = fws + fl.gg; a.cstate = fws + fl.cg; a.dh_static = dh_static;
    a.mask_h = in.mask_gen_h; a.mask_c = in.mask_gen_c; a.kind = s.cell_kind; a.training = s.training; a.rate_h = s.rate_h; a.rate_c = s.rate_c;
    a.dgates = dgates;
    size_t off = 0;
    a.dgb = reinterpret_cast<__nv_bfloat16*>(extra + off); off += ((size_t)B * 4 * D * 2 + 255) / 256 * 256;
    a.part = reinterpret_cast<float*>(extra + off); off += ((size_t)KB * B * D * 4 + 255) / 256 * 256;
    a.hcol = 0;
    B200_TRY(reset_grid_barrier(extra + off, a, st));
    const size_t smem = ((size_t)4 * a.UK * (a.UN + 8) + (size_t)BT * (4 * a.UK + 8)) * 2;
    B200_REQUIRE(smem <= 227 * 1024, "persistent backward: %zu B of shared memory needed", smem);
    void* params[] = {&a};
    B200_TRY(launch_persistent((void*)lstm_bwd_loop_kernel, KB * NBK * a.NBH, PT, smem, params, st, "persistent backward",
                               "lstm_bwd_loop_kernel"));
    return B200TTS_OK;
}

}  // namespace b200tts
