// Persistent recurrent kernels of the bf16 perf mode (forward): ONE cooperative launch per LSTM loop.
//
//   * weight-stationary: CTA (rb, bh) keeps the bf16 slice [64 gate rows = 16 hidden units x {i,f,g,o}] x K of the
//     recurrent weight matrix in shared memory for the whole sequence (169 KB for K = 1312) and owns a batch
//     half of 32 utterances -> 64 x 2 = 128 CTAs, one per SM;
//   * per step the bf16 activation operand [32 x K] streams L2 -> shared memory with cp.async in 256-column chunks
//     (double buffered); the 8 warps split K inside a chunk and feed mma.sync.m16n8k16 from ldmatrix fragments;
//     a tree reduction over the warps is followed by the LSTM cell / regulariser epilogue in registers;
//   * attention loop only: after a grid barrier the first B CTAs run the location-sensitive attention of one
//     utterance each (query from the per-CTA partial projections, warp-shuffle softmax, context), second barrier;
//   * grid barriers are monotonic counters in global memory (acquire/release, L2-only loads for exchanged data)
//     with a clock64 watchdog so a protocol bug can never hang the GPU.
// fp32 state (c, h, gates, cumulative weights, context, alignments) is written exactly where the per-step (v1)
// path writes it, so the backward pass and the fp32 parity path are unaffected.
// Reference semantics: modules/tacotron2.py:180-198, modules/layers.py:18-47, modules/attention.py:39-86.
#include <cuda_bf16.h>
#include <cooperative_groups.h>
#include "decoder_internal.cuh"
#include "persist.cuh"

namespace b200tts {

namespace {

constexpr int PT = 256;             // threads per CTA
constexpr int UNITS = 16;           // hidden units per CTA
constexpr int ROWS = 4 * UNITS;     // gate rows per CTA
constexpr int BT = 32;              // utterances per CTA
constexpr int CHUNK = 128;          // activation columns per cp.async stage (8 k-steps: one per warp)
constexpr int ALD = CHUNK + 8;      // bf16 row stride of an activation stage
constexpr int ATT_STAGES = 4;       // 4 x 128 columns in flight (shared memory is almost full: 169 KB of weights)
constexpr int GEN_STAGES = 8;       // the whole 1024-column operand in flight

struct LoopArgs {
    int B, T, D, K, Kp, RB, NBH;
    const float* W; int ldw;                  // recurrent weights fp32 [4D, ldw]
    __nv_bfloat16* actb;                      // [T+1, B, Kp] bf16 operand of step i in row i
    float* actf; int ldf; int hcol;           // fp32 mirror ([T+1, B, ldf]); h lives at column hcol
    float* gates;                             // [T, B, 4D] in: input projection (+biases); out: activated gates
    float* cstate;                            // [T+1, B, D]
    const uint8_t* mask_h; const uint8_t* mask_c;   // [T, B, D] or null
    int kind, training; float rate_h, rate_c;
    // attention (ATT instantiation only)
    int L, M, A, KC;
    const float* Wq;                          // [A, D]
    float* qpart;                             // [RB, B, A]
    float* qsave;                             // [T, B, A]
    const __nv_bfloat16* WcB;                 // [A][40] bf16 Wcomb[a][k] (k contiguous, zero beyond KC)
    const __nv_bfloat16* memTf; int MT;       // [B][MT][32][64] fragment-major bf16 memory projection
    const float* bias; const float* v;        // [A]
    const __nv_bfloat16* memb; int ldm;       // [B, L, ldm]
    const uint4* memFf; int M16;              // [B][M16][MT][32] A fragments (m16 x k16 over positions) of memory^T, bf16
    const int* lengths;
    float* cum;                               // [T+1, B, L]
    float* align; long long align_bstride;    // [B, T, L]
    unsigned* barrier; int* abort_flag;
    long long* prof;                          // optional [gridDim.x][8] per-phase cycle totals (thread 0 of each CTA)
};

using namespace tcx;

struct Smem {
    __nv_bfloat16* W;      // [ROWS][Kp + 8]
    __nv_bfloat16* act;    // [2][BT][ALD]   (aliased by the reduction scratch and the attention scratch)
    float* wq;             // [A][UNITS + 1]
    float* hs;             // [BT][UNITS + 1]
    float* sum;            // [BT][ROWS + 1]
};

template <bool ATT, int NSTAGE>
__global__ void __launch_bounds__(PT, 1) lstm_loop_kernel(const LoopArgs p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int s_ok;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int cta = blockIdx.x;
    const int rb = cta % p.RB, bh = cta / p.RB;
    const int u0 = rb * UNITS, b0 = bh * BT;
    const int Kp = p.Kp, WLD = Kp + 8, D = p.D, B = p.B;
    const unsigned nblocks = gridDim.x;

    Smem s;
    size_t off = 0;
    s.W = reinterpret_cast<__nv_bfloat16*>(smem_raw + off); off += (size_t)ROWS * WLD * 2;
    s.act = reinterpret_cast<__nv_bfloat16*>(smem_raw + off); off += (size_t)NSTAGE * BT * ALD * 2;
    s.hs = reinterpret_cast<float*>(smem_raw + off); off += (size_t)UNITS * (BT + 4) * 4;      // [UNITS][BT + 4] (transposed)
    s.wq = reinterpret_cast<float*>(smem_raw + off); off += ATT ? (size_t)p.A * (UNITS + 1) * 4 : 0;
    __nv_bfloat16* sWcB = reinterpret_cast<__nv_bfloat16*>(smem_raw + off);     // [A][40] resident (ATT only)
    float* scratch = reinterpret_cast<float*>(s.act);          // >= 4 * BT * ALD * 2 B = 34,816 B = 8704 floats
    s.sum = scratch + 4096;                                    // [BT][ROWS+1] = 2080 floats, past the last reduction round's reads

    // ---- one-time: resident weight slice (fp32 -> bf16), query-projection slice ----
    for (int idx = tid; idx < ROWS * Kp; idx += PT) {
        const int r = idx / Kp, k = idx % Kp;
        const int g = r / UNITS, u = r % UNITS;
        float w = 0.f;
        if (k < p.K && u0 + u < D) w = p.W[(size_t)(g * D + u0 + u) * p.ldw + k];
        s.W[r * WLD + k] = __float2bfloat16_rn(w);
    }
    if (ATT) {
        for (int idx = tid; idx < p.A * UNITS; idx += PT) {
            const int a = idx / UNITS, u = idx % UNITS;
            s.wq[a * (UNITS + 1) + u] = (u0 + u < D) ? p.Wq[(size_t)a * D + u0 + u] : 0.f;
        }
        for (int idx = tid; idx < p.A * 40; idx += PT) sWcB[idx] = p.WcB[idx];
    }
    __syncthreads();

    const int nchunks = (Kp + CHUNK - 1) / CHUNK;
    const float inv_h = 1.f / (1.f - p.rate_h), inv_c = 1.f / (1.f - p.rate_c);
    unsigned target = 0;
    PROF_DECL

    for (int i = 0; i < p.T; ++i) {
        // =================== gate GEMM: acc[b, r] = sum_k act[b, k] * W[r, k] ===================
        float acc[2][8][4];
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
#pragma unroll
            for (int nt = 0; nt < 8; ++nt)
#pragma unroll
                for (int e = 0; e < 4; ++e) acc[mt][nt][e] = 0.f;

        // prefetch the epilogue operands of this thread's (b, u) pairs: their DRAM latency hides behind the GEMM
        float pre[2][6];
        uint8_t pm[2][2];
#pragma unroll
        for (int e2 = 0; e2 < 2; ++e2) {
            const int idx = tid + e2 * PT;
            const int bl = idx / UNITS, uu = idx % UNITS, b = b0 + bl, u = u0 + uu;
            pm[e2][0] = 1; pm[e2][1] = 1;
#pragma unroll
            for (int j = 0; j < 6; ++j) pre[e2][j] = 0.f;
            if (idx < BT * UNITS && b < B && u < D) {
                const size_t g0 = ((size_t)i * B + b) * 4 * D + u, mi = ((size_t)i * B + b) * D + u;
                pre[e2][0] = p.gates[g0]; pre[e2][1] = p.gates[g0 + D]; pre[e2][2] = p.gates[g0 + 2 * D]; pre[e2][3] = p.gates[g0 + 3 * D];
                pre[e2][4] = p.cstate[mi];
                if (p.kind == B200TTS_CELL_ZONEOUT) pre[e2][5] = p.actf[((size_t)i * B + b) * p.ldf + p.hcol + u];
                if (p.training && p.mask_h) pm[e2][0] = p.mask_h[mi];
                if (p.training && p.mask_c) pm[e2][1] = p.mask_c[mi];
            }
        }

        const __nv_bfloat16* arow = p.actb + ((size_t)i * B + b0) * Kp;
        auto issue = [&](int c) {
            if (c < nchunks) {
                __nv_bfloat16* dst = s.act + (size_t)(c % NSTAGE) * BT * ALD;
                const int kbase = c * CHUNK;
                const int segs = min(CHUNK, Kp - kbase) / 8;            // 16-byte segments per row in this chunk
                for (int idx = tid; idx < BT * segs; idx += PT) {
                    const int r = idx / segs, sg = idx % segs;
                    __nv_bfloat16* d = dst + r * ALD + sg * 8;
                    if (b0 + r < B) cp_async16(d, arow + (size_t)r * Kp + kbase + sg * 8);
                    else *reinterpret_cast<uint4*>(d) = make_uint4(0u, 0u, 0u, 0u);
                }
            }
            cp_async_commit();          // always commit (possibly empty) so that the group count stays uniform
        };
#pragma unroll
        for (int c = 0; c < NSTAGE - 1; ++c) issue(c);
        for (int c = 0; c < nchunks; ++c) {
            cp_async_wait<NSTAGE - 2>();
            __syncthreads();            // chunk c has landed for everyone; everyone is done computing chunk c-1
            issue(c + NSTAGE - 1);      // refills the stage chunk c-1 used
            const __nv_bfloat16* ab = s.act + (size_t)(c % NSTAGE) * BT * ALD;
            const int kbase = c * CHUNK;
            const int ksteps = min(CHUNK, Kp - kbase) / 16;
            for (int ks = warp; ks < ksteps; ks += 8) {
                const int kk = ks * 16;
                uint32_t af[2][4], bf[4][4];
#pragma unroll
                for (int mt = 0; mt < 2; ++mt)
                    ldmatrix_x4(af[mt][0], af[mt][1], af[mt][2], af[mt][3], ab + (mt * 16 + (lane & 15)) * ALD + kk + (lane >> 4) * 8);
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    ldmatrix_x4(bf[j][0], bf[j][1], bf[j][2], bf[j][3],
                                s.W + (size_t)(j * 16 + (lane & 7) + ((lane >> 4) << 3)) * WLD + kbase + kk + ((lane >> 3) & 1) * 8);
#pragma unroll
                for (int mt = 0; mt < 2; ++mt)
#pragma unroll
                    for (int nt = 0; nt < 8; ++nt) mma_bf16(acc[mt][nt], af[mt], bf[nt >> 1][(nt & 1) * 2], bf[nt >> 1][(nt & 1) * 2 + 1]);
            }
        }
        cp_async_wait<0>();
        __syncthreads();                // the stages are free: the reduction scratch aliases them

        PROF_MARK(0);
        // =================== tree reduction over the 8 warps (K split) ===================
        // accumulator element (mt, nt, e): b = mt*16 + g + 8*(e>>1), r = nt*8 + 2*tq + (e&1)
        const int g = lane >> 2, tq = lane & 3;
#pragma unroll
        for (int half = 4; half >= 1; half >>= 1) {
            if (warp >= half && warp < 2 * half) {
                float* dst = scratch + (size_t)(warp - half) * (BT * ROWS);
#pragma unroll
                for (int mt = 0; mt < 2; ++mt)
#pragma unroll
                    for (int nt = 0; nt < 8; ++nt)
#pragma unroll
                        for (int e = 0; e < 4; ++e) dst[((mt * 8 + nt) * 4 + e) * 32 + lane] = acc[mt][nt][e];
            }
            __syncthreads();
            if (warp < half) {
                const float* src = scratch + (size_t)warp * (BT * ROWS);
#pragma unroll
                for (int mt = 0; mt < 2; ++mt)
#pragma unroll
                    for (int nt = 0; nt < 8; ++nt)
#pragma unroll
                        for (int e = 0; e < 4; ++e) acc[mt][nt][e] += src[((mt * 8 + nt) * 4 + e) * 32 + lane];
            }
            __syncthreads();
        }
        if (warp == 0) {
#pragma unroll
            for (int mt = 0; mt < 2; ++mt)
#pragma unroll
                for (int nt = 0; nt < 8; ++nt)
#pragma unroll
                    for (int e = 0; e < 4; ++e)
                        s.sum[(mt * 16 + g + 8 * (e >> 1)) * (ROWS + 1) + nt * 8 + 2 * tq + (e & 1)] = acc[mt][nt][e];
        }
        __syncthreads();

        PROF_MARK(1);
        // =================== LSTM cell + regulariser (2 (b, u) pairs per thread) ===================
#pragma unroll
        for (int e2 = 0; e2 < 2; ++e2) {
            const int idx = tid + e2 * PT;
            if (idx >= BT * UNITS) continue;
            const int bl = idx / UNITS, uu = idx % UNITS, b = b0 + bl, u = u0 + uu;
            float hs = 0.f;
            if (b < B && u < D) {
                const size_t g0 = ((size_t)i * B + b) * 4 * D + u;
                const float zi = pre[e2][0] + s.sum[bl * (ROWS + 1) + uu];
                const float zf = pre[e2][1] + s.sum[bl * (ROWS + 1) + UNITS + uu];
                const float zg = pre[e2][2] + s.sum[bl * (ROWS + 1) + 2 * UNITS + uu];
                const float zo = pre[e2][3] + s.sum[bl * (ROWS + 1) + 3 * UNITS + uu];
                const float gi = sigmoidf_acc(zi), gf = sigmoidf_acc(zf), gg = tanhf(zg), go = sigmoidf_acc(zo);
                const size_t bu = (size_t)b * D + u;
                const float cp = pre[e2][4];
                float cn = gf * cp + gi * gg;
                float hn = go * tanhf(cn);
                p.gates[g0] = gi; p.gates[g0 + D] = gf; p.gates[g0 + 2 * D] = gg; p.gates[g0 + 3 * D] = go;
                if (p.kind == B200TTS_CELL_ZONEOUT) {
                    const float hp = pre[e2][5];
                    if (p.training) {
                        float dh = hn - hp, dc = cn - cp;
                        if (p.mask_h) dh = dh * (float)pm[e2][0] * inv_h;
                        if (p.mask_c) dc = dc * (float)pm[e2][1] * inv_c;
                        hn = (1.f - p.rate_h) * dh + hp;
                        cn = (1.f - p.rate_c) * dc + cp;
                    } else {
                        hn = p.rate_h * hp + (1.f - p.rate_h) * hn;
                        cn = p.rate_c * cp + (1.f - p.rate_c) * cn;
                    }
                } else if (p.training && p.mask_h) {
                    hn = hn * (float)pm[e2][0] * inv_h;
                }
                p.cstate[(size_t)(i + 1) * B * D + bu] = cn;
                p.actf[((size_t)(i + 1) * B + b) * p.ldf + p.hcol + u] = hn;
                p.actb[((size_t)(i + 1) * B + b) * Kp + p.hcol + u] = __float2bfloat16_rn(hn);
                hs = hn;
            }
            if (ATT) s.hs[uu * (BT + 4) + bl] = hs;
        }

        if (ATT) {
            __syncthreads();
            // partial query projection of this CTA's 16 hidden units: qpart[rb, b, a]; thread = (a, 16 utterances)
            for (int idx = tid; idx < p.A * (BT / 16); idx += PT) {
                const int a = idx % p.A, bg = idx / p.A;
                float qa[16];
#pragma unroll
                for (int j = 0; j < 16; ++j) qa[j] = 0.f;
#pragma unroll
                for (int uu = 0; uu < UNITS; ++uu) {
                    const float wv = s.wq[a * (UNITS + 1) + uu];
                    const float4* h4 = reinterpret_cast<const float4*>(&s.hs[uu * (BT + 4) + bg * 16]);
#pragma unroll
                    for (int j4 = 0; j4 < 4; ++j4) {
                        const float4 hv = h4[j4];
                        qa[4 * j4] = fmaf(wv, hv.x, qa[4 * j4]); qa[4 * j4 + 1] = fmaf(wv, hv.y, qa[4 * j4 + 1]);
                        qa[4 * j4 + 2] = fmaf(wv, hv.z, qa[4 * j4 + 2]); qa[4 * j4 + 3] = fmaf(wv, hv.w, qa[4 * j4 + 3]);
                    }
                }
#pragma unroll
                for (int j = 0; j < 16; ++j)
                    if (b0 + bg * 16 + j < B) p.qpart[((size_t)rb * B + b0 + bg * 16 + j) * p.A + a] = qa[j];
            }
        }
        PROF_MARK(2);
        if (!grid_barrier<false>(p.barrier, target, nblocks, p.abort_flag, &s_ok)) return;
        PROF_MARK(3);

        if (ATT) {
            // =================== attention of utterance `cta` (CTAs 0 .. B-1) ===================
            if (cta < B) {
                const int b = cta, L = p.L, A = p.A, M = p.M, half = (p.KC - 1) / 2;
                float* qb = scratch;                       // [A]
                float* vv = qb + A;                        // [A]
                float* e = vv + A;                         // [L16]
                float* red = e + p.MT * 16;                // [64]
                float* cred = red + 64;                    // [8][M]  (first used as [PT/A][A] query partials)
                uint32_t* Ph = reinterpret_cast<uint32_t*>(cred + 8 * M);     // [L16 + 48] Toeplitz pair arrays (hi / lo bf16 split)
                uint32_t* Pl = Ph + (p.MT * 16 + 48);
                int len = p.lengths[b];
                len = len < 0 ? 0 : (len > L ? L : len);
                const float* cum_prev = p.cum + ((size_t)i * B + b) * L;
                {   // q[a] = sum over the RB per-CTA partial projections: thread = (4 attention dims, one eighth of the row blocks),
                    // all of its 16-byte loads in flight at once
                    {
                        const int a4 = tid & 31, sl = tid >> 5;
                        const int per = (p.RB + 7) / 8, r0 = sl * per, r1 = min(p.RB, r0 + per);
                        float4 qs = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (a4 * 4 < A) {
                            for (int r = r0; r < r1; r += 8) {
                                float4 v[8];
#pragma unroll
                                for (int j = 0; j < 8; ++j)
                                    v[j] = (r + j < r1) ? __ldcg(reinterpret_cast<const float4*>(p.qpart + ((size_t)(r + j) * B + b) * A) + a4)
                                                        : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                                for (int j = 0; j < 8; ++j) { qs.x += v[j].x; qs.y += v[j].y; qs.z += v[j].z; qs.w += v[j].w; }
                            }
                            *reinterpret_cast<float4*>(cred + sl * A + a4 * 4) = qs;
                        }
                    }
                    // cumulative weights -> (hi, lo) bf16 pairs: Ph[x] = (c[x], c[x+1]) with c[j] = cum[j - half]
                    for (int x = tid; x < p.MT * 16 + 48; x += PT) {
                        float c0 = 0.f, c1 = 0.f;
                        const int la = x - half, lb = x + 1 - half;
                        if (la >= 0 && la < L) c0 = __ldcg(cum_prev + la);
                        if (lb >= 0 && lb < L) c1 = __ldcg(cum_prev + lb);
                        const __nv_bfloat16 h0 = __float2bfloat16_rn(c0), h1 = __float2bfloat16_rn(c1);
                        __nv_bfloat162 hp2; hp2.x = h0; hp2.y = h1;
                        Ph[x] = *reinterpret_cast<uint32_t*>(&hp2);
                        Pl[x] = pack2(c0 - __bfloat162float(h0), c1 - __bfloat162float(h1));
                    }
                    __syncthreads();
                    for (int a2 = tid; a2 < A; a2 += PT) {
                        float q = 0.f;
#pragma unroll
                        for (int sl2 = 0; sl2 < 8; ++sl2) q += cred[sl2 * A + a2];
                        p.qsave[((size_t)i * B + b) * A + a2] = q;
                        qb[a2] = q + p.bias[a2];
                        vv[a2] = p.v[a2];
                    }
                }
                __syncthreads();
                PROF_MARK(4);
                // energies on the tensor cores: S[l, a] = sum_k cumpad[l + k] * Wcomb[a, k]; warp owns position tiles {warp, warp+8}
                {
                    const int g = lane >> 2, tq = lane & 3;
                    const int mtiles = (len + 15) / 16;
                    for (int mt = warp; mt < mtiles; mt += 8) {
                        const int l0 = mt * 16;
                        float sacc[16][4];
#pragma unroll
                        for (int nt = 0; nt < 16; ++nt)
#pragma unroll
                            for (int e4 = 0; e4 < 4; ++e4) sacc[nt][e4] = 0.f;
#pragma unroll
                        for (int ks = 0; ks < 2; ++ks) {
                            const int x = l0 + ks * 16 + g + 2 * tq;
                            const uint32_t ah[4] = {Ph[x], Ph[x + 8], Ph[x + 8], Ph[x + 16]};
                            const uint32_t al[4] = {Pl[x], Pl[x + 8], Pl[x + 8], Pl[x + 16]};
#pragma unroll
                            for (int np = 0; np < 8; ++np) {
                                uint32_t bfr[4];
                                ldmatrix_x4(bfr[0], bfr[1], bfr[2], bfr[3],
                                            sWcB + (size_t)(np * 16 + (lane & 7) + ((lane >> 4) << 3)) * 40 + ks * 16 + ((lane >> 3) & 1) * 8);
                                mma_bf16(sacc[2 * np], ah, bfr[0], bfr[1]);
                                mma_bf16(sacc[2 * np], al, bfr[0], bfr[1]);
                                mma_bf16(sacc[2 * np + 1], ah, bfr[2], bfr[3]);
                                mma_bf16(sacc[2 * np + 1], al, bfr[2], bfr[3]);
                            }
                        }
                        const uint4* mf = reinterpret_cast<const uint4*>(p.memTf + (((size_t)b * p.MT + mt) * 32 + lane) * 64);
                        float e0 = 0.f, e1 = 0.f;
#pragma unroll
                        for (int c4 = 0; c4 < 8; ++c4) {
                            const uint4 raw = mf[c4];
                            const uint32_t words[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
                            for (int hf = 0; hf < 2; ++hf) {
                                const int nt = 2 * c4 + hf, a0 = nt * 8 + 2 * tq;
                                const float2 m01 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&words[2 * hf]));
                                const float2 m23 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&words[2 * hf + 1]));
                                e0 = fmaf(vv[a0], tanh_fast(sacc[nt][0] + qb[a0] + m01.x), e0);
                                e0 = fmaf(vv[a0 + 1], tanh_fast(sacc[nt][1] + qb[a0 + 1] + m01.y), e0);
                                e1 = fmaf(vv[a0], tanh_fast(sacc[nt][2] + qb[a0] + m23.x), e1);
                                e1 = fmaf(vv[a0 + 1], tanh_fast(sacc[nt][3] + qb[a0 + 1] + m23.y), e1);
                            }
                        }
                        e0 += __shfl_xor_sync(0xffffffffu, e0, 1); e0 += __shfl_xor_sync(0xffffffffu, e0, 2);
                        e1 += __shfl_xor_sync(0xffffffffu, e1, 1); e1 += __shfl_xor_sync(0xffffffffu, e1, 2);
                        if (tq == 0) { e[l0 + g] = e0; e[l0 + g + 8] = e1; }
                    }
                }
                __syncthreads();
                PROF_MARK(5);
                float mx = -INFINITY;
                for (int l = tid; l < len; l += PT) mx = fmaxf(mx, e[l]);
                mx = block_max(mx, red);
                float sum = 0.f;
                for (int l = tid; l < len; l += PT) { const float ex = expf(e[l] - mx); e[l] = ex; sum += ex; }
                sum = block_sum(sum, red);
                float* cum_next = p.cum + ((size_t)(i + 1) * B + b) * L;
                const float inv_sum = 1.f / sum;
                for (int l = tid; l < p.MT * 16; l += PT) {      // the padded tail must be zero: the context MMA reads whole 16-position tiles
                    const float w = l < len ? e[l] * inv_sum : 0.f;
                    e[l] = w;
                    if (l < L) {
                        p.align[(size_t)b * p.align_bstride + (size_t)i * L + l] = w;
                        cum_next[l] = __ldcg(cum_prev + l) + w;
                    }
                }
                __syncthreads();
                // context on the tensor cores: ctx[m] = sum_l memory[l, m] * w[l].  A = memory^T fragments (fragment-major bf16, one
                // 16-byte load per lane per MMA), B = (hi(w), lo(w)) in columns 0 / 1 -> column 0 + column 1 of D is the fp32-weighted sum.
                {
                    const int g = lane >> 2, tq = lane & 3;
                    const int ktiles = (len + 15) / 16;
                    for (int mt = warp; mt < p.M16; mt += 8) {
                        const uint4* fr = p.memFf + (((size_t)b * p.M16 + mt) * p.MT) * 32 + lane;
                        float dacc[4] = {0.f, 0.f, 0.f, 0.f};
                        for (int kt0 = 0; kt0 < ktiles; kt0 += 6) {
                            uint4 av[6];
#pragma unroll
                            for (int j = 0; j < 6; ++j)
                                if (kt0 + j < ktiles) av[j] = __ldg(fr + (size_t)(kt0 + j) * 32);
#pragma unroll
                            for (int j = 0; j < 6; ++j) {
                                if (kt0 + j < ktiles) {
                                    uint32_t b0 = 0u, b1 = 0u;
                                    if (g < 2) {
                                        const float* wl = e + (kt0 + j) * 16 + 2 * tq;
                                        float w0 = wl[0], w1 = wl[1], w2 = wl[8], w3 = wl[9];
                                        const __nv_bfloat16 h0 = __float2bfloat16_rn(w0), h1 = __float2bfloat16_rn(w1);
                                        const __nv_bfloat16 h2 = __float2bfloat16_rn(w2), h3 = __float2bfloat16_rn(w3);
                                        if (g == 1) { w0 -= __bfloat162float(h0); w1 -= __bfloat162float(h1); w2 -= __bfloat162float(h2); w3 -= __bfloat162float(h3); }
                                        else { w0 = __bfloat162float(h0); w1 = __bfloat162float(h1); w2 = __bfloat162float(h2); w3 = __bfloat162float(h3); }
                                        b0 = pack2(w0, w1); b1 = pack2(w2, w3);
                                    }
                                    const uint32_t af[4] = {av[j].x, av[j].y, av[j].z, av[j].w};
                                    mma_bf16(dacc, af, b0, b1);
                                }
                            }
                        }
                        if (tq == 0) {
                            const int m0 = mt * 16 + g;
                            const float c0 = dacc[0] + dacc[1], c1 = dacc[2] + dacc[3];
                            if (m0 < M) {
                                p.actf[((size_t)(i + 1) * B + b) * p.ldf + m0] = c0;
                                p.actb[((size_t)(i + 1) * B + b) * Kp + m0] = __float2bfloat16_rn(c0);
                            }
                            if (m0 + 8 < M) {
                                p.actf[((size_t)(i + 1) * B + b) * p.ldf + m0 + 8] = c1;
                                p.actb[((size_t)(i + 1) * B + b) * Kp + m0 + 8] = __float2bfloat16_rn(c1);
                            }
                        }
                    }
                }
            }
            PROF_MARK(6);
            if (!grid_barrier<false>(p.barrier, target, nblocks, p.abort_flag, &s_ok)) return;
            PROF_MARK(7);
        }
    }
    PROF_FLUSH;
}

size_t loop_smem_bytes(int Kp, int A, bool att, int L, int M, int nstage) {
    size_t b = (size_t)ROWS * (Kp + 8) * 2 + (size_t)nstage * BT * ALD * 2 + (size_t)UNITS * (BT + 4) * 4;
    if ((size_t)nstage * BT * ALD * 2 < (size_t)4 * BT * ROWS * 4) return 0;   // reduction scratch (the gate sums live inside it)
    if (att) {
        b += (size_t)A * (UNITS + 1) * 4 + (size_t)A * 40 * 2;
        const int L16 = (L + 15) / 16 * 16;
        // the attention scratch aliases the activation stages; it must fit there
        const size_t need = ((size_t)2 * A + L16 + 64 + (size_t)8 * M + 2 * (L16 + 48)) * 4;
        if (need > (size_t)nstage * BT * ALD * 2 || PT % A != 0 || A != 128) return 0;
    }
    return b;
}

__global__ void f32_to_bf16_rows_kernel(__nv_bfloat16* __restrict__ dst, int ldd, const float* __restrict__ src, int lds, size_t rows,
                                        int cols) {
    const size_t total = rows * ldd;
    for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const size_t r = idx / ldd;
        const int c = idx % ldd;
        dst[idx] = __float2bfloat16_rn(c < cols ? src[r * lds + c] : 0.f);
    }
}

// WcB[a][40] = bf16 Wcomb[a][k] (zero for k >= KC);  memTf = fragment-major bf16 memory projection:
// memTf[b][mt][lane][nt*4 + e] = memT[b][mt*16 + (lane>>2) + 8*(e>>1)][nt*8 + 2*(lane&3) + (e&1)]
__global__ void att_prep_kernel(__nv_bfloat16* __restrict__ WcB, __nv_bfloat16* __restrict__ memTf, const float* __restrict__ WcombT,
                                const float* __restrict__ memT, int B, int L, int A, int KC, int MT) {
    const size_t n1 = (size_t)A * 40, n3 = (size_t)B * MT * 32 * 64;
    for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < n1 + n3; idx += (size_t)gridDim.x * blockDim.x) {
        if (idx < n1) {
            const int a = idx / 40, k = idx % 40;
            WcB[idx] = __float2bfloat16_rn(k < KC ? WcombT[(size_t)k * A + a] : 0.f);
        } else {
            const size_t j = idx - n1;
            const int v = j % 64, lane = (j / 64) % 32, mt = (j / (64 * 32)) % MT, b = j / ((size_t)64 * 32 * MT);
            const int nt = v / 4, e = v % 4, g = lane >> 2, tq = lane & 3;
            const int l = mt * 16 + g + 8 * (e >> 1), a = nt * 8 + 2 * tq + (e & 1);
            memTf[j] = __float2bfloat16_rn((l < L && a < A) ? memT[((size_t)b * L + l) * A + a] : 0.f);
        }
    }
}

// Fragment-major bf16 copies of the encoder memory for mma.m16n8k16 A operands (one 16-byte load per lane per MMA):
//   memFf[b][mt][kt][lane] : A[r][c] = memory[b][kt*16 + c][mt*16 + r]   (memory^T: rows = memory dims, k = positions)   -> context
//   memFb[b][lt][kt][lane] : A[r][c] = memory[b][lt*16 + r][kt*16 + c]   (rows = positions, k = memory dims)             -> d weights
// lane (g = lane>>2, tq = lane&3) holds {A[g][2tq..+1], A[g+8][2tq..+1], A[g][2tq+8..+9], A[g+8][2tq+8..+9]}; zero padded.
__global__ void mem_frag_kernel(uint4* __restrict__ memFf, uint4* __restrict__ memFb, const float* __restrict__ memory, int B, int L, int M,
                                int M16, int MT) {
    const size_t per = (size_t)B * M16 * MT * 32;
    for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < 2 * per; idx += (size_t)gridDim.x * blockDim.x) {
        const bool fwd = idx < per;
        const size_t j = fwd ? idx : idx - per;
        const int lane = j % 32, g = lane >> 2, tq = lane & 3;
        int kt, ot, b;
        if (fwd) { kt = (j / 32) % MT; ot = (j / ((size_t)32 * MT)) % M16; b = j / ((size_t)32 * MT * M16); }
        else { kt = (j / 32) % M16; ot = (j / ((size_t)32 * M16)) % MT; b = j / ((size_t)32 * M16 * MT); }
        auto at = [&](int r, int c) -> float {
            const int l = fwd ? kt * 16 + c : ot * 16 + r;
            const int m = fwd ? ot * 16 + r : kt * 16 + c;
            return (l < L && m < M) ? memory[((size_t)b * L + l) * M + m] : 0.f;
        };
        uint4 v;
        v.x = pack2(at(g, 2 * tq), at(g, 2 * tq + 1));
        v.y = pack2(at(g + 8, 2 * tq), at(g + 8, 2 * tq + 1));
        v.z = pack2(at(g, 2 * tq + 8), at(g, 2 * tq + 9));
        v.w = pack2(at(g + 8, 2 * tq + 8), at(g + 8, 2 * tq + 9));
        (fwd ? memFf : memFb)[j] = v;
    }
}

// WcombT[k, a] = sum_c Wloc[a, c] * Wc[c, k]
__global__ void wcomb_kernel(float* __restrict__ WcombT, const float* __restrict__ Wloc, const float* __restrict__ Wc, int A, int C, int K) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= K * A) return;
    const int k = idx / A, a = idx % A;
    float s = 0.f;
    for (int c = 0; c < C; ++c) s = fmaf(Wloc[a * C + c], Wc[c * K + k], s);
    WcombT[idx] = s;
}

inline int grid_for(size_t n) {
    size_t g = (n + 255) / 256;
    return (int)(g > 148 * 16 ? 148 * 16 : (g < 1 ? 1 : g));
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
PersistLayout persist_layout(const b200tts_decoder_shape& s) {
    PersistLayout l;
    size_t off = 0;     // in bytes, 256-aligned regions
    auto take = [&](size_t n) { size_t o = off; off = (off + n + 255) / 256 * 256; return o; };
    const size_t T = s.T, B = s.B;
    l.Kp_att = (s.M + s.D + 15) / 16 * 16;
    l.Kp_gen = (s.D + 15) / 16 * 16;
    l.ldm = (s.M + 7) / 8 * 8;
    // sized for the 64-column k-block padding of the tcgen05 loops (decoder_persist_tc.cu) as well
    l.aib = take((T + 1) * B * (size_t)((s.M + s.D + 63) / 64 * 64) * 2);
    l.hgb = take((T + 1) * B * (size_t)((s.D + 63) / 64 * 64) * 2);
    l.memTb = take(B * (size_t)s.L * s.A * 2);
    l.memb = take(B * (size_t)s.L * l.ldm * 2);
    l.wcombT = take((size_t)s.K * s.A * 4);
    l.wcb = take((size_t)s.A * 40 * 2);
    l.MT = (s.L + 15) / 16;
    l.memTf = take((size_t)s.B * l.MT * 32 * 64 * 2);
    l.M16 = (s.M + 15) / 16;
    l.memFf = take((size_t)s.B * l.M16 * l.MT * 32 * 16);
    l.memFb = take((size_t)s.B * l.M16 * l.MT * 32 * 16);
    l.barrier = take(256 + 148 * 8 * 8 * 4);   // barrier + abort flag, then 4 x [148][8] profile counters (att, gen, att roles, gen roles)
    l.total = off;
    return l;
}

bool persist_supported(const b200tts_decoder_shape& s) {
    if (s.D % UNITS != 0) return false;
    const int RB = s.D / UNITS, NBH = (s.B + BT - 1) / BT;
    if (RB * NBH > 148 || s.B > RB * NBH) return false;
    const PersistLayout l = persist_layout(s);
    if (s.K > 32) return false;
    const size_t a = loop_smem_bytes(l.Kp_att, s.A, true, s.L, s.M, ATT_STAGES), g = loop_smem_bytes(l.Kp_gen, s.A, false, 0, 0, GEN_STAGES);
    return a != 0 && g != 0 && a <= 227 * 1024 && g <= 227 * 1024;
}

static int launch_loop(bool att, const LoopArgs& a, size_t smem, cudaStream_t st) {
    void* fn = att ? (void*)lstm_loop_kernel<true, ATT_STAGES> : (void*)lstm_loop_kernel<false, GEN_STAGES>;
    LoopArgs args = a;
    void* params[] = {&args};
    return launch_persistent(fn, a.RB * a.NBH, PT, smem, params, st, "persistent loop", nullptr);
}

// bf16 memory, Wcomb and the fragment-major projections shared by the forward and backward persistent kernels
int persist_att_prep(const b200tts_decoder_shape& s, const b200tts_decoder_params& w, const b200tts_decoder_inputs& in,
                     const DecoderLayout& fl, float* ws, unsigned char* pws, cudaStream_t st) {
    const PersistLayout l = persist_layout(s);
    const int B = s.B, M = s.M;
    __nv_bfloat16* memb = reinterpret_cast<__nv_bfloat16*>(pws + l.memb);
    float* wcombT = reinterpret_cast<float*>(pws + l.wcombT);
    f32_to_bf16_rows_kernel<<<grid_for((size_t)B * s.L * l.ldm), 256, 0, st>>>(memb, l.ldm, in.memory, M, (size_t)B * s.L, M);
    B200_LAUNCH_CHECK();
    wcomb_kernel<<<cdiv(s.K * s.A, 256), 256, 0, st>>>(wcombT, w.attn_location, w.attn_loc_features, s.A, s.C, s.K);
    B200_LAUNCH_CHECK();
    __nv_bfloat16* wcb = reinterpret_cast<__nv_bfloat16*>(pws + l.wcb);
    __nv_bfloat16* memTf = reinterpret_cast<__nv_bfloat16*>(pws + l.memTf);
    att_prep_kernel<<<148 * 4, 256, 0, st>>>(wcb, memTf, wcombT, ws + fl.memT, B, s.L, s.A, s.K, l.MT);
    B200_LAUNCH_CHECK();
    mem_frag_kernel<<<148 * 4, 256, 0, st>>>(reinterpret_cast<uint4*>(pws + l.memFf), reinterpret_cast<uint4*>(pws + l.memFb), in.memory, B,
                                             s.L, M, l.M16, l.MT);
    B200_LAUNCH_CHECK();
    return B200TTS_OK;
}

// Attention-LSTM + attention loop (all T steps), mma.sync variant (any D % 16 == 0).  Expects: ga = input projection, ai row 0 = 0,
// ca row 0 = 0, cum row 0 = 0 and persist_att_prep() done.
int persist_att_loop(const b200tts_decoder_shape& s, const b200tts_decoder_params& w, const b200tts_decoder_inputs& in,
                     const DecoderLayout& fl, float* ws, unsigned char* pws, float* align, cudaStream_t st) {
    const PersistLayout l = persist_layout(s);
    const int B = s.B, T = s.T, D = s.D, M = s.M, MD = M + D;
    __nv_bfloat16* aib = reinterpret_cast<__nv_bfloat16*>(pws + l.aib);
    __nv_bfloat16* memb = reinterpret_cast<__nv_bfloat16*>(pws + l.memb);
    B200_CUDA(cudaMemsetAsync(aib, 0, (size_t)B * l.Kp_att * 2, st));                 // operand of step 0
    __nv_bfloat16* wcb = reinterpret_cast<__nv_bfloat16*>(pws + l.wcb);
    __nv_bfloat16* memTf = reinterpret_cast<__nv_bfloat16*>(pws + l.memTf);
    uint4* memFf = reinterpret_cast<uint4*>(pws + l.memFf);
    // padding columns [MD, Kp) of every operand row must be zero (weights there are zero too, but NaN * 0 would poison)
    if (l.Kp_att != MD) B200_CUDA(cudaMemsetAsync(aib, 0, (size_t)(T + 1) * B * l.Kp_att * 2, st));
    LoopArgs a{};
    a.B = B; a.T = T; a.D = D; a.K = MD; a.Kp = l.Kp_att; a.RB = D / UNITS; a.NBH = (B + BT - 1) / BT;
    a.W = ws + fl.wcat_att; a.ldw = MD;
    a.actb = aib; a.actf = ws + fl.ai; a.ldf = MD; a.hcol = M;
    a.gates = ws + fl.ga; a.cstate = ws + fl.ca;
    a.mask_h = in.mask_att_h; a.mask_c = in.mask_att_c; a.kind = s.cell_kind; a.training = s.training; a.rate_h = s.rate_h; a.rate_c = s.rate_c;
    a.L = s.L; a.M = M; a.A = s.A; a.KC = s.K;
    a.Wq = w.attn_query; a.qpart = ws + fl.qpart; a.qsave = ws + fl.q; a.WcB = wcb; a.memTf = memTf; a.MT = l.MT; a.bias = w.attn_bias; a.v = w.attn_energy;
    a.memb = memb; a.ldm = l.ldm; a.memFf = memFf; a.M16 = l.M16; a.lengths = in.text_lengths; a.cum = ws + fl.cum;
    a.align = align; a.align_bstride = (long long)T * s.L;
    B200_TRY(reset_grid_barrier(pws + l.barrier, a, st));
    return launch_loop(true, a, loop_smem_bytes(l.Kp_att, s.A, true, s.L, M, ATT_STAGES), st);
}

// Generator-LSTM loop.  Expects: gg = input projection, hg row 0 = 0, cg row 0 = 0.
int persist_gen_loop(const b200tts_decoder_shape& s, const b200tts_decoder_params& w, const b200tts_decoder_inputs& in,
                     const DecoderLayout& fl, float* ws, unsigned char* pws, cudaStream_t st) {
    const PersistLayout l = persist_layout(s);
    const int B = s.B, T = s.T, D = s.D;
    __nv_bfloat16* hgb = reinterpret_cast<__nv_bfloat16*>(pws + l.hgb);
    B200_CUDA(cudaMemsetAsync(hgb, 0, (size_t)(l.Kp_gen != D ? (size_t)(T + 1) : 1) * B * l.Kp_gen * 2, st));
    LoopArgs a{};
    a.B = B; a.T = T; a.D = D; a.K = D; a.Kp = l.Kp_gen; a.RB = D / UNITS; a.NBH = (B + BT - 1) / BT;
    a.W = w.gen_w_hh; a.ldw = D;
    a.actb = hgb; a.actf = ws + fl.hg; a.ldf = D; a.hcol = 0;
    a.gates = ws + fl.gg; a.cstate = ws + fl.cg;
    a.mask_h = in.mask_gen_h; a.mask_c = in.mask_gen_c; a.kind = s.cell_kind; a.training = s.training; a.rate_h = s.rate_h; a.rate_c = s.rate_c;
    B200_TRY(reset_grid_barrier(pws + l.barrier, a, st));
    a.prof += 148 * 8;
    return launch_loop(false, a, loop_smem_bytes(l.Kp_gen, s.A, false, 0, 0, GEN_STAGES), st);
}

}  // namespace b200tts
