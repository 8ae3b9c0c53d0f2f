// Persistent recurrent kernels of the bf16 perf mode (forward), Blackwell-native: TMA + tcgen05 + TMEM.
//
// ONE cooperative launch runs all T steps of an LSTM recurrence (attention-LSTM + location-sensitive attention, or the
// generator LSTM).  CTA (rb, bh) owns 16 hidden units x {i,f,g,o} = 64 gate rows and a batch half of 32 utterances:
//   * weight-stationary: the bf16 slice W[64 rows, K] lives in shared memory for the whole sequence, laid out as
//     K-major SWIZZLE_128B tiles of 64 x 64 (8 KB) -- the A operand of tcgen05.mma (M = 64);
//   * per step the bf16 activation operand [32 utterances x K] is fetched by TMA (cp.async.bulk.tensor, 64-column boxes,
//     SWIZZLE_128B) into a small ring -- the B operand (N = 32); one elected thread issues tcgen05.mma.kind::f16
//     (K = 16 per instruction), the fp32 accumulator [64 x 32] lives in TMEM; tcgen05.commit recycles ring slots;
//   * warp roles: warps 0-7 compute (epilogue: tcgen05.ld -> LSTM cell / regulariser -> state stores, attention),
//     warp 8 lane 0 = TMA producer, warp 9 lane 0 = MMA issuer;
//   * the K range is ordered [h | ctx]: the h part (available after the cell barrier) is loaded and multiplied WHILE
//     the attention of the same step runs; only the short ctx part (5 boxes) follows the attention barrier;
//   * grid barriers are monotonic counters in global memory; every wait carries a clock64 watchdog.
// fp32 state (c, h, gates, cumulative weights, context, alignments) is written exactly where the fp32 per-step path
// writes it, so the backward pass is unaffected.
// Reference semantics: modules/tacotron2.py:180-198, modules/layers.py:18-47, modules/attention.py:39-86.
#include <cuda.h>
#include <stdlib.h>
#include <cuda_bf16.h>
#include "decoder_internal.cuh"
#include "persist.cuh"

namespace b200tts {

namespace {

constexpr int NCW = 8;                  // compute warps
constexpr int CT = 32 * NCW;            // compute threads
constexpr int PT = CT + 64;             // + TMA producer warp + MMA issuer warp
constexpr int UNITS = 16;               // hidden units per CTA
constexpr int ROWS = 4 * UNITS;         // gate rows per CTA (MMA M)
constexpr int BT = 32;                  // utterances per CTA (MMA N)
constexpr int KB = 64;                  // K columns per tile / TMA box (128-byte rows)
constexpr int WTILE = ROWS * KB * 2;    // 8 KB
constexpr int ATILE = BT * KB * 2;      // 4 KB
constexpr int TMEM_COLS = 32;

struct TcLoopArgs {
    int B, T, D, K, Kp, RB, NBH;
    int nkb, nkb_h;                           // k-blocks in total / in the h part
    int ch_h, n_h, ch_c, n_c, slot_kb;        // TMA chunking: n_h instructions of ch_h k-blocks (h part), n_c of ch_c (ctx part); slot capacity
    int alias_sum;                            // 1: the accumulator staging s_sum lives in the (then idle) TMA slot (large memory dims)
    int use_btab;                             // 1: the context product's B fragments come from a per-step shared table (built once per CTA)
    const float* W; int ldw; int wcol_h, wcol_c;   // fp32 weights [4D, ldw]: operand column k < D -> wcol_h + k, else wcol_c + k - D
    __nv_bfloat16* actb;                      // [T+1, B, Kp] bf16 operand rows: [h | ctx | 0]
    float* actf; int ldf; int hcol;           // fp32 mirror ([T+1, B, ldf]); h at column hcol, ctx at column 0
    float* gates;                             // [T, B, 4D] in: input projection (+biases); out: activated gates
    float* cstate;                            // [T+1, B, D]
    const uint8_t* mask_h; const uint8_t* mask_c;
    int kind, training; float rate_h, rate_c;
    // attention (ATT instantiation only)
    int L, M, A, KC;
    const float* Wq; float* qpart; float* qsave;
    const __nv_bfloat16* WcB;                 // [A][40]
    const __nv_bfloat16* memTf; int MT;       // [B][MT][32][64]
    const float* bias; const float* v;
    const uint4* memFf; int M16;              // [B][M16][MT][32]
    const int* lengths;
    float* cum; float* align; long long align_bstride;
    unsigned* barrier; int* abort_flag;
    long long* prof;                          // [grid][8] phase cycles seen by compute thread 0
    long long* prof2;                         // [grid][8] MMA issuer (0-3) / TMA producer (4-7) waits
};

using namespace tcx;

// named barrier among the compute warps only
__device__ __forceinline__ void csync() { asm volatile("bar.sync 1, %0;" ::"n"(CT) : "memory"); }

// Block-wide max / sum among the CT compute threads (named barrier 1); `scratch` holds >= 33 floats.
__device__ __forceinline__ float cblock_max(float v, float* scratch) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    v = warp_max(v);
    csync();
    if (lane == 0) scratch[warp] = v;
    csync();
    float t = scratch[lane & (NCW - 1)];
#pragma unroll
    for (int o = NCW / 2; o > 0; o >>= 1) t = fmaxf(t, __shfl_xor_sync(0xffffffffu, t, o));
    return t;
}
__device__ __forceinline__ float cblock_sum(float v, float* scratch) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    v = warp_sum(v);
    csync();
    if (lane == 0) scratch[warp] = v;
    csync();
    float t = scratch[lane & (NCW - 1)];
#pragma unroll
    for (int o = NCW / 2; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    return t;
}

// ALIAS (large memory dims only): the accumulator staging lives in the TMA slot and the ctx part arrives in p.n_c TMA instructions; the
// common instantiation keeps both compile-time constant (this kernel sits at its register cap: every live value counts)
template <bool ATT, bool ALIAS>
__global__ void __launch_bounds__(PT, 1) lstm_loop_tc_kernel(const __grid_constant__ CUtensorMap tmH, const __grid_constant__ CUtensorMap tmC,
                                                             const TcLoopArgs p) {
    extern __shared__ __align__(1024) unsigned char smem_raw0[];
    unsigned char* smem_raw = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw0) + 1023) & ~(uintptr_t)1023);
    __shared__ uint64_t full_bar, full2_bar, empty_bar, accum_bar, xchg_bar;
    __shared__ uint32_t tmem_base_s;
    __shared__ int s_ok;

    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);     // warp-uniform by construction (lets the role loops use uniform registers)
    const int cta = blockIdx.x;
    const int rb = cta % p.RB, bh = cta / p.RB;
    const int u0 = rb * UNITS, b0 = bh * BT;
    const int Kp = p.Kp, D = p.D, B = p.B;
    // the two batch halves never exchange data (a CTA's LSTM rows and the attention pairs it hosts serve the same 32 utterances):
    // each half synchronises on its own barrier counter, 64 arrivals instead of 128
    // (per-batch-half barrier counters were measured SLOWER than one grid-wide counter: +0.9 ms on the attention loop; the cost of a
    // barrier is its latency chain -- store acks, atomic round trip, poll -- not the number of arrivals: tools/microbench/barrier_latency.cu)
    const unsigned nblocks = gridDim.x;
    unsigned* const bar_counter = p.barrier;
    const bool compute = warp < NCW;
    const bool is_producer = (warp == NCW);        // whole warps run the role loops; one elected lane issues the TMA / MMA instructions
    const bool is_mma = (warp == NCW + 1);

    // ---- shared memory carve-up (1024-byte aligned base: SWIZZLE_128B atoms) ----
    size_t off = 0;
    unsigned char* sW = smem_raw + off; off += (size_t)p.nkb * WTILE;                 // [nkb][64 rows][128 B] swizzled
    unsigned char* ring = smem_raw + off;                                             // one slot of [slot_kb][32 rows][128 B] swizzled (TMA)
    {
        const size_t ring_b = (size_t)p.slot_kb * ATILE, sum_b = (size_t)BT * (ROWS + 1) * 4;
        off += ALIAS ? (ring_b > sum_b ? ring_b : sum_b) : ring_b;
    }
    // accumulator staging [32 utterances][64 gate rows + 1]: its own buffer, or (large memory dims, where the resident weight slice leaves no
    // room) the TMA slot itself -- between the commit of a step's last MMA and the next TMA issue nobody else touches the slot
    float* s_sum = ALIAS ? reinterpret_cast<float*>(ring) : reinterpret_cast<float*>(smem_raw + off);
    off += ALIAS ? 0 : (size_t)BT * (ROWS + 1) * 4;
    float* s_hs = reinterpret_cast<float*>(smem_raw + off); off += ATT ? (size_t)UNITS * (BT + 4) * 4 : 0;
    __nv_bfloat16* sWcB = reinterpret_cast<__nv_bfloat16*>(smem_raw + off); off += ATT ? (size_t)(p.A / 2) * 40 * 2 : 0;   // this rank's 64 attention dims
    float* scratch = reinterpret_cast<float*>(smem_raw + off);                        // attention scratch (ATT only)

    // ---- one-time: resident weight slice fp32 -> bf16 in the canonical K-major SWIZZLE_128B layout ----
    for (int idx = tid; idx < ROWS * p.nkb * KB; idx += PT) {
        const int r = idx / (p.nkb * KB), k = idx % (p.nkb * KB);
        const int g = r / UNITS, u = r % UNITS;
        float w = 0.f;
        if (k < p.K && u0 + u < D) w = p.W[(size_t)(g * D + u0 + u) * p.ldw + (k < D ? p.wcol_h + k : p.wcol_c + (k - D))];
        const int kb = k / KB, kc = k % KB, chunk = kc >> 3, e = kc & 7;
        *reinterpret_cast<__nv_bfloat16*>(sW + (size_t)kb * WTILE + r * 128 + ((chunk ^ (r & 7)) << 4) + e * 2) = __float2bfloat16_rn(w);
    }
    if (ATT) {
        for (int idx = tid; idx < (p.A / 2) * 40; idx += PT) sWcB[idx] = p.WcB[(size_t)(cta & 1) * (p.A / 2) * 40 + idx];
    }
    if (tid == 0) {
        mbar_init(&full_bar, 1); mbar_init(&full2_bar, 1); mbar_init(&empty_bar, 1); mbar_init(&xchg_bar, 1);
        mbar_init(&accum_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == NCW + 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "n"(TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    proxy_fence_shared();              // the weight tiles were written through the generic proxy; tcgen05.mma reads via the async proxy
    tc_fence_before();
    __syncthreads();
    if (ATT) { cluster_arrive(); cluster_wait(); }      // one-time: the peer's exchange mbarrier is initialised before any remote st.async targets it
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;
    // instruction descriptor: D = F32, A = B = BF16, both K-major, N >> 3 at bit 17, M >> 4 at bit 24
    const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BT >> 3) << 17) | ((uint32_t)(ROWS >> 4) << 24);

    // A TMA instruction costs ~500 cycles of issue time whatever its size (measured), so the operand is fetched with FEW LARGE
    // boxes: the tensor maps are 3-D {64 columns, rows, k-block} (k-block stride 128 B), one instruction brings ch k-blocks
    // of [32 rows x 128 B] = ch swizzled 4 KB tiles into the single ring slot.
    uint32_t prod_it = 0, cons_it = 0;            // running chunk counters of the producer / MMA thread
    long long rp[4] = {0, 0, 0, 0};               // role-thread cycle counters (see prof2)
    // TMA producer: operand row block of `step`; part 0 = ctx k-blocks (one instruction), part 1 = h k-blocks (n_h instructions)
    auto produce = [&](int step, int part) {
        const long long t0 = clock64();
        proxy_fence_global();          // generic-proxy writes of other CTAs (ordered by the grid barrier) -> async-proxy reads
        const long long t1 = clock64();
        const int n = part ? p.n_h : (ALIAS ? p.n_c : 1), ch = part ? p.ch_h : p.ch_c;
        if (!ATT) {
            // generator loop: the whole operand fits in the ring, so its (<= 2) chunks go to their own offsets with their own barriers and
            // are requested back to back -- the MMAs of the first half run while the second half is still in flight.  (All slots are free
            // here: the previous step's MMAs completed before its cell phase, and the grid barrier lies in between.)
            if (elect_one()) {
                for (int j = 0; j < n; ++j) {
                    uint64_t* fb = j ? &full2_bar : &full_bar;
                    mbar_expect_tx(fb, (uint32_t)ch * ATILE);
                    tma_load_3d(ring + (size_t)j * ch * ATILE, &tmH, fb, 0, step * B + b0, j * ch);
                }
            }
            __syncwarp();
            ++prod_it;
            rp[2 * part] += t1 - t0; rp[2 * part + 1] += clock64() - t1;
            return;
        }
        for (int j = 0; j < n; ++j) {
            mbar_wait(&empty_bar, (prod_it & 1) ^ 1);
            if (elect_one()) {
                if (ALIAS) proxy_fence_shared();           // the slot doubled as the accumulator staging (generic proxy) since its last MMA
                mbar_expect_tx(&full_bar, (uint32_t)ch * ATILE);
                tma_load_3d(ring, part ? &tmH : &tmC, &full_bar, 0, step * B + b0, part ? j * ch : p.nkb_h + j * ch);
            }
            __syncwarp();
            ++prod_it;
        }
        rp[2 * part] += t1 - t0; rp[2 * part + 1] += clock64() - t1;
    };
    // MMA issuer: acc (+)= W[:, kb] . act[:, kb]^T over the k-blocks of the part
    auto consume = [&](int part, bool signal_accum) {
        const long long t0 = clock64();
        long long t1 = t0;
        const int n = part ? p.n_h : (ALIAS ? p.n_c : 1), ch = part ? p.ch_h : p.ch_c;
        if (!ATT) {
            for (int j = 0; j < n; ++j) {
                mbar_wait(j ? &full2_bar : &full_bar, cons_it & 1);
                if (j == 0) t1 = clock64();
                tc_fence_after();
                if (elect_one()) {
                    for (int c = 0; c < ch; ++c) {
                        const uint64_t adesc = make_sw128_desc(smem_u32(sW + (size_t)(j * ch + c) * WTILE));
                        const uint64_t bdesc = make_sw128_desc(smem_u32(ring + (size_t)(j * ch + c) * ATILE));
#pragma unroll
                        for (int k = 0; k < KB / 16; ++k) umma_bf16(tmem_base, adesc + 2 * k, bdesc + 2 * k, idesc, (j == 0 && c == 0 && k == 0) ? 0u : 1u);
                    }
                    if (j == n - 1) umma_commit(&accum_bar);
                }
                __syncwarp();
            }
            ++cons_it;
            rp[2 * part] += t1 - t0; rp[2 * part + 1] += clock64() - t1;
            return;
        }
        for (int j = 0; j < n; ++j) {
            mbar_wait(&full_bar, cons_it & 1);
            if (j == 0) t1 = clock64();
            tc_fence_after();
            const int kb0 = part ? j * ch : p.nkb_h + j * ch;
            if (elect_one()) {
                for (int c = 0; c < ch; ++c) {
                    const uint64_t adesc = make_sw128_desc(smem_u32(sW + (size_t)(kb0 + c) * WTILE));
                    const uint64_t bdesc = make_sw128_desc(smem_u32(ring + (size_t)c * ATILE));
#pragma unroll
                    for (int k = 0; k < KB / 16; ++k)
                        umma_bf16(tmem_base, adesc + 2 * k, bdesc + 2 * k, idesc, (part == 1 && j == 0 && c == 0 && k == 0) ? 0u : 1u);
                }
                umma_commit(&empty_bar);
                if (signal_accum && j == n - 1) umma_commit(&accum_bar);
            }
            __syncwarp();
            ++cons_it;
        }
        rp[2 * part] += t1 - t0; rp[2 * part + 1] += clock64() - t1;
    };

    // B fragments (k = this CTA's 16 hidden units, n = attention dims of the n-tiles {2 warp, 2 warp + 1}) of the query projection,
    // split into bf16 hi + lo, resident in registers for the whole sequence
    uint32_t wqh[2][2] = {{0u, 0u}, {0u, 0u}}, wql[2][2] = {{0u, 0u}, {0u, 0u}};
    if (ATT && compute) {
        const int g = lane >> 2, tq = lane & 3;
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int r2 = 0; r2 < 2; ++r2) {
                const int a = (2 * warp + j) * 8 + g, u = u0 + 2 * tq + 8 * r2;
                const float x0 = (a < p.A && u < D) ? p.Wq[(size_t)a * D + u] : 0.f, x1 = (a < p.A && u + 1 < D) ? p.Wq[(size_t)a * D + u + 1] : 0.f;
                const __nv_bfloat16 h0 = __float2bfloat16_rn(x0), h1 = __float2bfloat16_rn(x1);
                __nv_bfloat162 hp2; hp2.x = h0; hp2.y = h1;
                wqh[j][r2] = *reinterpret_cast<uint32_t*>(&hp2);
                wql[j][r2] = pack2(x0 - __bfloat162float(h0), x1 - __bfloat162float(h1));
            }
    }
    const float inv_h = 1.f / (1.f - p.rate_h), inv_c = 1.f / (1.f - p.rate_c);
    unsigned target = 0;
    PROF_DECL

    // prologue: the h part of step 0 (operand row 0 is all zeros)
    if (is_producer) produce(0, 1);
    if (is_mma) consume(1, !ATT || p.nkb_h == p.nkb);
    __syncwarp();

    // Epilogue operands of this thread's two (b, u) pairs.  The input-projection gates and the keep masks of step i+1 are fetched
    // (from DRAM) right after the cell barrier of step i, i.e. a whole attention phase ahead; c and the regularised h are carried
    // in registers from step to step.
    float pre[2][6];
    uint8_t pm[2][2];
    auto prefetch = [&](int step, bool state) {
#pragma unroll
        for (int e2 = 0; e2 < 2; ++e2) {
            const int idx = tid + e2 * CT;
            const int bl = idx / UNITS, uu = idx % UNITS, b = b0 + bl, u = u0 + uu;
            pm[e2][0] = 1; pm[e2][1] = 1;
#pragma unroll
            for (int j = 0; j < 4; ++j) pre[e2][j] = 0.f;
            if (state) { pre[e2][4] = 0.f; pre[e2][5] = 0.f; }
            if (b < B && u < D) {
                const size_t g0 = ((size_t)step * B + b) * 4 * D + u, mi = ((size_t)step * B + b) * D + u;
                pre[e2][0] = p.gates[g0]; pre[e2][1] = p.gates[g0 + D]; pre[e2][2] = p.gates[g0 + 2 * D]; pre[e2][3] = p.gates[g0 + 3 * D];
                if (state) {
                    pre[e2][4] = p.cstate[mi];
                    pre[e2][5] = p.actf[((size_t)step * B + b) * p.ldf + p.hcol + u];
                }
                if (p.training && p.mask_h) pm[e2][0] = p.mask_h[mi];
                if (p.training && p.mask_c) pm[e2][1] = p.mask_c[mi];
            }
        }
    };
    // DRAM -> L2 two steps ahead, so that the register prefetch above is an L2 hit (the load-return path is in order: a DRAM-latency
    // load in front of the attention's L2 loads would stall them)
    auto prefetch_l2 = [&](int step) {
        if (step >= p.T) return;
#pragma unroll
        for (int e2 = 0; e2 < 2; ++e2) {
            const int idx = tid + e2 * CT;
            const int bl = idx / UNITS, uu = idx % UNITS, b = b0 + bl, u = u0 + uu;
            if (b < B && u < D && (uu & 7) == 0) {
                const size_t g0 = ((size_t)step * B + b) * 4 * D + u, mi = ((size_t)step * B + b) * D + u;
                l2_prefetch(p.gates + g0); l2_prefetch(p.gates + g0 + D); l2_prefetch(p.gates + g0 + 2 * D); l2_prefetch(p.gates + g0 + 3 * D);
                if (uu == 0 && p.training && p.mask_h) l2_prefetch(p.mask_h + mi);
                if (uu == 0 && p.training && p.mask_c) l2_prefetch(p.mask_c + mi);
            }
        }
    };
    if (compute) { prefetch_l2(0); prefetch(0, true); prefetch_l2(1); }

    int att_len = 0;               // ATT: clamped text length of the utterance this CTA pair serves
    if (ATT && (cta >> 1) < B) { const int l0 = p.lengths[cta >> 1]; att_len = l0 < 0 ? 0 : (l0 > p.L ? p.L : l0); }
    bool alive = true;
    for (int i = 0; i < p.T && alive; ++i) {
        // =================== ctx part of the gate product (the context of step i-1 is visible now) ===================
        if (ATT && p.nkb_h < p.nkb) {
            if (is_producer) produce(i, 0);
            if (is_mma) consume(0, true);
            __syncwarp();
        }
        if (compute) {
            // accumulator [64 gate rows x 32 utterances]: TMEM lane 32 * gate + unit, column = utterance
            mbar_wait(&accum_bar, i & 1);
            tc_fence_after();
            {
                const int q = warp & 3, c0 = (warp >> 2) * 16;
                uint32_t r[16];
                tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c0, r);
                if (lane < UNITS) {
#pragma unroll
                    for (int j = 0; j < 16; ++j) s_sum[(c0 + j) * (ROWS + 1) + q * UNITS + lane] = __uint_as_float(r[j]);
                }
            }
            tc_fence_before();
            csync();
            PROF_MARK(0);
            // =================== LSTM cell + regulariser (2 (b, u) pairs per thread) ===================
#pragma unroll
            for (int e2 = 0; e2 < 2; ++e2) {
                const int idx = tid + e2 * CT;
                const int bl = idx / UNITS, uu = idx % UNITS, b = b0 + bl, u = u0 + uu;
                float hs = 0.f;
                if (b < B && u < D) {
                    const size_t g0 = ((size_t)i * B + b) * 4 * D + u;
                    const float zi = pre[e2][0] + s_sum[bl * (ROWS + 1) + uu];
                    const float zf = pre[e2][1] + s_sum[bl * (ROWS + 1) + UNITS + uu];
                    const float zg = pre[e2][2] + s_sum[bl * (ROWS + 1) + 2 * UNITS + uu];
                    const float zo = pre[e2][3] + s_sum[bl * (ROWS + 1) + 3 * UNITS + uu];
                    const float gi = sigmoid_fast(zi), gf = sigmoid_fast(zf), gg = tanh_exp(zg), go = sigmoid_fast(zo);
                    const size_t bu = (size_t)b * D + u;
                    const float cp = pre[e2][4];
                    float cn = gf * cp + gi * gg;
                    float hn = go * tanh_exp(cn);
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
                    p.actb[((size_t)(i + 1) * B + b) * Kp + u] = __float2bfloat16_rn(hn);
                    hs = hn;
                    pre[e2][4] = cn; pre[e2][5] = hn;           // state of the next step
                }
                if (ATT) s_hs[uu * (BT + 4) + bl] = hs;
            }
            if (ATT) {
                csync();
                // partial query projection of this CTA's 16 hidden units on the tensor cores: qpart[rb, b, a] = sum_u h[b, u] Wq[a, u].
                // h and Wq are split into bf16 hi + lo and three products are summed (hi.hi + lo.hi + hi.lo), i.e. fp32-equivalent.
                {
                    const int g = lane >> 2, tq = lane & 3;
                    uint32_t ah[2][4], al[2][4];
#pragma unroll
                    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
                        for (int r4 = 0; r4 < 4; ++r4) {
                            const int bl = mt * 16 + g + 8 * (r4 & 1), k = 2 * tq + 8 * (r4 >> 1);
                            const float x0 = s_hs[k * (BT + 4) + bl], x1 = s_hs[(k + 1) * (BT + 4) + bl];
                            const __nv_bfloat16 h0 = __float2bfloat16_rn(x0), h1 = __float2bfloat16_rn(x1);
                            __nv_bfloat162 hp2; hp2.x = h0; hp2.y = h1;
                            ah[mt][r4] = *reinterpret_cast<uint32_t*>(&hp2);
                            al[mt][r4] = pack2(x0 - __bfloat162float(h0), x1 - __bfloat162float(h1));
                        }
#pragma unroll
                    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
                        for (int j = 0; j < 2; ++j) {
                            float acc[4] = {0.f, 0.f, 0.f, 0.f};
                            mma_bf16(acc, ah[mt], wqh[j][0], wqh[j][1]);
                            mma_bf16(acc, al[mt], wqh[j][0], wqh[j][1]);
                            mma_bf16(acc, ah[mt], wql[j][0], wql[j][1]);
                            const int a = (2 * warp + j) * 8 + 2 * tq;
                            const int bA = b0 + mt * 16 + g, bB = bA + 8;
                            if (bA < B) *reinterpret_cast<float2*>(p.qpart + ((size_t)rb * B + bA) * p.A + a) = make_float2(acc[0], acc[1]);
                            if (bB < B) *reinterpret_cast<float2*>(p.qpart + ((size_t)rb * B + bB) * p.A + a) = make_float2(acc[2], acc[3]);
                        }
                }
            }
        }
        PROF_MARK(1);
        if (ALIAS) proxy_fence_shared();             // generic-proxy accesses of the staging precede the TMA writes that follow the barrier
        if (!grid_barrier<true>(bar_counter, target, nblocks, p.abort_flag, &s_ok)) { alive = false; break; }
        PROF_MARK(2);

        // =================== h part of step i+1: TMA + tcgen05 run while the attention of step i is computed ===================
        if (i + 1 < p.T) {
            if (is_producer) produce(i + 1, 1);
            if (is_mma) { tc_fence_after(); consume(1, !ATT || p.nkb_h == p.nkb); }
            __syncwarp();
            if (compute) { prefetch_l2(i + 2); if (!ATT) prefetch(i + 1, false); }
        }

        if (ATT) {
            // =================== attention: one CTA PAIR (cluster of 2) per utterance ===================
            // pair pc = cta >> 1 serves utterance pc; rank hf = cta & 1 owns the attention dims [64 hf, 64 hf + 64) of the energies
            // (partial sums exchanged through distributed shared memory, one cluster barrier) and one half of the context tiles.
            const int pc = cta >> 1, hf = cta & 1;
            if (compute && pc < B) {
                const int b = pc, L = p.L, A = p.A, AH = p.A / 2, M = p.M, half = (p.KC - 1) / 2, L16 = p.MT * 16;
                float* qb = scratch;                       // [AH]  query + bias of this rank's attention dims
                float* vv = qb + AH;                       // [AH]  persistent: energy vector
                float* bias_s = vv + AH;                   // [AH]  persistent: attention bias
                float* cum_s = bias_s + AH;                // [L16] persistent: cumulative attention weights of this utterance
                float* e = cum_s + L16;                    // [L16] energies -> weights
                float* eq = e + L16;                       // [2][L16] quarter-job partial energies
                float* epart = eq + 2 * L16;               // [2][L16] per-rank partial energies (slot 1 - hf is written by the peer CTA)
                float* red = epart + 2 * L16;              // [64]
                float* cred = red + 64;                    // [16][AH] query partials
                uint32_t* Ph = reinterpret_cast<uint32_t*>(cred + 16 * AH);   // [L16 + 48] Toeplitz pair arrays (hi / lo bf16 split)
                uint32_t* Pl = Ph + (L16 + 48);
                uint2* btab = reinterpret_cast<uint2*>(Pl + (L16 + 48));     // [MT][32] B fragments of the context product (p.use_btab)
                const int len = att_len;                   // text length of this pair's utterance (loaded once, before the loop)
                const int mtiles = (len + 15) / 16, ktiles = mtiles;
                if (i == 0) {                              // one-time: constants and the initial cumulative weights into shared memory
                    for (int a2 = tid; a2 < AH; a2 += CT) { vv[a2] = p.v[hf * AH + a2]; bias_s[a2] = p.bias[hf * AH + a2]; }
                    for (int l = tid; l < L16; l += CT) cum_s[l] = l < L ? p.cum[(size_t)b * L + l] : 0.f;
                    csync();
                }
                // memory-projection fragments of this warp's first energy job and memory fragments of its first context tile:
                // neither depends on this step's state, so they are requested first and land behind the query reduction
                constexpr int KTMAX = 12;                  // k-tiles (16 positions) per register batch of the context product
                const int mt_lo = hf * ((p.M16 + 1) / 2), mt_hi = min(p.M16, mt_lo + (p.M16 + 1) / 2);
                uint4 nraw[2];
                uint4 av[KTMAX];
                {   // q[a] = sum over the RB per-CTA partial projections: thread = (4 attention dims, one sixteenth of the row blocks)
                    const int a4 = tid & 15, sl = tid >> 4;
                    const int per = (p.RB + 15) / 16, r0 = sl * per, r1 = min(p.RB, r0 + per);
                    float4 qv[4];                 // first the loads the critical path waits for ...
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        qv[j] = (r0 + j < r1) ? __ldcg(reinterpret_cast<const float4*>(p.qpart + ((size_t)(r0 + j) * B + b) * A + hf * AH) + a4)
                                              : make_float4(0.f, 0.f, 0.f, 0.f);
                    // ... then (the load-return path is in order) the fragments that do not depend on this step's state: the memory projection
                    // of this warp's first energy job and the memory tile of its first context product
                    if (warp < 2 * mtiles) {
                        const uint4* mf = reinterpret_cast<const uint4*>(p.memTf + (((size_t)b * p.MT + (warp >> 1)) * 32 + lane) * 64) + hf * 4 + (warp & 1) * 2;
                        nraw[0] = __ldg(mf); nraw[1] = __ldg(mf + 1);
                    }
                    if (mt_lo + warp < mt_hi) {
                        const uint4* fr = p.memFf + (((size_t)b * p.M16 + mt_lo + warp) * p.MT) * 32 + lane;
#pragma unroll
                        for (int j = 0; j < KTMAX; ++j)
                            if (j < ktiles) av[j] = __ldg(fr + (size_t)j * 32);
                    }
                    // cumulative weights -> (hi, lo) bf16 pairs: Ph[x] = (c[x], c[x+1]) with c[j] = cum[j - half].  Pair-local state only: done here,
                    // while the query partials requested above are still on their way from L2
                    for (int x = tid; x < L16 + 48; x += CT) {
                        float c0 = 0.f, c1 = 0.f;
                        const int la = x - half, lb = x + 1 - half;
                        if (la >= 0 && la < L) c0 = cum_s[la];
                        if (lb >= 0 && lb < L) c1 = cum_s[lb];
                        const __nv_bfloat16 h0 = __float2bfloat16_rn(c0), h1 = __float2bfloat16_rn(c1);
                        __nv_bfloat162 hp2; hp2.x = h0; hp2.y = h1;
                        Ph[x] = *reinterpret_cast<uint32_t*>(&hp2);
                        Pl[x] = pack2(c0 - __bfloat162float(h0), c1 - __bfloat162float(h1));
                    }
                    float4 qs = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                    for (int j = 0; j < 4; ++j) { qs.x += qv[j].x; qs.y += qv[j].y; qs.z += qv[j].z; qs.w += qv[j].w; }
                    for (int r = r0 + 4; r < r1; r += 4) {          // more than 64 row blocks: further rounds
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            if (r + j < r1) {
                                const float4 v4 = __ldcg(reinterpret_cast<const float4*>(p.qpart + ((size_t)(r + j) * B + b) * A + hf * AH) + a4);
                                qs.x += v4.x; qs.y += v4.y; qs.z += v4.z; qs.w += v4.w;
                            }
                    }
                    *reinterpret_cast<float4*>(cred + sl * AH + a4 * 4) = qs;
                    csync();
                    for (int a2 = tid; a2 < AH; a2 += CT) {
                        float q = 0.f;
#pragma unroll
                        for (int sl2 = 0; sl2 < 16; ++sl2) q += cred[sl2 * AH + a2];
                        p.qsave[((size_t)i * B + b) * A + hf * AH + a2] = q;
                        qb[a2] = q + bias_s[a2];
                    }
                }
                csync();
                PROF_MARK(3);
                // energies on the tensor cores: S[l, a] = sum_k cumpad[l + k] * Wcomb[a, k].  job = (16-position tile, quarter of the
                // attention dims: 4 n-tiles of 8 within this rank's half) -> 2 mtiles jobs, 3 per warp for L = 180
                {
                    const int g = lane >> 2, tq = lane & 3;
                    for (int job = warp; job < 2 * mtiles; job += NCW) {
                        const int mt = job >> 1, qh = job & 1, l0 = mt * 16;
                        const uint4 raw[2] = {nraw[0], nraw[1]};
                        if (job + NCW < 2 * mtiles) {        // next job's fragments: in flight during this job's MMAs
                            const int nj = job + NCW;
                            const uint4* mf = reinterpret_cast<const uint4*>(p.memTf + (((size_t)b * p.MT + (nj >> 1)) * 32 + lane) * 64) + hf * 4 + (nj & 1) * 2;
                            nraw[0] = __ldg(mf); nraw[1] = __ldg(mf + 1);
                        }
                        float sacc[4][4];
#pragma unroll
                        for (int nt = 0; nt < 4; ++nt)
#pragma unroll
                            for (int e4 = 0; e4 < 4; ++e4) sacc[nt][e4] = 0.f;
#pragma unroll
                        for (int ks = 0; ks < 2; ++ks) {
                            const int x = l0 + ks * 16 + g + 2 * tq;
                            const uint32_t ah[4] = {Ph[x], Ph[x + 8], Ph[x + 8], Ph[x + 16]};
                            const uint32_t al[4] = {Pl[x], Pl[x + 8], Pl[x + 8], Pl[x + 16]};
#pragma unroll
                            for (int np = 0; np < 2; ++np) {
                                uint32_t bfr[4];
                                ldmatrix_x4(bfr[0], bfr[1], bfr[2], bfr[3],
                                            sWcB + (size_t)((qh * 2 + np) * 16 + (lane & 7) + ((lane >> 4) << 3)) * 40 + ks * 16 + ((lane >> 3) & 1) * 8);
                                mma_bf16(sacc[2 * np], ah, bfr[0], bfr[1]);
                                mma_bf16(sacc[2 * np], al, bfr[0], bfr[1]);
                                mma_bf16(sacc[2 * np + 1], ah, bfr[2], bfr[3]);
                                mma_bf16(sacc[2 * np + 1], al, bfr[2], bfr[3]);
                            }
                        }
                        float e0 = 0.f, e1 = 0.f;
#pragma unroll
                        for (int c4 = 0; c4 < 2; ++c4) {
                            const uint32_t words[4] = {raw[c4].x, raw[c4].y, raw[c4].z, raw[c4].w};
#pragma unroll
                            for (int h2 = 0; h2 < 2; ++h2) {
                                const int nt = 2 * c4 + h2, a0 = (qh * 4 + nt) * 8 + 2 * tq;      // index inside this rank's 64 dims
                                const float2 m01 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&words[2 * h2]));
                                const float2 m23 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&words[2 * h2 + 1]));
                                e0 = fmaf(vv[a0], tanh_fast(sacc[nt][0] + qb[a0] + m01.x), e0);
                                e0 = fmaf(vv[a0 + 1], tanh_fast(sacc[nt][1] + qb[a0 + 1] + m01.y), e0);
                                e1 = fmaf(vv[a0], tanh_fast(sacc[nt][2] + qb[a0] + m23.x), e1);
                                e1 = fmaf(vv[a0 + 1], tanh_fast(sacc[nt][3] + qb[a0 + 1] + m23.y), e1);
                            }
                        }
                        e0 += __shfl_xor_sync(0xffffffffu, e0, 1); e0 += __shfl_xor_sync(0xffffffffu, e0, 2);
                        e1 += __shfl_xor_sync(0xffffffffu, e1, 1); e1 += __shfl_xor_sync(0xffffffffu, e1, 2);
                        if (tq == 0) { eq[qh * L16 + l0 + g] = e0; eq[qh * L16 + l0 + g + 8] = e1; }
                    }
                }
                csync();
                // this rank's partial energies: own copy + the peer's copy through distributed shared memory.  Every remote store completes its
                // 4 bytes on the PEER's exchange mbarrier (st.async), which that CTA armed with the L16 * 4 bytes it expects: no cluster barrier
                if (tid == 0) mbar_expect_tx(&xchg_bar, (uint32_t)L16 * 4);
                for (int l = tid; l < L16; l += CT) {
                    const float v = l < mtiles * 16 ? eq[l] + eq[L16 + l] : 0.f;
                    epart[hf * L16 + l] = v;
                    st_async_peer_f32(epart + hf * L16 + l, &xchg_bar, (uint32_t)(hf ^ 1), v);
                }
                csync();                                   // own copies visible to the whole CTA
                mbar_wait(&xchg_bar, i & 1);               // the peer's L16 values have landed (acquire)
                PROF_MARK(4);
                float mx = -INFINITY;
                for (int l = tid; l < len; l += CT) { const float ev = epart[l] + epart[L16 + l]; e[l] = ev; mx = fmaxf(mx, ev); }
                mx = cblock_max(mx, red);
                float sum = 0.f;
                for (int l = tid; l < len; l += CT) { const float ex = expf(e[l] - mx); e[l] = ex; sum += ex; }
                sum = cblock_sum(sum, red + 32);
                float* cum_next = p.cum + ((size_t)(i + 1) * B + b) * L;
                const float inv_sum = 1.f / sum;
                for (int l = tid; l < L16; l += CT) {       // the padded tail must be zero: the context MMA reads whole 16-position tiles
                    const float w = l < len ? e[l] * inv_sum : 0.f;
                    e[l] = w;
                    if (l < L) {
                        const float cn = cum_s[l] + w;
                        cum_s[l] = cn;                      // both ranks keep the full cumulative weights; the global stores are shared out
                        if (hf == 0) p.align[(size_t)b * p.align_bstride + (size_t)i * L + l] = w;
                        else cum_next[l] = cn;
                    }
                }
                csync();
                if (p.use_btab) {
                    // B fragments (hi(w) in column 0, lo(w) in column 1) of every 16-position k-tile, built ONCE per CTA: they depend on the k-tile
                    // only, and every warp used to rebuild all of them (~40 instructions per fragment and warp)
                    for (int idx = tid; idx < ktiles * 32; idx += CT) {
                        const int kt = idx >> 5, gg = (idx >> 2) & 7, tt = idx & 3;
                        uint2 f = make_uint2(0u, 0u);
                        if (gg < 2) {
                            const float* wl = e + kt * 16 + 2 * tt;
                            const float w0 = wl[0], w1 = wl[1], w2 = wl[8], w3 = wl[9];
                            const float h0 = __bfloat162float(__float2bfloat16_rn(w0)), h1 = __bfloat162float(__float2bfloat16_rn(w1));
                            const float h2 = __bfloat162float(__float2bfloat16_rn(w2)), h3 = __bfloat162float(__float2bfloat16_rn(w3));
                            f = gg == 0 ? make_uint2(pack2(h0, h1), pack2(h2, h3)) : make_uint2(pack2(w0 - h0, w1 - h1), pack2(w2 - h2, w3 - h3));
                        }
                        btab[idx] = f;
                    }
                    csync();
                }
                PROF_MARK(5);
                // context on the tensor cores: ctx[m] = sum_l memory[l, m] * w[l] for this rank's half of the 16-row tiles.  A = memory^T
                // fragments (fragment-major bf16, one 16-byte load per lane per MMA), B = (hi(w), lo(w)) in columns 0 / 1, so that
                // column 0 + column 1 of D is the fp32-weighted sum.
                {
                    const int g = lane >> 2, tq = lane & 3;
                    uint32_t bfr[KTMAX][2];                // B fragments: lanes g = 0 hold hi(w), g = 1 hold lo(w), other columns zero
                    auto build_b = [&](int kt0) {
                        if (p.use_btab) {
#pragma unroll
                            for (int j = 0; j < KTMAX; ++j) {
                                bfr[j][0] = 0u; bfr[j][1] = 0u;
                                if (kt0 + j < ktiles) { const uint2 f = btab[(kt0 + j) * 32 + lane]; bfr[j][0] = f.x; bfr[j][1] = f.y; }
                            }
                            return;
                        }
#pragma unroll
                        for (int j = 0; j < KTMAX; ++j) {
                            bfr[j][0] = 0u; bfr[j][1] = 0u;
                            if (kt0 + j < ktiles) {
                                const float* wl = e + (kt0 + j) * 16 + 2 * tq;
                                const float w0 = wl[0], w1 = wl[1], w2 = wl[8], w3 = wl[9];
                                const float h0 = __bfloat162float(__float2bfloat16_rn(w0)), h1 = __bfloat162float(__float2bfloat16_rn(w1));
                                const float h2 = __bfloat162float(__float2bfloat16_rn(w2)), h3 = __bfloat162float(__float2bfloat16_rn(w3));
                                const float s0 = g == 0 ? h0 : (g == 1 ? w0 - h0 : 0.f), s1 = g == 0 ? h1 : (g == 1 ? w1 - h1 : 0.f);
                                const float s2 = g == 0 ? h2 : (g == 1 ? w2 - h2 : 0.f), s3 = g == 0 ? h3 : (g == 1 ? w3 - h3 : 0.f);
                                bfr[j][0] = pack2(s0, s1); bfr[j][1] = pack2(s2, s3);
                            }
                        }
                    };
                    const bool single = ktiles <= KTMAX;
                    if (single) build_b(0);
                    for (int mt = mt_lo + warp; mt < mt_hi; mt += NCW) {
                        float dacc[4] = {0.f, 0.f, 0.f, 0.f}, dacc2[4] = {0.f, 0.f, 0.f, 0.f};
                        for (int kt0 = 0; kt0 < ktiles; kt0 += KTMAX) {
                            if (kt0 > 0 || mt != mt_lo + warp) {      // everything but the prefetched first batch
                                const uint4* fr = p.memFf + (((size_t)b * p.M16 + mt) * p.MT) * 32 + lane;
#pragma unroll
                                for (int j = 0; j < KTMAX; ++j)
                                    if (kt0 + j < ktiles) av[j] = __ldg(fr + (size_t)(kt0 + j) * 32);
                            }
                            if (!single) build_b(kt0);
#pragma unroll
                            for (int j = 0; j < KTMAX; j += 2) {   // two independent accumulation chains
                                if (kt0 + j < ktiles) {
                                    const uint32_t af[4] = {av[j].x, av[j].y, av[j].z, av[j].w};
                                    mma_bf16(dacc, af, bfr[j][0], bfr[j][1]);
                                }
                                if (kt0 + j + 1 < ktiles) {
                                    const uint32_t af[4] = {av[j + 1].x, av[j + 1].y, av[j + 1].z, av[j + 1].w};
                                    mma_bf16(dacc2, af, bfr[j + 1][0], bfr[j + 1][1]);
                                }
                            }
                        }
                        if (tq == 0) {
                            const int m0 = mt * 16 + g;
                            const float c0 = (dacc[0] + dacc2[0]) + (dacc[1] + dacc2[1]), c1 = (dacc[2] + dacc2[2]) + (dacc[3] + dacc2[3]);
                            if (m0 < M) {
                                p.actf[((size_t)(i + 1) * B + b) * p.ldf + m0] = c0;
                                p.actb[((size_t)(i + 1) * B + b) * Kp + D + m0] = __float2bfloat16_rn(c0);
                            }
                            if (m0 + 8 < M) {
                                p.actf[((size_t)(i + 1) * B + b) * p.ldf + m0 + 8] = c1;
                                p.actb[((size_t)(i + 1) * B + b) * Kp + D + m0 + 8] = __float2bfloat16_rn(c1);
                            }
                        }
                    }
                }
            }
            PROF_MARK(6);
            // next step's epilogue operands (L2 hits: prefetched a step ago) are requested between the arrival and the wait
            if (!grid_barrier<true>(bar_counter, target, nblocks, p.abort_flag, &s_ok, [&]() { if (compute && i + 1 < p.T) prefetch(i + 1, false); })) {
                alive = false; break;
            }
            PROF_MARK(7);
        }
    }
    PROF_FLUSH;
    if (p.prof2 && (is_mma || is_producer) && lane == 0)
        for (int k = 0; k < 4; ++k) p.prof2[(size_t)cta * 8 + (is_producer ? 4 : 0) + k] = rp[k];
    tc_fence_before();
    __syncthreads();
    if (warp == NCW + 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS));
    }
}

// shared memory of one loop CTA with a ring slot of slot_kb k-blocks; alias: the accumulator staging shares the slot
size_t tc_loop_smem_bytes(int nkb, int slot_kb, int A, bool att, int L, bool alias = false) {
    const size_t ring_b = (size_t)slot_kb * ATILE, sum_b = (size_t)BT * (ROWS + 1) * 4;
    size_t b = 1024 + (size_t)nkb * WTILE + (alias ? (ring_b > sum_b ? ring_b : sum_b) : ring_b + sum_b);
    if (att) {
        const int L16 = (L + 15) / 16 * 16;
        b += (size_t)UNITS * (BT + 4) * 4 + (size_t)(A / 2) * 40 * 2;
        b += ((size_t)3 * (A / 2) + 6 * L16 + 64 + 16 * (A / 2) + 2 * (L16 + 48)) * 4;
    }
    return b;
}
constexpr size_t SMEM_LIMIT = 227 * 1024 - 1088;    // leave room for the static barriers (1 KB of static shared memory)

// largest ring slot (in k-blocks, <= want) that fits
int pick_slot(int nkb, int A, bool att, int L, int want, bool alias = false) {
    int kb = want;
    while (kb >= 1 && tc_loop_smem_bytes(nkb, kb, A, att, L, alias) > SMEM_LIMIT) --kb;
    return kb;
}
int largest_divisor_le(int n, int cap) {
    for (int d = cap < n ? cap : n; d >= 1; --d)
        if (n % d == 0) return d;
    return 1;
}

}  // namespace

// column geometry of the bf16 operand rows of the tcgen05 loops: [h (D) | ctx (M) | zero pad], 64-column k-blocks
TcPersistGeom tc_persist_geom(const b200tts_decoder_shape& s) {
    TcPersistGeom g{};
    g.nkb_att = (s.D + s.M + KB - 1) / KB;
    g.nkb_gen = (s.D + KB - 1) / KB;
    g.nkb_h = s.D / KB;
    g.Kp_att = g.nkb_att * KB;
    g.Kp_gen = g.nkb_gen * KB;
    const int nkb_c = g.nkb_att - g.nkb_h;
    g.alias_att = 0;
    g.slot_att = pick_slot(g.nkb_att, s.A, true, s.L, g.nkb_h);
    if (g.slot_att < nkb_c) {           // large memory dims (M = 512: 192 KB of resident weights): the accumulator staging moves into the slot
        g.alias_att = 1;                // and the ctx part arrives in several TMA instructions
        g.slot_att = pick_slot(g.nkb_att, s.A, true, s.L, g.nkb_h, true);
    }
    g.ch_c_att = g.slot_att >= 1 ? largest_divisor_le(nkb_c, g.slot_att) : 0;
    g.n_c_att = g.ch_c_att >= 1 ? nkb_c / g.ch_c_att : 0;
    g.ch_h_att = g.slot_att >= 1 ? largest_divisor_le(g.nkb_h, g.slot_att) : 0;
    g.slot_gen = pick_slot(g.nkb_gen, s.A, false, 0, g.nkb_gen);
    g.ch_h_gen = g.slot_gen >= 1 ? largest_divisor_le(g.nkb_gen, g.slot_gen) : 0;
    // the generator loop requests its operand in (at most) two chunks with separate barriers; it needs the whole operand in the ring
    if (g.slot_gen >= g.nkb_gen && g.nkb_gen % 2 == 0) g.ch_h_gen = g.nkb_gen / 2;
    return g;
}

bool tc_persist_supported(const b200tts_decoder_shape& s) {
    if (s.D % KB != 0 || s.D % UNITS != 0) return false;
    const int RB = s.D / UNITS, NBH = (s.B + BT - 1) / BT;
    if (RB * NBH > 148 || s.B > RB * NBH) return false;
    if (s.K > 32 || s.A != 128) return false;
    const TcPersistGeom g = tc_persist_geom(s);
    return g.ch_c_att >= 1 && g.ch_c_att <= 256 && g.slot_att >= g.ch_c_att && g.ch_h_att >= 1 && g.ch_h_gen >= 1 && g.slot_att >= 2 &&
           g.slot_gen >= g.nkb_gen;          // generator loop: the whole operand row block is ring resident
}

static int launch_tc_loop(bool att, const TcLoopArgs& a, const CUtensorMap& tmH, const CUtensorMap& tmC, size_t smem, cudaStream_t st) {
    void* fn = att ? (a.alias_sum ? (void*)lstm_loop_tc_kernel<true, true> : (void*)lstm_loop_tc_kernel<true, false>) : (void*)lstm_loop_tc_kernel<false, false>;
    const int grid = a.RB * a.NBH;
    TcLoopArgs args = a;
    CUtensorMap mapH = tmH, mapC = tmC;
    void* params[] = {&mapH, &mapC, &args};
    if (att) {      // the attention runs on CTA pairs: clusters of 2 (distributed shared memory + cluster barrier)
        B200_REQUIRE(grid % 2 == 0 && grid / 2 >= a.B, "tcgen05 attention loop: %d CTAs cannot form %d pairs", grid, a.B);
        return launch_persistent(fn, grid, PT, smem, params, st, "tcgen05 attention loop", "lstm_loop_tc_kernel<att>", 2, true);
    }
    return launch_persistent(fn, grid, PT, smem, params, st, "tcgen05 persistent loop", "lstm_loop_tc_kernel<gen>", 1, true);
}

// Attention-LSTM + attention loop (all T steps).  Expects: ga = input projection, ai row 0 = 0, ca row 0 = 0, cum row 0 = 0,
// and the attention operands (wcb, memTf, memFf) already prepared in the persistent workspace.
int tc_persist_att_loop(const b200tts_decoder_shape& s, const b200tts_decoder_params& w, const b200tts_decoder_inputs& in,
                        const DecoderLayout& fl, float* ws, unsigned char* pws, float* align, cudaStream_t st) {
    const PersistLayout l = persist_layout(s);
    const TcPersistGeom g = tc_persist_geom(s);
    const int B = s.B, T = s.T, D = s.D, M = s.M, MD = M + D;
    __nv_bfloat16* aib = reinterpret_cast<__nv_bfloat16*>(pws + l.aib);
    // operand of step 0 and the zero padding columns [MD, Kp)
    B200_CUDA(cudaMemsetAsync(aib, 0, (size_t)(g.Kp_att != MD ? (size_t)(T + 1) : 1) * B * g.Kp_att * 2, st));   // step 0 + padding
    CUtensorMap tmH, tmC;       // {64 columns, rows, k-block}: k-block stride 128 B, row stride Kp * 2 B
    B200_TRY(tc_make_map3_bf16(&tmH, aib, KB, (T + 1) * B, g.nkb_att, (size_t)g.Kp_att * 2, 128, KB, BT, g.ch_h_att));
    B200_TRY(tc_make_map3_bf16(&tmC, aib, KB, (T + 1) * B, g.nkb_att, (size_t)g.Kp_att * 2, 128, KB, BT, g.ch_c_att));
    TcLoopArgs a{};
    a.B = B; a.T = T; a.D = D; a.K = MD; a.Kp = g.Kp_att; a.RB = D / UNITS; a.NBH = (B + BT - 1) / BT;
    a.nkb = g.nkb_att; a.nkb_h = g.nkb_h; a.ch_h = g.ch_h_att; a.n_h = g.nkb_h / g.ch_h_att; a.ch_c = g.ch_c_att; a.n_c = g.n_c_att;
    a.alias_sum = g.alias_att;
    a.slot_kb = g.ch_h_att > g.ch_c_att ? g.ch_h_att : g.ch_c_att;
    a.W = ws + fl.wcat_att; a.ldw = MD; a.wcol_h = M; a.wcol_c = 0;
    a.actb = aib; a.actf = ws + fl.ai; a.ldf = MD; a.hcol = M;
    a.gates = ws + fl.ga; a.cstate = ws + fl.ca;
    a.mask_h = in.mask_att_h; a.mask_c = in.mask_att_c; a.kind = s.cell_kind; a.training = s.training; a.rate_h = s.rate_h; a.rate_c = s.rate_c;
    a.L = s.L; a.M = M; a.A = s.A; a.KC = s.K;
    a.Wq = w.attn_query; a.qpart = ws + fl.qpart; a.qsave = ws + fl.q;
    a.WcB = reinterpret_cast<const __nv_bfloat16*>(pws + l.wcb);
    a.memTf = reinterpret_cast<const __nv_bfloat16*>(pws + l.memTf); a.MT = l.MT;
    a.bias = w.attn_bias; a.v = w.attn_energy;
    a.memFf = reinterpret_cast<const uint4*>(pws + l.memFf); a.M16 = l.M16;
    a.lengths = in.text_lengths; a.cum = ws + fl.cum;
    a.align = align; a.align_bstride = (long long)T * s.L;
    B200_TRY(reset_grid_barrier(pws + l.barrier, a, st));
    a.prof2 = a.prof + 2 * 148 * 8;
    size_t smem = tc_loop_smem_bytes(g.nkb_att, a.slot_kb, s.A, true, s.L, g.alias_att != 0);
    const size_t tab = (size_t)l.MT * 32 * 8;          // shared B-fragment table of the context product, when it fits behind the scratch
    a.use_btab = (smem + tab <= SMEM_LIMIT && !getenv("B200TTS_NO_BTAB")) ? 1 : 0;
    if (a.use_btab) smem += tab;
    return launch_tc_loop(true, a, tmH, tmC, smem, st);
}

// Generator-LSTM loop.  Expects: gg = input projection, hg row 0 = 0, cg row 0 = 0.
int tc_persist_gen_loop(const b200tts_decoder_shape& s, const b200tts_decoder_params& w, const b200tts_decoder_inputs& in,
                        const DecoderLayout& fl, float* ws, unsigned char* pws, cudaStream_t st) {
    const PersistLayout l = persist_layout(s);
    const TcPersistGeom g = tc_persist_geom(s);
    const int B = s.B, T = s.T, D = s.D;
    __nv_bfloat16* hgb = reinterpret_cast<__nv_bfloat16*>(pws + l.hgb);
    B200_CUDA(cudaMemsetAsync(hgb, 0, (size_t)(g.Kp_gen != D ? (size_t)(T + 1) : 1) * B * g.Kp_gen * 2, st));
    CUtensorMap tmH;
    B200_TRY(tc_make_map3_bf16(&tmH, hgb, KB, (T + 1) * B, g.nkb_gen, (size_t)g.Kp_gen * 2, 128, KB, BT, g.ch_h_gen));
    TcLoopArgs a{};
    a.B = B; a.T = T; a.D = D; a.K = D; a.Kp = g.Kp_gen; a.RB = D / UNITS; a.NBH = (B + BT - 1) / BT;
    a.nkb = g.nkb_gen; a.nkb_h = g.nkb_gen; a.ch_h = g.ch_h_gen; a.n_h = g.nkb_gen / g.ch_h_gen; a.ch_c = 0; a.n_c = 0; a.alias_sum = 0; a.use_btab = 0; a.slot_kb = g.nkb_gen;
    a.W = w.gen_w_hh; a.ldw = D; a.wcol_h = 0; a.wcol_c = 0;
    a.actb = hgb; a.actf = ws + fl.hg; a.ldf = D; a.hcol = 0;
    a.gates = ws + fl.gg; a.cstate = ws + fl.cg;
    a.mask_h = in.mask_gen_h; a.mask_c = in.mask_gen_c; a.kind = s.cell_kind; a.training = s.training; a.rate_h = s.rate_h; a.rate_c = s.rate_c;
    B200_TRY(reset_grid_barrier(pws + l.barrier, a, st));
    a.prof += 148 * 8;
    a.prof2 = a.prof + 2 * 148 * 8;
    return launch_tc_loop(false, a, tmH, tmH, tc_loop_smem_bytes(g.nkb_gen, a.slot_kb, s.A, false, 0), st);
}

}  // namespace b200tts
