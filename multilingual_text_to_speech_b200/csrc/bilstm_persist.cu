// Persistent packed bidirectional LSTM of the vanilla encoder (reference modules/encoder.py:33,41-44: nn.LSTM over a
// pack_padded_sequence; SURVEY.md K7).  ONE launch runs all L steps of both directions, forward or backward pass.
//
// Decomposition (thread-block clusters + distributed shared memory, no grid barrier, no cooperative launch):
//   * a CLUSTER of CS = H / 32 CTAs serves (direction, group of 8 utterances); CTA rank r owns hidden units [32 r, 32 r + 32):
//     its 128 gate rows of W_hh (forward) / its 32 columns of W_hh (backward) stay in shared memory in fp32 for the whole
//     sequence (H = 256: 130 KB) -- exact fp32 FFMA products in both precision modes;
//   * per step every CTA needs the whole previous hidden state (forward) / the whole gate gradient (backward) of its 8
//     utterances: each CTA stores its slice straight into the shared memory of all CS peers (st.shared::cluster) and ONE
//     cluster barrier (arrive.release / wait.acquire, a few hundred cycles instead of a 2.4 k-cycle grid barrier) publishes it;
//     the exchange buffers are double-buffered, so one barrier per step suffices;
//   * utterances shard over clusters, directions run concurrently: B = 64, H = 256 -> 2 x 8 clusters x 8 CTAs = 128 CTAs.
// Packed-sequence semantics as in rnn.cu: the state of utterance b is frozen and its output zero at positions >= lengths[b]
// (the reverse direction thereby starts at each utterance's own last token); a group whose 8 utterances are all frozen skips
// the product.  Saved tensors (activated gates, hs, cs) keep the layout of the per-step chain, which remains the fallback for
// shapes this kernel does not take (H % 32 != 0 or H > 256).
#include "decoder_internal.cuh"
#include "ptx.cuh"

namespace b200tts {

namespace {

constexpr int RU = 32;             // hidden units per CTA
constexpr int RROWS = 4 * RU;      // gate rows per CTA
constexpr int RBG = 8;             // utterances per cluster
constexpr int RT = 256;            // threads per CTA

struct BiLoopArgs {
    int B, L, H, CS, NG;
    const float* w_hh0; const float* w_hh1;   // [4H, H] per direction
    float* gates;                  // [2][L][B][4H] forward: in = input projection (+ biases), out = activated gates (valid steps)
    float* hs; float* cs;          // [2][L + 1][B][H]
    float* out;                    // forward: [B, L, 2H]
    const float* dout;             // backward: [B, L, 2H]
    float* dg;                     // backward: [2][L][B][4H] pre-activation gate gradients (zero at frozen steps)
    const int* lengths;
};

using namespace tcx;

// ------------------------------------------------------------------------------------------------
// forward: z[b, row] = sum_k h_prev[b, k] W_hh[row, k]; thread = (gate row, 4 utterances) for the product, (utterance, unit) for the cell
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(RT, 1) bilstm_fwd_loop_kernel(const BiLoopArgs p) {
    extern __shared__ __align__(16) float smf[];
    const int H = p.H, B = p.B, L = p.L, CS = p.CS, WLD = H + 4;
    float* Ws = smf;                                   // [RROWS][WLD]
    float* hbuf = Ws + (size_t)RROWS * WLD;            // [2][RBG][H]
    float* zs = hbuf + (size_t)2 * RBG * H;            // [RBG][RROWS]
    __shared__ int s_len[RBG];
    const int tid = threadIdx.x;
    const int rank = blockIdx.x % CS, grp = (blockIdx.x / CS) % p.NG, dir = blockIdx.x / (CS * p.NG);
    const int u0 = rank * RU, bg0 = grp * RBG;
    const float* W = dir ? p.w_hh1 : p.w_hh0;
    for (int idx = tid; idx < RROWS * H; idx += RT) {
        const int r = idx / H, k = idx % H;
        Ws[r * WLD + k] = W[(size_t)((r >> 5) * H + u0 + (r & 31)) * H + k];
    }
    for (int idx = tid; idx < 2 * RBG * H; idx += RT) hbuf[idx] = 0.f;
    if (tid < RBG) { const int b = bg0 + tid; int l = b < B ? p.lengths[b] : 0; s_len[tid] = l < 0 ? 0 : (l > L ? L : l); }
    __syncthreads();
    int gmax = 0;
#pragma unroll
    for (int j = 0; j < RBG; ++j) gmax = max(gmax, s_len[j]);
    // cell role
    const int cb = tid >> 5, cu = tid & 31, bglob = bg0 + cb, u = u0 + cu;
    const bool cvalid_b = bglob < B;
    const int clen = s_len[cb];
    float c_reg = 0.f, h_reg = 0.f;
    // product role
    const int prow = tid & (RROWS - 1), pb0 = (tid >> 7) * 4;
    const size_t dirBH = (size_t)dir * (L + 1) * B * H, dirG = (size_t)dir * L * B * 4 * H;
    if (cvalid_b) { p.hs[dirBH + (size_t)bglob * H + u] = 0.f; p.cs[dirBH + (size_t)bglob * H + u] = 0.f; }
    cluster_arrive(); cluster_wait();    // peers' exchange buffers are initialised before anyone stores into them
    for (int j = 0; j < L; ++j) {
        const int t = dir ? L - 1 - j : j;
        const int cur = j & 1, nxt = cur ^ 1;
        const bool any = t < gmax;
        const bool valid = cvalid_b && t < clen;
        float xp[4] = {0.f, 0.f, 0.f, 0.f};
        const size_t g0 = dirG + ((size_t)j * B + bglob) * 4 * H + u;
        if (valid) {
#pragma unroll
            for (int g = 0; g < 4; ++g) xp[g] = p.gates[g0 + (size_t)g * H];      // (rewritten below: no read-only path)
        }
        if (any) {
            float acc[4] = {0.f, 0.f, 0.f, 0.f};
            const float* wr = Ws + prow * WLD;
            const float* hb = hbuf + (size_t)cur * RBG * H + (size_t)pb0 * H;
#pragma unroll 4
            for (int k = 0; k < H; k += 4) {
                const float4 w4 = *reinterpret_cast<const float4*>(wr + k);
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const float4 h4 = *reinterpret_cast<const float4*>(hb + q * H + k);
                    acc[q] = fmaf(w4.x, h4.x, acc[q]); acc[q] = fmaf(w4.y, h4.y, acc[q]);
                    acc[q] = fmaf(w4.z, h4.z, acc[q]); acc[q] = fmaf(w4.w, h4.w, acc[q]);
                }
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) zs[(pb0 + q) * RROWS + prow] = acc[q];
            __syncthreads();
        }
        float hn = h_reg, cn = c_reg, y = 0.f;
        if (valid) {
            const float zi = xp[0] + zs[cb * RROWS + cu], zf = xp[1] + zs[cb * RROWS + RU + cu];
            const float zg = xp[2] + zs[cb * RROWS + 2 * RU + cu], zo = xp[3] + zs[cb * RROWS + 3 * RU + cu];
            const float gi = sigmoidf_acc(zi), gf = sigmoidf_acc(zf), gg = tanhf(zg), go = sigmoidf_acc(zo);
            cn = gf * c_reg + gi * gg;
            hn = go * tanhf(cn);
            y = hn;
            p.gates[g0] = gi; p.gates[g0 + H] = gf; p.gates[g0 + 2 * (size_t)H] = gg; p.gates[g0 + 3 * (size_t)H] = go;
        }
        if (cvalid_b) {
            const size_t so = dirBH + ((size_t)(j + 1) * B + bglob) * H + u;
            p.hs[so] = hn; p.cs[so] = cn;
            p.out[((size_t)bglob * L + t) * 2 * H + (size_t)dir * H + u] = y;
        }
        c_reg = cn; h_reg = hn;
        if (any) {                 // publish this CTA's slice of the new hidden state to every CTA of the cluster
            const uint32_t offb = (uint32_t)(((size_t)nxt * RBG * H + (size_t)cb * H + u) * 4);
            for (int r = 0; r < CS; ++r) st_cluster_f32(peer_addr(hbuf, (uint32_t)r) + offb, hn);
            cluster_arrive(); cluster_wait();
        }
        // else: the whole group is frozen at this position.  Along a direction's processing order that happens only BEFORE the first valid
        // step (reverse direction: the state is still the zero initial state, which both exchange buffers hold) or AFTER the last one
        // (forward direction: nobody reads the buffers again), so neither a store nor a barrier is needed.
    }
}

// ------------------------------------------------------------------------------------------------
// backward: dh_prev[b, u] = sum_n dg[b, n] W_hh[n, u] over all 4H gate rows for the CTA's 32 units; thread = (unit, 1/8 of the rows)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(RT, 1) bilstm_bwd_loop_kernel(const BiLoopArgs p) {
    extern __shared__ __align__(16) float smf[];
    const int H = p.H, B = p.B, L = p.L, CS = p.CS, N4 = 4 * H;
    float* Wt = smf;                                   // [4H][RU]   Wt[n][uu] = W_hh[n][u0 + uu]
    float* dgb = Wt + (size_t)N4 * RU;                 // [2][4H][RBG]
    float* red = dgb + (size_t)2 * N4 * RBG;           // [8][RBG][RU]
    __shared__ int s_len[RBG];
    const int tid = threadIdx.x;
    const int rank = blockIdx.x % CS, grp = (blockIdx.x / CS) % p.NG, dir = blockIdx.x / (CS * p.NG);
    const int u0 = rank * RU, bg0 = grp * RBG;
    const float* W = dir ? p.w_hh1 : p.w_hh0;
    for (int idx = tid; idx < N4 * RU; idx += RT) {
        const int n = idx / RU, uu = idx % RU;
        Wt[idx] = W[(size_t)n * H + u0 + uu];
    }
    for (int idx = tid; idx < 2 * N4 * RBG; idx += RT) dgb[idx] = 0.f;
    if (tid < RBG) { const int b = bg0 + tid; int l = b < B ? p.lengths[b] : 0; s_len[tid] = l < 0 ? 0 : (l > L ? L : l); }
    __syncthreads();
    int gmax = 0;
#pragma unroll
    for (int j = 0; j < RBG; ++j) gmax = max(gmax, s_len[j]);
    const int cb = tid >> 5, cu = tid & 31, bglob = bg0 + cb, u = u0 + cu;
    const bool cvalid_b = bglob < B;
    const int clen = s_len[cb];
    const int ks = tid >> 5;                           // product role: rows [ks * 4H / 8, (ks + 1) * 4H / 8)
    const size_t dirBH = (size_t)dir * (L + 1) * B * H, dirG = (size_t)dir * L * B * 4 * H;
    float dc_reg = 0.f, dh_rec = 0.f;
    cluster_arrive(); cluster_wait();
    for (int j = L - 1; j >= 0; --j) {
        const int t = dir ? L - 1 - j : j;
        const int cur = j & 1;
        const bool any = t < gmax;
        const bool valid = cvalid_b && t < clen;
        const size_t g0 = dirG + ((size_t)j * B + bglob) * 4 * H + u;
        float d4[4] = {0.f, 0.f, 0.f, 0.f};
        if (valid) {
            const float gi = __ldg(p.gates + g0), gf = __ldg(p.gates + g0 + H), gg = __ldg(p.gates + g0 + 2 * (size_t)H), go = __ldg(p.gates + g0 + 3 * (size_t)H);
            const float cp = __ldg(p.cs + dirBH + ((size_t)j * B + bglob) * H + u);
            const float dh = __ldg(p.dout + ((size_t)bglob * L + t) * 2 * H + (size_t)dir * H + u) + dh_rec;
            const float tc = tanhf(gf * cp + gi * gg);
            const float dcn = dc_reg + dh * go * (1.f - tc * tc);
            d4[0] = dcn * gg * gi * (1.f - gi);
            d4[1] = dcn * cp * gf * (1.f - gf);
            d4[2] = dcn * gi * (1.f - gg * gg);
            d4[3] = dh * tc * go * (1.f - go);
            dc_reg = dcn * gf;
            dh_rec = 0.f;              // consumed; the product below refills it.  (A frozen step keeps both carries untouched.)
        }
        if (cvalid_b) {
#pragma unroll
            for (int g = 0; g < 4; ++g) p.dg[g0 + (size_t)g * H] = d4[g];
        }
        if (!any) continue;            // whole group frozen at this position: no gradient flows, carries stay as they are
        {
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                const uint32_t offb = (uint32_t)((((size_t)cur * N4 + (size_t)g * H + u) * RBG + cb) * 4);
                for (int r = 0; r < CS; ++r) st_cluster_f32(peer_addr(dgb, (uint32_t)r) + offb, d4[g]);
            }
        }
        cluster_arrive(); cluster_wait();
        if (j > 0) {
            float acc[RBG];
#pragma unroll
            for (int q = 0; q < RBG; ++q) acc[q] = 0.f;
            const int nper = N4 / 8, n0 = ks * nper;
            const float* wt = Wt + (size_t)n0 * RU + cu;
            const float* dgp = dgb + ((size_t)cur * N4 + n0) * RBG;
#pragma unroll 4
            for (int n = 0; n < nper; ++n) {
                const float w = wt[(size_t)n * RU];
                const float4 a0 = *reinterpret_cast<const float4*>(dgp + (size_t)n * RBG);
                const float4 a1 = *reinterpret_cast<const float4*>(dgp + (size_t)n * RBG + 4);
                acc[0] = fmaf(w, a0.x, acc[0]); acc[1] = fmaf(w, a0.y, acc[1]); acc[2] = fmaf(w, a0.z, acc[2]); acc[3] = fmaf(w, a0.w, acc[3]);
                acc[4] = fmaf(w, a1.x, acc[4]); acc[5] = fmaf(w, a1.y, acc[5]); acc[6] = fmaf(w, a1.z, acc[6]); acc[7] = fmaf(w, a1.w, acc[7]);
            }
#pragma unroll
            for (int q = 0; q < RBG; ++q) red[((size_t)ks * RBG + q) * RU + cu] = acc[q];
            __syncthreads();
            float s = 0.f;
#pragma unroll
            for (int k2 = 0; k2 < 8; ++k2) s += red[((size_t)k2 * RBG + cb) * RU + cu];
            dh_rec += s;               // frozen utterance: its own dg column is zero, so s = 0 and the carry passes through
            __syncthreads();           // `red` is rewritten by the next step's product
        }
    }
}

size_t bi_fwd_smem(int H) { return ((size_t)RROWS * (H + 4) + (size_t)2 * RBG * H + (size_t)RBG * RROWS) * 4; }
size_t bi_bwd_smem(int H) { return ((size_t)4 * H * RU + (size_t)2 * 4 * H * RBG + (size_t)8 * RBG * RU) * 4; }

int launch_bi(void* fn, const BiLoopArgs& a, size_t smem, const char* name, cudaStream_t st) {
    B200_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    BiLoopArgs args = a;
    void* params[] = {&args};
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(2 * a.NG * a.CS); cfg.blockDim = dim3(RT); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attrs[1];
    attrs[0].id = cudaLaunchAttributeClusterDimension;
    attrs[0].val.clusterDim.x = a.CS; attrs[0].val.clusterDim.y = 1; attrs[0].val.clusterDim.z = 1;
    cfg.attrs = attrs; cfg.numAttrs = 1;
    KernelTimer kt(name, st);
    B200_CUDA(cudaLaunchKernelExC(&cfg, fn, params));
    B200_LAUNCH_CHECK();
    return B200TTS_OK;
}

}  // namespace

bool bilstm_persist_supported(const b200tts_bilstm_shape& s) {
    if (getenv("B200TTS_BILSTM_CHAIN")) return false;          // A/B switch: force the per-step chain
    return s.H % RU == 0 && s.H / RU >= 1 && s.H / RU <= 8 && bi_fwd_smem(s.H) <= 227 * 1024 && bi_bwd_smem(s.H) <= 227 * 1024;
}

// gates: input projection in / activated gates out; hs, cs: [2][L + 1][B][H]; out [B, L, 2H]
int bilstm_persist_forward(const b200tts_bilstm_shape& s, const float* w_hh, const float* w_hh_reverse, float* gates, float* hs, float* cs,
                           float* out, const int* lengths, cudaStream_t st) {
    BiLoopArgs a{};
    a.B = s.B; a.L = s.L; a.H = s.H; a.CS = s.H / RU; a.NG = (s.B + RBG - 1) / RBG;
    a.w_hh0 = w_hh; a.w_hh1 = w_hh_reverse; a.gates = gates; a.hs = hs; a.cs = cs; a.out = out; a.lengths = lengths;
    return launch_bi((void*)bilstm_fwd_loop_kernel, a, bi_fwd_smem(s.H), "bilstm_fwd_loop_kernel", st);
}

int bilstm_persist_backward(const b200tts_bilstm_shape& s, const float* w_hh, const float* w_hh_reverse, const float* gates, const float* cs,
                            const float* dout, float* dg, const int* lengths, cudaStream_t st) {
    BiLoopArgs a{};
    a.B = s.B; a.L = s.L; a.H = s.H; a.CS = s.H / RU; a.NG = (s.B + RBG - 1) / RBG;
    a.w_hh0 = w_hh; a.w_hh1 = w_hh_reverse; a.gates = const_cast<float*>(gates); a.cs = const_cast<float*>(cs); a.dout = dout; a.dg = dg;
    a.lengths = lengths;
    return launch_bi((void*)bilstm_bwd_loop_kernel, a, bi_bwd_smem(s.H), "bilstm_bwd_loop_kernel", st);
}

}  // namespace b200tts
