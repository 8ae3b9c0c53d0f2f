// Inline PTX wrappers shared by the hand-written kernels (sm_100a): mbarrier, TMA (cp.async.bulk.tensor), tcgen05.mma / commit / ld,
// TMEM allocation and UMMA descriptors, proxy fences, cp.async, ldmatrix + mma.sync, thread-block cluster / distributed shared memory
// stores, and the fast activation functions of the bf16 perf mode.  Each kernel file pulls them in with `using namespace tcx;`.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <stdint.h>

namespace b200tts {
namespace tcx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier, TMA ----
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// spin on the phase parity; a protocol bug must not hang the GPU: trap after ~2 s
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    const long long t0 = clock64();
    for (;;) {
        uint32_t done;
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(addr), "r"(parity)
            : "memory");
        if (done) return;
        if (clock64() - t0 > 4000000000ll) __trap();
    }
}
__device__ __forceinline__ void tma_load_3d(void* smem, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_u32(smem)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
__device__ __forceinline__ void tma_load_5d(void* smem, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3, int c4) {
    asm volatile(
        "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
        ::"r"(smem_u32(smem)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
        : "memory");
}

// ---- tcgen05 / TMEM ----
// D[tmem] (+)= A[smem desc] . B[smem desc]^T, bf16 operands, fp32 accumulate, one CTA
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// 32 lanes x 8 consecutive 32-bit columns (lane l of the warp reads TMEM lane (warp % 4) * 32 + l); the caller issues tmem_ld_wait()
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// 16 / 32 consecutive columns, followed by the wait: the registers are valid on return
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
    tmem_ld_wait();
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    tmem_ld_wait();
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void proxy_fence_global() { asm volatile("fence.proxy.async.global;" ::: "memory"); }
__device__ __forceinline__ void proxy_fence_shared() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}" : "=r"(pred));
    return pred != 0;
}
template <int COLS>
__device__ __forceinline__ void tmem_alloc(uint32_t* slot_in_smem) {      // one full warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot_in_smem)), "n"(COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t tmem_base) {         // one full warp
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(COLS));
}
// K-major, 128-byte swizzled operand tile (rows of 64 bf16 = 128 B, 8-row groups 1024 B apart): UMMA shared-memory descriptor
// (cute::UMMA::SmemDescriptor: start >> 4 | LBO << 16 | SBO << 32 | version 1 << 46 | SWIZZLE_128B (2) << 61)
__device__ __forceinline__ uint64_t make_sw128_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
    d |= (uint64_t)1 << 16;                 // leading byte offset (unused for swizzled K-major; canonical value 1)
    d |= (uint64_t)(1024 >> 4) << 32;       // stride byte offset: next 8-row group
    d |= (uint64_t)1 << 46;                 // descriptor version (Blackwell)
    d |= (uint64_t)2 << 61;                 // SWIZZLE_128B
    return d;
}
// MN-major, 128-byte swizzled operand tile: 64-element (128 B) lines along MN, one line per k row, 8-row groups 1024 B apart (stride
// byte offset), the next 64-element MN chunk 8 KB further (leading byte offset); a K = 16 instruction step advances 16 rows = 2048 B
// (canonical layout Swizzle<3,4,3> o ((8,n),(8,k)):((1,LBO),(8,SBO)) in 16-byte units, cute::UMMA::make_umma_desc<Major::MN>)
__device__ __forceinline__ uint64_t make_sw128_mn_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
    d |= (uint64_t)(8192 >> 4) << 16;       // leading byte offset: next 64-wide MN chunk
    d |= (uint64_t)(1024 >> 4) << 32;       // stride byte offset: next group of 8 k rows
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
// instruction descriptor: bf16 x bf16 -> f32, both operands K-major, M x N tile
__device__ __forceinline__ uint32_t make_idesc_bf16(int M, int N) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// ---- cp.async, ldmatrix, mma.sync ----
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(smem_u32(smem)), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }
__device__ __forceinline__ void cp_async_commit_wait() { asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;\n" ::); }
__device__ __forceinline__ void ldmatrix_x4(uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3, const void* p) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];\n" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(smem_u32(p)));
}
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3, const void* p) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];\n"
                 : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(smem_u32(p)));
}
__device__ __forceinline__ void mma_bf16(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// ---- thread-block cluster (CTA pair / group) primitives: split arrive / wait barrier, distributed-shared-memory stores ----
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
// address of the same shared-memory location in the CTA of cluster rank `rank`
__device__ __forceinline__ uint32_t peer_addr(const void* local_smem, uint32_t rank) {
    uint32_t ra;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(smem_u32(local_smem)), "r"(rank));
    return ra;
}
__device__ __forceinline__ void st_cluster_f32(uint32_t addr, float v) { asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory"); }
__device__ __forceinline__ void st_peer_f32(const float* local_smem, uint32_t peer_rank, float v) {
    st_cluster_f32(peer_addr(local_smem, peer_rank), v);
}
// remote store that completes its 4 bytes on the PEER's mbarrier (data + signal in one instruction): the pair exchanges need no cluster
// barrier and none of the memory fence its release semantics imply
__device__ __forceinline__ void st_async_peer_f32(const float* local_smem, const uint64_t* local_bar, uint32_t peer_rank, float v) {
    const uint32_t ra = peer_addr(local_smem, peer_rank), rb = peer_addr(local_bar, peer_rank);
    asm volatile("st.async.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];" ::"r"(ra), "r"(__float_as_uint(v)), "r"(rb) : "memory");
}
__device__ __forceinline__ void l2_prefetch(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// ---- conversions and activations of the bf16 perf mode ----
__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float tanh_fast(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// gate nonlinearities: ex2-based, ~1e-6 relative error (the operands of the products are bf16 anyway); the reverse loops recompute the
// cell-state tanh with the same form
__device__ __forceinline__ float sigmoid_fast(float x) { return __fdividef(1.f, 1.f + __expf(-x)); }
__device__ __forceinline__ float tanh_exp(float x) { return 2.f * __fdividef(1.f, 1.f + __expf(-2.f * x)) - 1.f; }

}  // namespace tcx
}  // namespace b200tts
