// Shared pieces of the persistent decoder loops (one cooperative launch runs all T steps): the grid barrier, the per-phase cycle
// counters, the barrier-region layout and the launch helper.
#pragma once
#include <stdlib.h>
#include "common.cuh"
#include "ptx.cuh"

namespace b200tts {

struct NoOverlap { __device__ __forceinline__ void operator()() const {} };

// Monotonic-counter grid barrier over ALL threads of every CTA.  Returns false if the watchdog fired (~2 s, or another CTA's watchdog
// raised *abort_flag): the caller must leave its loop.  `s_ok` is a __shared__ int of the calling kernel.
//   * arrival = ONE release-reduction: it is cumulative over the CTA's writes, which the __syncthreads before it made visible to thread 0;
//   * the wait polls with relaxed loads (nothing else in the loop: its round trip is the barrier latency) and issues a single acquire
//     fence after the last one;
//   * ASYNC_FENCE: global data written before the barrier is read by other CTAs through TMA (async proxy), so thread 0 orders the
//     generic-proxy writes against the async proxy before it arrives;
//   * `overlap` runs on every thread BETWEEN the CTA's arrival and its wait: work that does not depend on other CTAs (next step's
//     operand prefetch) hides under the barrier latency instead of delaying the arrival.
template <bool ASYNC_FENCE, typename Overlap = NoOverlap>
__device__ __forceinline__ bool grid_barrier(unsigned* counter, unsigned& target, unsigned nblocks, int* abort_flag, int* s_ok,
                                             Overlap overlap = Overlap()) {
    __syncthreads();
    if (threadIdx.x == 0) {
        target += nblocks;
        if (ASYNC_FENCE) tcx::proxy_fence_global();
        asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(counter) : "memory");
    }
    overlap();
    if (threadIdx.x == 0) {
        int ok = 1;
        const long long t0 = clock64();
        unsigned polls = 0;
        for (;;) {
            unsigned v;
            asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(counter) : "memory");
            if (v >= target) break;
            if ((++polls & 255u) == 0 && (clock64() - t0 > 4000000000ll || *reinterpret_cast<volatile int*>(abort_flag))) {
                ok = 0; *abort_flag = 1; break;
            }
        }
        asm volatile("fence.acquire.gpu;" ::: "memory");
        *s_ok = ok;
    }
    __syncthreads();
    return *s_ok != 0;
}

// Per-phase cycle totals seen by thread 0 of each CTA, written to the optional p.prof [gridDim.x][8] when the loop ends.
#define PROF_DECL                                                                                                   \
    long long prof_acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};                                                               \
    long long prof_t = clock64();
#define PROF_MARK(slot)                                                                                             \
    do {                                                                                                            \
        if (p.prof && threadIdx.x == 0) { const long long now = clock64(); prof_acc[slot] += now - prof_t; prof_t = now; } \
    } while (0)
#define PROF_FLUSH                                                                                                  \
    do {                                                                                                            \
        if (p.prof && threadIdx.x == 0)                                                                             \
            for (int k9 = 0; k9 < 8; ++k9) p.prof[(size_t)blockIdx.x * 8 + k9] = prof_acc[k9];                      \
    } while (0)

// Barrier region of a persistent loop: 256 bytes zeroed before each launch, the counter at +0 and the abort flag at +128 B; the
// per-phase profile counters follow at +256 B.  Sets a.barrier, a.abort_flag and a.prof.
template <typename Args>
int reset_grid_barrier(unsigned char* region, Args& a, cudaStream_t st) {
    a.barrier = reinterpret_cast<unsigned*>(region);
    a.abort_flag = reinterpret_cast<int*>(region + 128);
    a.prof = reinterpret_cast<long long*>(region + 256);
    B200_CUDA(cudaMemsetAsync(region, 0, 256, st));
    return B200TTS_OK;
}

// Cooperative launch of a persistent kernel whose `grid` CTAs must all be co-resident (its grid barriers would deadlock otherwise).
//   cluster = 2: CTA pairs; co-residency is checked in clusters, else per SM.
//   profile_no_coop: B200TTS_PROFILE_NO_COOP drops the cooperative attribute (profiling aid: ncu cannot capture a launch that is BOTH
//   cooperative and clustered; the kernel carries its own grid barrier, so on an otherwise idle GPU with all CTAs resident the attribute
//   can be dropped for a capture).
//   timer: KernelTimer name, or nullptr for none.
inline int launch_persistent(const void* fn, int grid, int block, size_t smem, void** params, cudaStream_t st, const char* what,
                             const char* timer, int cluster = 1, bool profile_no_coop = false) {
    B200_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(block); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attrs[2];
    attrs[0].id = cudaLaunchAttributeCooperative;
    attrs[0].val.cooperative = profile_no_coop && getenv("B200TTS_PROFILE_NO_COOP") ? 0 : 1;
    cfg.attrs = attrs; cfg.numAttrs = 1;
    if (cluster > 1) {
        attrs[1].id = cudaLaunchAttributeClusterDimension;
        attrs[1].val.clusterDim.x = cluster; attrs[1].val.clusterDim.y = 1; attrs[1].val.clusterDim.z = 1;
        cfg.numAttrs = 2;
        int nclusters = 0;
        B200_CUDA(cudaOccupancyMaxActiveClusters(&nclusters, fn, &cfg));
        B200_REQUIRE(nclusters * cluster >= grid, "%s: only %d CTA clusters of %d can be co-resident, %d needed", what, nclusters, cluster,
                     grid / cluster);
    } else {
        int per_sm = 0, dev = 0, sms = 0;
        B200_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, block, smem));
        B200_CUDA(cudaGetDevice(&dev));
        B200_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        B200_REQUIRE(per_sm * sms >= grid, "%s: %d CTAs cannot be co-resident (%d per SM x %d SMs)", what, grid, per_sm, sms);
    }
    {
        KernelTimer kt(timer, st);
        B200_CUDA(cudaLaunchKernelExC(&cfg, fn, params));
    }
    B200_LAUNCH_CHECK();
    return B200TTS_OK;
}

}  // namespace b200tts
