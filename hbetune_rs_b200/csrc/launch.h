// Kernel launches with a per-launch scheduling priority.
//
// The recursion of factor + inverse alternates launches that fill the GPU for a millisecond (the products of the top
// levels: thousands of CTAs) with launches that are pure latency (the 128-wide nodes and the products of the bottom
// levels: a few dozen CTAs for tens of microseconds).  Stream groups overlap the two kinds across matrices, but the
// block scheduler hands out CTAs of equal priority in launch order: a short kernel of one group launched behind a big
// product of another waits until the whole product has been *dispatched*, i.e. nearly until it ends.  Giving the
// short kernels a higher priority lets their CTAs take the next free slot instead, so a group's dependent chain keeps
// moving underneath the other groups' throughput-bound products.  (cudaLaunchAttributePriority is honoured per
// launch and is recorded into captured graph nodes.)
#pragma once
#include <cuda_runtime.h>

#include <utility>

namespace hbegp {

struct LaunchPriority {
    int least = 0, greatest = 0;
    long small_ctas = 0;  // 0: feature off

    static const LaunchPriority& get() {
        static LaunchPriority p = make();
        return p;
    }
    // Priority for a grid of `ctas` CTAs.
    int for_grid(long ctas) const {
        if (small_ctas <= 0 || ctas > small_ctas) return least;
        // shortest first: every halving of the grid below the threshold is one level up (numerically down)
        int pr = least - 1;
        for (long c = small_ctas / 2; ctas <= c && pr > greatest; c /= 2) pr--;
        return pr < greatest ? greatest : pr;
    }

private:
    static LaunchPriority make() {
        LaunchPriority p;
        if (cudaDeviceGetStreamPriorityRange(&p.least, &p.greatest) != cudaSuccess) {
            cudaGetLastError();
            p.least = p.greatest = 0;
        }
        // One resident wave of the 64 x 64 GEMM tile is 3 CTAs x 148 SMs; anything that fits in it is latency bound.
        p.small_ctas = 444;
        if (p.least == p.greatest) p.small_ctas = 0;  // no priority range on this device: feature off
        return p;
    }
};

template <typename... KArgs, typename... Args>
inline cudaError_t launch_prio(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
    const LaunchPriority& lp = LaunchPriority::get();
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributePriority;
    at[0].val.priority = lp.for_grid((long)grid.x * grid.y * grid.z);
    cfg.attrs = at;
    cfg.numAttrs = lp.small_ctas > 0 ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
}

}  // namespace hbegp
