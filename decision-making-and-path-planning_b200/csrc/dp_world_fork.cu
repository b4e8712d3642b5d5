// csrc/dp_world_fork.cu -- forking closed-loop worlds on the device (include/dmpp_b200.h section 17): world dst + j becomes a byte
// copy of world src[j] in every per-world buffer the episode carries.  One warp per destination world walks a table of segments
// (base, bytes per world); the table and the source indices travel in the kernel parameters, so a fork needs no staging buffer and
// no host-to-device copy ahead of it.  A translation unit of its own: every other kernel compiles to what it compiled to before.
#include "dp_kernels.h"

namespace {
constexpr int FORK_WPB = 8;                                 // warps (= destination worlds) per CTA
// words of type T per lane, DP_FORK_BATCH loads in flight before their stores (source and destination may share a buffer, so the
// compiler could not hoist the loads of later iterations above the stores of earlier ones by itself)
constexpr int DP_FORK_BATCH = 4;
template <class T>
__device__ __forceinline__ void fork_copy(unsigned char* base, unsigned bytes, int s, int d, int lane) {
    const T* __restrict__ from = reinterpret_cast<const T*>(base + (size_t)s * bytes);
    T* __restrict__ to = reinterpret_cast<T*>(base + (size_t)d * bytes);
    const int words = (int)(bytes / sizeof(T));
    for (int i0 = 0; i0 < words; i0 += 32 * DP_FORK_BATCH) {
        T v[DP_FORK_BATCH];
#pragma unroll
        for (int b = 0; b < DP_FORK_BATCH; ++b) {
            const int i = i0 + b * 32 + lane;
            if (i < words) v[b] = from[i];
        }
#pragma unroll
        for (int b = 0; b < DP_FORK_BATCH; ++b) {
            const int i = i0 + b * 32 + lane;
            if (i < words) to[i] = v[b];
        }
    }
}

// world d becomes a copy of world s in every segment of the table (one warp)
__device__ __forceinline__ void fork_world(const DpForkSeg* seg, int n_seg, int s, int d, int lane) {
    for (int k = 0; k < n_seg; ++k) {
        const DpForkSeg& g = seg[k];
        switch (g.width) {
            case 16: fork_copy<uint4>(g.base, g.bytes, s, d, lane); break;
            case 8: fork_copy<unsigned long long>(g.base, g.bytes, s, d, lane); break;
            case 4: fork_copy<unsigned>(g.base, g.bytes, s, d, lane); break;
            default: fork_copy<unsigned char>(g.base, g.bytes, s, d, lane); break;
        }
    }
}

__global__ void __launch_bounds__(FORK_WPB * 32) dp_world_fork_kernel(const __grid_constant__ DpForkArgs a) {
    const int lane = threadIdx.x & 31, j = blockIdx.x * FORK_WPB + (threadIdx.x >> 5);
    if (j >= a.count) return;
    fork_world(a.seg, a.n_seg, a.src[j], a.dst + j, lane);
}

// the copy of a split (include/dmpp_b200.h section 18): world i becomes a copy of world map[i] where map[i] >= 0.  The map lives in
// device memory (the select launch wrote it), so one launch covers any number of worlds
__global__ void __launch_bounds__(FORK_WPB * 32) dp_world_fork_map_kernel(const __grid_constant__ DpForkTable t, int n, const int32_t* __restrict__ map) {
    const int lane = threadIdx.x & 31, i = blockIdx.x * FORK_WPB + (threadIdx.x >> 5);
    if (i >= n) return;
    const int s = map[i];
    if (s < 0) return;
    fork_world(t.seg, t.n_seg, s, i, lane);
}
}  // namespace

cudaError_t dp_launch_world_fork(const DpForkArgs& a, cudaStream_t st) {
    if (a.count <= 0) return cudaSuccess;
    dp_world_fork_kernel<<<(a.count + FORK_WPB - 1) / FORK_WPB, FORK_WPB * 32, 0, st>>>(a);
    return cudaGetLastError();
}

cudaError_t dp_launch_world_fork_map(const DpForkTable& t, int n, const int32_t* map, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    dp_world_fork_map_kernel<<<(n + FORK_WPB - 1) / FORK_WPB, FORK_WPB * 32, 0, st>>>(t, n, map);
    return cudaGetLastError();
}
