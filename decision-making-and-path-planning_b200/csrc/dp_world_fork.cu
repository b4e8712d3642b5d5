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

__global__ void __launch_bounds__(FORK_WPB * 32) dp_world_fork_kernel(const __grid_constant__ DpForkArgs a) {
    const int lane = threadIdx.x & 31, j = blockIdx.x * FORK_WPB + (threadIdx.x >> 5);
    if (j >= a.count) return;
    const int s = a.src[j], d = a.dst + j;
    for (int k = 0; k < a.n_seg; ++k) {
        const DpForkSeg& g = a.seg[k];
        switch (g.width) {
            case 16: fork_copy<uint4>(g.base, g.bytes, s, d, lane); break;
            case 8: fork_copy<unsigned long long>(g.base, g.bytes, s, d, lane); break;
            case 4: fork_copy<unsigned>(g.base, g.bytes, s, d, lane); break;
            default: fork_copy<unsigned char>(g.base, g.bytes, s, d, lane); break;
        }
    }
}
}  // namespace

cudaError_t dp_launch_world_fork(const DpForkArgs& a, cudaStream_t st) {
    if (a.count <= 0) return cudaSuccess;
    dp_world_fork_kernel<<<(a.count + FORK_WPB - 1) / FORK_WPB, FORK_WPB * 32, 0, st>>>(a);
    return cudaGetLastError();
}
