// csrc/dp_world_split.cu -- splitting worlds between the parts of an episode (include/dmpp_b200.h section 18): the select launch
// (one CTA per population: potentials, the sequential prefix, systematic resampling, the lineage update and the map) and the
// perturb launch (one warp per world).  The copy between them is dp_world_fork.cu's.  The arithmetic restates
// tools/junction_oracle/world_split.cpp expression for expression (-fmad=false; fma only where written).  A translation unit of its
// own: every other kernel compiles to what it compiled to before.
#include "dp_kernels.h"

namespace {
__device__ __forceinline__ unsigned long long split_mix(unsigned long long z) {
    z ^= z >> 30; z *= 0xbf58476d1ce4e5b9ull;
    z ^= z >> 27; z *= 0x94d049bb133111ebull;
    return z ^ (z >> 31);
}
__device__ __forceinline__ unsigned long long split_key(unsigned long long seed, int level, unsigned long long a, unsigned long long b) {
    return split_mix(split_mix(split_mix(split_mix(seed) ^ (unsigned long long)level) ^ a) ^ b);
}
__device__ __forceinline__ double split_u01(unsigned long long h) { return (double)(h >> 11) * 0x1.0p-53; }

__device__ __forceinline__ double spec_exp(double x) {
    const double k = rint(x * 1.44269504088896338700e+00);
    double r = fma(-k, 6.93147180369123816490e-01, x);
    r = fma(-k, 1.90821492927058770002e-10, r);
    double q = 1.0 / 6227020800.0;
    q = fma(r, q, 1.0 / 479001600.0);
    q = fma(r, q, 1.0 / 39916800.0);
    q = fma(r, q, 1.0 / 3628800.0);
    q = fma(r, q, 1.0 / 362880.0);
    q = fma(r, q, 1.0 / 40320.0);
    q = fma(r, q, 1.0 / 5040.0);
    q = fma(r, q, 1.0 / 720.0);
    q = fma(r, q, 1.0 / 120.0);
    q = fma(r, q, 1.0 / 24.0);
    q = fma(r, q, 1.0 / 6.0);
    q = fma(r, q, 0.5);
    q = fma(r, q, 1.0);
    q = fma(r, q, 1.0);
    return q * __longlong_as_double(((long long)k + 1023) << 52);
}

constexpr int SPLIT_MAX_M = 1024;

// inclusive scan of one int per thread over the CTA (Hillis-Steele through shared memory; blockDim.x <= SPLIT_MAX_M)
__device__ __forceinline__ int cta_scan(int v, int* buf) {
    const int t = threadIdx.x;
    buf[t] = v;
    __syncthreads();
    for (int d = 1; d < (int)blockDim.x; d <<= 1) {
        const int x = t >= d ? buf[t - d] : 0;
        __syncthreads();
        buf[t] += x;
        __syncthreads();
    }
    const int r = buf[t];
    __syncthreads();
    return r;
}

// population blockIdx.x, thread j = world j of it
__global__ void __launch_bounds__(SPLIT_MAX_M) dp_world_split_select_kernel(dp_split_params p, int level, const dp_episode_metrics* __restrict__ met,
                                                                            dp_split_row* __restrict__ rows, dp_split_group* __restrict__ groups,
                                                                            int32_t* __restrict__ map) {
    __shared__ double s_w[SPLIT_MAX_M];                     // the potentials, then the prefix C_j
    __shared__ int s_a[SPLIT_MAX_M];                        // scan buffer, then the extra copies' inclusive scan
    __shared__ int s_root[SPLIT_MAX_M];                     // distinct roots after the copy
    const int M = p.group, g = blockIdx.x, j = threadIdx.x;
    const size_t i = (size_t)g * M + j;
    dp_split_row row = rows[i];
    dp_split_group grp = groups[g];
    if (level == 0) {
        row = dp_split_row{-p.c_max, 1.0, j, 0};
        grp = dp_split_group{1.0, 0, 0, M, 0};
    }
    const double c = met[i].min_clearance;
    const double V = -(c < p.c_max ? c : p.c_max);
    const double w = spec_exp(p.beta * (V - row.v_prev));
    s_w[j] = w;
    s_root[j] = 0;
    __syncthreads();
    if (j == 0) {                                           // the sequential prefix: M dependent adds, as the checker sums them
        double acc = 0;
        for (int t = 0; t < M; ++t) { acc = acc + s_w[t]; s_w[t] = acc; }
    }
    __syncthreads();
    const double W = s_w[M - 1];
    const double u = split_u01(split_key(p.seed, level, (1ull << 63) | (unsigned long long)g, 0));
    auto A = [&](int t) -> int {
        if (t < 0) return 0;
        if (t == M - 1) return M;
        const double x = ceil(((double)M * s_w[t]) / W - u);
        return x < 0 ? 0 : (x > (double)M ? M : (int)x);
    };
    const int N = A(j) - A(j - 1);
    // lineage (before the copy, so copies inherit it)
    row.lw = row.lw * w;
    row.v_prev = V;
    rows[i] = row;
    // extra copies of j: ranks [ex - (N - 1), ex) among all extras; empty slot j: rank ez - 1 among the empties
    const int ex = cta_scan(N > 1 ? N - 1 : 0, s_a);
    const int ez = cta_scan(N == 0 ? 1 : 0, s_a);
    s_a[j] = ex;
    __syncthreads();
    int src = -1;
    if (N == 0) {                                           // the first t whose inclusive extra count exceeds this slot's rank
        const int r = ez - 1;
        int lo = 0, hi = M - 1;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (s_a[mid] > r) hi = mid; else lo = mid + 1;
        }
        src = lo;
    }
    map[i] = src >= 0 ? (int32_t)((size_t)g * M + src) : -1;
    const int root = src >= 0 ? rows[(size_t)g * M + src].root : row.root;   // (rows of this CTA, written above)
    __syncthreads();
    if (root >= 0 && root < M) s_root[root] = 1;
    __syncthreads();
    const int alive = cta_scan(s_root[j], s_a);
    if (j == M - 1) {
        grp.norm = grp.norm * (W / (double)M);
        grp.levels += 1;
        grp.copies += ex;
        grp.roots_alive = alive;
        groups[g] = grp;
    }
}

constexpr int PERTURB_WPB = 8;                              // warps (= worlds) per CTA

__global__ void __launch_bounds__(PERTURB_WPB * 32) dp_world_perturb_kernel(dp_split_params p, int level, int n, int max_obs,
                                                                            const dp_scene_hdr* __restrict__ hdr, dp_agent* __restrict__ agents,
                                                                            double* __restrict__ v0) {
    const int lane = threadIdx.x & 31, i = blockIdx.x * PERTURB_WPB + (threadIdx.x >> 5);
    if (i >= n) return;
    const int na = min((int)hdr[i].n_obs, max_obs);
    for (int k = lane; k < na; k += 32) {
        const size_t e = (size_t)i * max_obs + k;
        const double x = split_u01(split_key(p.seed, level, (unsigned long long)i, 2 * (unsigned long long)k));
        const double f = 1.0 + p.amp_v * (2.0 * x - 1.0);
        agents[e].v = agents[e].v * f;
        if (v0) {
            const double x1 = split_u01(split_key(p.seed, level, (unsigned long long)i, 2 * (unsigned long long)k + 1));
            const double f1 = 1.0 + p.amp_v0 * (2.0 * x1 - 1.0);
            v0[e] = v0[e] * f1;
        }
    }
}
}  // namespace

cudaError_t dp_launch_world_split_select(const dp_split_params& p, int n, int level, const dp_episode_metrics* met, dp_split_row* rows,
                                         dp_split_group* groups, int32_t* map, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    dp_world_split_select_kernel<<<n / p.group, p.group, 0, st>>>(p, level, met, rows, groups, map);
    return cudaGetLastError();
}

cudaError_t dp_launch_world_perturb(const dp_split_params& p, int n, int level, int max_obs, const dp_scene_hdr* hdr, dp_agent* agents,
                                    double* v0, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    dp_world_perturb_kernel<<<(n + PERTURB_WPB - 1) / PERTURB_WPB, PERTURB_WPB * 32, 0, st>>>(p, level, n, max_obs, hdr, agents, v0);
    return cudaGetLastError();
}
