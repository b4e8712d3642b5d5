// tools/junction_oracle/world_split.cpp -- TEST INFRASTRUCTURE: see world_split.h
#include "world_split.h"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <vector>

namespace split {
uint64_t mix(uint64_t z) {
    z ^= z >> 30; z *= 0xbf58476d1ce4e5b9ull;
    z ^= z >> 27; z *= 0x94d049bb133111ebull;
    return z ^ (z >> 31);
}
uint64_t key(uint64_t seed, int level, uint64_t a, uint64_t b) { return mix(mix(mix(mix(seed) ^ (uint64_t)level) ^ a) ^ b); }
double u01(uint64_t h) { return (double)(h >> 11) * 0x1.0p-53; }

double spec_exp(double x) {
    const double k = std::rint(x * 1.44269504088896338700e+00);
    double r = std::fma(-k, 6.93147180369123816490e-01, x);    // ln 2, high part (k * ln2_hi is exact for |k| < 2^21)
    r = std::fma(-k, 1.90821492927058770002e-10, r);            // ln 2, low part
    double q = 1.0 / 6227020800.0;                              // 1/13!
    q = std::fma(r, q, 1.0 / 479001600.0);                      // 1/12!
    q = std::fma(r, q, 1.0 / 39916800.0);                       // 1/11!
    q = std::fma(r, q, 1.0 / 3628800.0);                        // 1/10!
    q = std::fma(r, q, 1.0 / 362880.0);                         // 1/9!
    q = std::fma(r, q, 1.0 / 40320.0);                          // 1/8!
    q = std::fma(r, q, 1.0 / 5040.0);                           // 1/7!
    q = std::fma(r, q, 1.0 / 720.0);                            // 1/6!
    q = std::fma(r, q, 1.0 / 120.0);                            // 1/5!
    q = std::fma(r, q, 1.0 / 24.0);                             // 1/4!
    q = std::fma(r, q, 1.0 / 6.0);                              // 1/3!
    q = std::fma(r, q, 0.5);                                    // 1/2!
    q = std::fma(r, q, 1.0);                                    // 1/1!
    q = std::fma(r, q, 1.0);                                    // 1/0!
    const uint64_t bits = (uint64_t)((int64_t)k + 1023) << 52;  // 2^k (|k| <= 73 on [-50, 50]: a normal number)
    double s;
    std::memcpy(&s, &bits, sizeof(s));
    return q * s;
}

void select(const dp_split_params& p, int M, int g, int level, const dp_episode_metrics* met, dp_split_row* rows, dp_split_group& grp,
            int32_t* map) {
    if (level == 0) {
        for (int j = 0; j < M; ++j) rows[j] = dp_split_row{-p.c_max, 1.0, j, 0};
        grp = dp_split_group{1.0, 0, 0, M, 0};
    }
    std::vector<double> w((size_t)M), V((size_t)M), C((size_t)M);
    for (int j = 0; j < M; ++j) {
        const double c = met[j].min_clearance;
        V[j] = -(c < p.c_max ? c : p.c_max);
        w[j] = spec_exp(p.beta * (V[j] - rows[j].v_prev));
    }
    double acc = 0;
    for (int j = 0; j < M; ++j) { acc = acc + w[j]; C[j] = acc; }
    const double W = C[M - 1];
    const double u = u01(key(p.seed, level, (1ull << 63) | (uint64_t)g, 0));
    std::vector<int> N((size_t)M);
    int a_prev = 0;
    for (int j = 0; j < M; ++j) {
        int a = M;
        if (j < M - 1) {
            const double t = std::ceil(((double)M * C[j]) / W - u);
            a = t < 0 ? 0 : (t > (double)M ? M : (int)t);
        }
        N[j] = a - a_prev;
        a_prev = a;
    }
    for (int j = 0; j < M; ++j) {
        rows[j].lw = rows[j].lw * w[j];
        rows[j].v_prev = V[j];
    }
    grp.norm = grp.norm * (W / (double)M);
    grp.levels += 1;
    // the extra copies in increasing j, the empty slots in increasing index, paired in order
    std::fill(map, map + M, -1);
    int e = 0, copies = 0;
    for (int j = 0; j < M; ++j)
        for (int r = 1; r < N[j]; ++r) {
            while (N[e] != 0) ++e;
            map[e++] = j;
            ++copies;
        }
    grp.copies += copies;
    std::vector<char> seen((size_t)M, 0);
    int alive = 0;
    for (int j = 0; j < M; ++j) {
        const int root = rows[map[j] >= 0 ? map[j] : j].root;
        if (root >= 0 && root < M && !seen[root]) { seen[root] = 1; ++alive; }
    }
    grp.roots_alive = alive;
}

void perturb(const dp_split_params& p, int level, int i, int n_obs, int max_obs, dp_agent* agents, double* v0) {
    const int na = std::min(n_obs, max_obs);
    for (int k = 0; k < na; ++k) {
        const double x = u01(key(p.seed, level, (uint64_t)i, 2 * (uint64_t)k));
        const double f = 1.0 + p.amp_v * (2.0 * x - 1.0);
        agents[k].v = agents[k].v * f;
        if (v0) {
            const double x1 = u01(key(p.seed, level, (uint64_t)i, 2 * (uint64_t)k + 1));
            const double f1 = 1.0 + p.amp_v0 * (2.0 * x1 - 1.0);
            v0[k] = v0[k] * f1;
        }
    }
}
}  // namespace split
