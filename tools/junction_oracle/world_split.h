// tools/junction_oracle/world_split.h -- TEST INFRASTRUCTURE: the frozen rules of splitting worlds between the parts of an episode
// (include/dmpp_b200.h section 18): the keys, spec_exp, the select of one population (potentials, systematic resampling, lineage,
// assignment) and the perturbation of one world.  IEEE binary64, operations in the order written, no contraction (fma only where
// written); csrc/dp_world_split.cu evaluates the same expressions.  The copy itself is a plain gather along the world axis.
#pragma once
#include <cstdint>

#include "../../include/dmpp_b200.h"

namespace split {
uint64_t mix(uint64_t z);
uint64_t key(uint64_t seed, int level, uint64_t a, uint64_t b);
double u01(uint64_t h);
double spec_exp(double x);
// population g of M worlds: met[M] / rows[M] / map[M] (sources relative to the population's first world, -1 for no copy), in place
void select(const dp_split_params& p, int M, int g, int level, const dp_episode_metrics* met, dp_split_row* rows, dp_split_group& grp,
            int32_t* map);
// world i (relative to the call's first world): agents[max_obs], v0[max_obs] (NULL: the reactive agents are disarmed)
void perturb(const dp_split_params& p, int level, int i, int n_obs, int max_obs, dp_agent* agents, double* v0);
}  // namespace split
