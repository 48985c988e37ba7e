// match_hostsim.cpp -- TEST-ONLY host build of the match arithmetic (gym_narde_b200/csrc/narde_match.cuh): the seat rule
// of narde_match_split_counts, the outcome of narde_match_tally and what a game adds to the tallies, compiled with g++
// from the same source the kernels use and wrapped in plain loops (HOST pointers), for tests/test_gpu_match.py's CPU tests.
#include <stdint.h>

#include "../../gym_narde_b200/csrc/narde_match.cuh"

using namespace narde;

extern "C" {

// g [n] global ids, meta [n] the hi lane's meta word, counts [n], kinds -> owner [n] (0 = A, 1 = B), counts_a / counts_b [n]
void hs_match_split(const uint64_t* g, const uint32_t* meta, const int32_t* counts, int64_t n, int kinds, int32_t* owner,
                    int32_t* counts_a, int32_t* counts_b) {
  for (int64_t i = 0; i < n; i++) {
    owner[i] = match_owner(g[i], meta[i]);
    match_split(g[i], meta[i], counts[i], kinds, &counts_a[i], &counts_b[i]);
  }
}

// per game: g, meta, terminated, truncated, plies -> outcome [n]; tallies [9] += every game's contribution
void hs_match_tally(const uint64_t* g, const uint32_t* meta, const uint8_t* terminated, const uint8_t* truncated,
                    const int32_t* plies, int64_t n, uint8_t* outcome, int64_t* tallies) {
  for (int64_t i = 0; i < n; i++) {
    const int code = match_outcome(g[i], meta[i], terminated[i] != 0, truncated[i] != 0);
    outcome[i] = (uint8_t)code;
    int v[kMatchTallies] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    match_tally_add(g[i], code, plies[i], v);
    for (int k = 0; k < kMatchTallies; k++) tallies[k] += v[k];
  }
}

// the choice rule's sign and order, and the env's uniform pick
float hs_rule_sign(int mode, uint32_t meta) { return rule_sign(mode, meta); }
int hs_uniform_pick(uint64_t seed, uint32_t env, uint64_t step, int c) { return uniform_pick(seed, env, step, c); }

}  // extern "C"
