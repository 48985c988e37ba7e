// lookahead_hostsim.cpp -- TEST-ONLY host build of the lookahead arithmetic (gym_narde_b200/csrc/narde_lookahead.cuh):
// the top-K order of narde_segment_topk and the value / choice of narde_lookahead_reduce, compiled with g++ from the same
// source the kernels use and wrapped in plain loops (HOST pointers), for tests/test_gpu_lookahead.py's CPU tests.
#include <stdint.h>

#include "../../gym_narde_b200/csrc/narde_lookahead.cuh"

using namespace narde;

extern "C" {

void hs_la_roll(int d, int32_t* ab, float* w) {
  la_roll(d, &ab[0], &ab[1]);
  *w = la_roll_weight(d);
}

// seg [n, width] f32 rows, counts [n], sign [n] -> idx [n, K], got [n]
void hs_la_topk(const float* seg, int64_t n, int width, const int32_t* counts, const float* sign, int K, int32_t* idx,
                int32_t* got) {
  for (int64_t i = 0; i < n; i++) got[i] = la_topk(seg + i * width, counts[i], sign[i], K, idx + i * K);
}

// per candidate c: s0, terminal, r / count / eff [c, 21] -> v [c], unfit [c]
void hs_la_value(const float* s0, const uint8_t* terminal, const float* r, const int32_t* count, const int32_t* eff,
                 int64_t n, float* v, uint8_t* unfit) {
  for (int64_t c = 0; c < n; c++) {
    bool u;
    v[c] = la_candidate_value(s0[c], terminal[c] != 0, r + 21 * c, count + 21 * c, eff + 21 * c, &u);
    unfit[c] = u ? 1 : 0;
  }
}

// v [n, K], count [n], sign [n] -> slot [n]
void hs_la_pick(const float* v, int64_t n, int K, const int32_t* count, const float* sign, int32_t* slot) {
  for (int64_t i = 0; i < n; i++) slot[i] = la_pick(v + i * K, count[i], sign[i]);
}

}  // extern "C"
