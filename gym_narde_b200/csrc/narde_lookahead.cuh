// narde_lookahead.cuh -- the arithmetic of the one-ply expectimax lookahead (include/narde_b200.h: narde_segment_topk,
// narde_lookahead_expand, narde_lookahead_reduce).  __host__ __device__, so that the test-only host harness
// (tests/hostsim/) compiles the same top-K order and the same value arithmetic the kernels run.
#pragma once
#include <math.h>
#include <stdint.h>

#include "narde_core.cuh"

namespace narde {

constexpr int kLookaheadRolls = 21;          // NARDE_LOOKAHEAD_ROLLS
constexpr int kLookaheadMaxCandidates = 32;  // NARDE_LOOKAHEAD_MAX_CANDIDATES

// Roll d of the fixed table 1-1, 1-2, ..., 1-6, 2-2, ..., 6-6 (a <= b); its weight out of 36 is 1 for doubles, else 2.
NHD void la_roll(int d, int* a, int* b) {
  int x = 1;
  while (d >= 7 - x) {
    d -= 7 - x;
    x++;
  }
  *a = x;
  *b = x + d;
}
NHD float la_roll_weight(int d) {
  int a, b;
  la_roll(d, &a, &b);
  return a == b ? 1.0f : 2.0f;
}

NHD bool la_isnan(float x) { return x != x; }

// The order of narde_segment_argmax's choice rule made total: (v, k) comes before (w, j) when v is a number and w is NaN,
// or both are numbers and v > w, or they are equal (-0 == +0) or both NaN and k < j.  The first entry of a segment in
// this order is narde_segment_argmax's choice; the first K are narde_segment_topk's candidates, in slot order.
NHD bool la_before(float v, int k, float w, int j) {
  const bool vn = la_isnan(v), wn = la_isnan(w);
  if (vn != wn) return wn;
  if (vn || v == w) return k < j;
  return v > w;
}

// The first entry, in la_before order, of sign * seg[k] over k = k0, k0 + stride, ... < c that comes after (pv, pk)
// (every entry when !has_prev).  Returns its index and stores its signed value in *best; -1 when there is none.
NHD int la_topk_scan(const float* seg, int c, float sign, bool has_prev, float pv, int pk, int k0, int stride, float* best) {
  int bk = -1;
  float bv = 0.0f;
  for (int k = k0; k < c; k += stride) {
    const float v = sign * seg[k];
    if (has_prev && !la_before(pv, pk, v, k)) continue;
    if (bk < 0 || la_before(v, k, bv, bk)) {
      bv = v;
      bk = k;
    }
  }
  *best = bv;
  return bk;
}

// The first min(K, c) entries of the segment in la_before order: idx[0] is narde_segment_argmax's choice.  Returns their
// number.
NHD int la_topk(const float* seg, int c, float sign, int K, int32_t* idx) {
  bool has = false;
  float pv = 0.0f;
  int pk = 0, got = 0;
  for (; got < K; got++) {
    float v;
    const int k = la_topk_scan(seg, c, sign, has, pv, pk, 0, 1, &v);
    if (k < 0) break;
    idx[got] = k;
    has = true;
    pv = v;
    pk = k;
  }
  return got;
}

// v of one candidate: s0 its 0-ply score, terminal when its afterstate ends the game; r / count / eff per roll of the
// table: the opponent's best-reply score, the legal count of the reply position and the length of the list prefix the
// reply was chosen from.  A blocked roll (count 0) contributes s0; a roll whose list was not scored in full
// (eff < count) makes v NaN and sets *unfit.  acc sums w_d * r in float32 in roll order; v = acc / 36.
NHD float la_candidate_value(float s0, bool terminal, const float* r, const int32_t* count, const int32_t* eff, bool* unfit) {
  *unfit = false;
  if (terminal) return s0;
  float acc = 0.0f;
  for (int d = 0; d < kLookaheadRolls; d++) {
    float x;
    if (count[d] == 0) {
      x = s0;
    } else if (eff[d] < count[d]) {
      *unfit = true;
      continue;
    } else {
      x = r[d];
    }
    acc += la_roll_weight(d) * x;  // (w_d * x is exact: an FMA gives the same sum)
  }
  return *unfit ? nanf("") : acc / 36.0f;
}

// The chosen candidate slot: the first of sign * v[j], j < n, in la_before order -- the largest, ties to the lower slot,
// a NaN never wins, all NaN (or n == 0) -> slot 0.
NHD int la_pick(const float* v, int n, float sign) {
  int best = 0;
  for (int j = 1; j < n; j++)
    if (la_before(sign * v[j], j, sign * v[best], best)) best = j;
  return best;
}

}  // namespace narde
