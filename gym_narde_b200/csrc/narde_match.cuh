// narde_match.cuh -- the per-env arithmetic of lock-step matches between two policies (include/narde_b200.h:
// narde_match_split_counts, narde_match_choose, narde_match_tally) and the parts of the choice rule the segment kernels
// share with them: the order of narde_segment_argmax (beats), its sign and the env's own uniform action.
// __host__ __device__, so that the test-only host harness (tests/hostsim/) compiles the same seat, outcome and tally
// rules the kernels run.
#pragma once
#include <math.h>
#include <stdint.h>

#include "narde_core.cuh"

namespace narde {

// The order of the choice rule (include/narde_b200.h, narde_segment_argmax), shared by the segment kernels, their
// shuffle reduction, the Gumbel path and narde_match_choose: (v, k) beats the current (best, best_k) when there is no
// current choice yet (best_k == kNoChoice), or v is a number and best is NaN, or v > best, or v == best at a lower index.
// A NaN never beats a number, so one diverged afterstate does not decide the move, and an all-NaN segment keeps its
// first index.
constexpr int kNoChoice = 0x7FFFFFFF;
NHD bool beats(float v, int k, float best, int best_k) {
  return best_k == kNoChoice || (!isnan(v) && (isnan(best) || v > best || (v == best && k < best_k)));
}

// The sign of the choice rule for a state's meta word: mode 1 (a net that scores positions for WHITE) negates the
// scores when BLACK is to move, so that BLACK minimises; mode 0 (the mover maximises) keeps them.
NHD float rule_sign(int mode, uint32_t meta) {
  return (mode == 1 && (int)(int8_t)((meta >> 16) & 0xFF) != 1) ? -1.0f : 1.0f;
}

// The env's own uniform action over c >= 1 actions: word z of Philox stream 0 of (global env id, turn), k = (z * c) >> 32.
// Over the whole list it is the action narde_step_full plays without an action index.
NHD int uniform_pick(uint64_t seed, uint32_t env, uint64_t step, int c) {
  return (int)mulhi32(turn_random(seed, env, step).z, (uint32_t)c);
}

// ---- matches ----------------------------------------------------------------------------------
// Seats: policy A plays WHITE in games of even global id g and BLACK in odd ones; policy B the other colour.
constexpr int kMatchTallies = 9;   // NARDE_MATCH_TALLIES
enum : int {                       // tally slots (NARDE_MATCH_* in include/narde_b200.h)
  MT_GAMES = 0, MT_A_WINS, MT_B_WINS, MT_A_MARS, MT_B_MARS, MT_TRUNCATED, MT_A_WHITE_WINS, MT_B_WHITE_WINS, MT_PLIES
};
enum : int { MO_RUNNING = 0, MO_A_WON = 1, MO_B_WON = 2, MO_TRUNCATED = 3, MO_MARS = 4 };  // outcome codes

NHD int match_a_colour(uint64_t g) { return (g & 1u) ? -1 : 1; }

// The seat (0 = A, 1 = B) that owns the side to move of game g, from its state's meta word.
NHD int match_owner(uint64_t g, uint32_t meta) {
  return (int)(int8_t)((meta >> 16) & 0xFF) == match_a_colour(g) ? 0 : 1;
}

// narde_match_split_counts for one env: its count goes to the pool of the seat that owns the side to move when that seat
// is a net (bit p of kinds), 0 everywhere else.
NHD void match_split(uint64_t g, uint32_t meta, int count, int kinds, int32_t* ca, int32_t* cb) {
  const int p = match_owner(g, meta);
  *ca = (p == 0 && (kinds & 1)) ? count : 0;
  *cb = (p == 1 && (kinds & 2)) ? count : 0;
}

// The outcome code of game g from its state after a turn that terminated or truncated it: the winner is the side with
// 15 checkers off and a mars is the loser having none off (complete_env's test); a truncated game is MO_TRUNCATED.
NHD int match_outcome(uint64_t g, uint32_t meta, bool terminated, bool truncated) {
  if (terminated) {
    const int ow = (int)(meta & 0xFF), ob = (int)((meta >> 8) & 0xFF);
    const int winner = ow == 15 ? 1 : -1;
    const int code = winner == match_a_colour(g) ? MO_A_WON : MO_B_WON;
    return code + (((winner == 1 ? ob : ow) == 0) ? MO_MARS : 0);
  }
  return truncated ? MO_TRUNCATED : MO_RUNNING;
}

// What one game adds to the tallies once it has an outcome (v[kMatchTallies]); plies = its episode steps.
NHD void match_tally_add(uint64_t g, int code, int plies, int v[kMatchTallies]) {
  if (code == MO_RUNNING) return;
  const int r = code & 3;
  const bool a_white = match_a_colour(g) == 1;
  v[MT_GAMES] += 1;
  v[MT_A_WINS] += r == MO_A_WON;
  v[MT_B_WINS] += r == MO_B_WON;
  v[MT_A_MARS] += code == (MO_A_WON | MO_MARS);
  v[MT_B_MARS] += code == (MO_B_WON | MO_MARS);
  v[MT_TRUNCATED] += r == MO_TRUNCATED;
  v[MT_A_WHITE_WINS] += r == MO_A_WON && a_white;
  v[MT_B_WHITE_WINS] += r == MO_B_WON && !a_white;
  v[MT_PLIES] += plies;
}

}  // namespace narde
