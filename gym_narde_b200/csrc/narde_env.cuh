// narde_env.cuh -- per-environment bodies of the C-ABI entry points (include/narde_b200.h).
// The CUDA kernels (narde_kernels.cu) wrap these with coalesced state loads/stores; the
// test-only host harness (tests/hostsim/) wraps the same bodies in plain loops.
#pragma once
#include "../../include/narde_b200.h"
#include "narde_core.cuh"

namespace narde {

enum : int {
  F_REWARD_MOVER12 = 1,
  F_AUTORESET = 2,
  F_HALF_MOVES_ONLY = 4,
  F_ACTION_FRACTION = 32,
  F_ENUMERATE_ONLY = 64,
  F_PACK_RESULT = 128,
  F_DEVICE_ADVANCE = 256,  // the step index is *step_dev + 1; the kernels store it back when the step is complete
  DONE_TERMINATED = 1,
  DONE_TRUNCATED = 2,
};

// ---- reset (narde_env.py:105-120) ---------------------------------------------------------
NHD State reset_env(uint64_t seed, uint32_t env, uint64_t step) {
  return initial_state(opening_player(seed, env, step));
}

// ---- Tier R1 -------------------------------------------------------------------------------
struct MoveWriter {
  uint8_t* out;
  int n;
  NHD void operator()(int from, int to) {
    out[2 * n] = (uint8_t)from;
    out[2 * n + 1] = (uint8_t)to;
    n++;
  }
};

NHD int half_moves_env(const State& s, const uint8_t* dice4, int player_override, uint8_t* moves) {
  int player = player_override ? player_override : s.turn();
  bool first_turn = (s.flags() & (player == 1 ? FLAG_FIRST_W : FLAG_FIRST_B)) != 0;
  Pos P = decode_pos(s, player);
  int nroll = 0;
  uint8_t roll[4];
  for (int k = 0; k < 4; k++)
    if (dice4[k] != 0) roll[nroll++] = dice4[k];
  MoveWriter mw = {moves, 0};
  return half_moves_list(P, roll, nroll, first_turn, mw);
}

// ---- Tier R2 -------------------------------------------------------------------------------
NHD void step_ref_env(State& s, int d1, int d2, int code1, int code2, int max_episode_steps,
                      int* reward, int* done_bits) {
  if (s.flags() & FLAG_DONE) {  // terminated envs are left untouched
    *reward = 0;
    *done_bits = DONE_TERMINATED;
    return;
  }
  int dn;
  step_reference(s, d1, d2, code1, code2, reward, &dn);
  int bits = dn ? DONE_TERMINATED : 0;
  if (!dn && max_episode_steps > 0 && (int)s.steps() >= max_episode_steps) bits |= DONE_TRUNCATED;
  *done_bits = bits;
}

// ---- Tier N: fused full-rules step ---------------------------------------------------------
struct StepFullArgs {
  int64_t env_base;
  uint64_t seed, step;
  const uint8_t* dice_in;
  const int32_t* action_idx;
  int cap;
  uint64_t* actions;
  int32_t* counts;
  uint8_t* dice_out;
  uint64_t* chosen;
  float* reward;
  uint8_t* done;       // terminated (0/1)
  uint8_t* truncated;  // TimeLimit hit without termination (0/1), may be NULL
  int flags;
  int max_episode_steps;
  // optional deferral of block-rule doubles turns to the CTA-per-env kernel (narde_deferred.cuh):
  // defer_count[0] = number of deferred envs, defer_list[k] = their local indices
  int32_t* defer_count;
  int32_t* defer_list;
  // optional device-resident step counter (overrides `step`): lets the whole step be replayed as a
  // CUDA graph with frozen kernel arguments
  const uint64_t* step_dev;
  // F_DEVICE_ADVANCE: arrival counter of the exact kernel's CTAs; the last one resets the list and adds 1 to *step_dev
  int32_t* ticket;
  // publication of the deferred list to the exact kernel (a programmatic dependent launch that starts before the
  // main kernel has completed): every main CTA adds 1 with release semantics after pushing its entries, the exact
  // kernel acquires `arrivals == n_primary` before it reads the list
  int32_t* arrivals;
  int32_t n_primary;
  // large batches (several waves of main CTAs): the main kernel triggers its dependent at its very START, so the exact
  // kernel's CTAs become resident as soon as the last main CTA has been dispatched, run the solver once on a built-in
  // position (its code executes once per CTA: cold, it is bound by instruction fetch) and then wait for the list
  int32_t early_trigger;
  int64_t list_cap;  // entries the list can hold (= n): CTAs of the exact kernel beyond it have no entry to wait for
  int32_t* last_count;  // diagnostic: number of deferred envs of the completed call (F_DEVICE_ADVANCE clears the counter)
  // optional second destination of the state planes (16-byte lanes like lo / hi): pinned host memory of a host-side
  // consumer, for which the 32-byte record IS the observation (gym_narde_b200.expand_obs198 decodes it to Box(198))
  void* mirror_lo;
  void* mirror_hi;
  // ... or, instead, ONE 20-byte record per env (NARDE_COMPACT_RECORD_BYTES, layout in include/narde_b200.h: 24 points of
  // 5 bits, off counts, side to move, flags, the result byte's bits, episode steps): 2.6 MB per 131 072 envs instead of
  // 4.2 MB, which is what lets the PCIe writes end before the kernel does
  uint32_t* mirror_compact;
};

// The arguments of a step call over n envs, set by name; the optional parts (deferral, mirrors) stay zero
inline StepFullArgs step_args(int64_t n, int64_t env_base, uint64_t seed, uint64_t step, const uint8_t* dice_in,
                              const int32_t* action_idx, int cap, uint64_t* actions, int32_t* counts, uint8_t* dice_out,
                              uint64_t* chosen, float* reward, uint8_t* done, uint8_t* truncated, int flags,
                              int max_episode_steps, const uint64_t* step_dev) {
  StepFullArgs A = {};
  A.env_base = env_base;
  A.seed = seed;
  A.step = step;
  A.dice_in = dice_in;
  A.action_idx = action_idx;
  A.cap = cap;
  A.actions = cap > 0 ? actions : nullptr;
  A.counts = counts;
  A.dice_out = dice_out;
  A.chosen = chosen;
  A.reward = reward;
  A.done = done;
  A.truncated = truncated;
  A.flags = flags;
  A.max_episode_steps = max_episode_steps;
  A.step_dev = step_dev;
  A.list_cap = n;
  return A;
}

// state (+ result bits) -> the 5 words of the compact host record
NHD void pack_compact(const State& s, int result, uint32_t out[5]) {
  uint64_t a = 0, b = 0;  // points 0..11 / 12..23, 5-bit two's complement each
#pragma unroll
  for (int p = 0; p < 12; p++) {
    a |= (uint64_t)((uint32_t)s.point(p) & 31u) << (5 * p);
    b |= (uint64_t)((uint32_t)s.point(p + 12) & 31u) << (5 * p);
  }
  const uint64_t x0 = a | (b << 60);
  const uint64_t x1 = (b >> 4) | ((uint64_t)(s.off_w() & 15) << 56) | ((uint64_t)(s.off_b() & 15) << 60);
  out[0] = (uint32_t)x0;
  out[1] = (uint32_t)(x0 >> 32);
  out[2] = (uint32_t)x1;
  out[3] = (uint32_t)(x1 >> 32);
  out[4] = (s.turn() == 1 ? 1u : 0u) | ((s.flags() & 7u) << 1) | (((uint32_t)result & 15u) << 4) | ((s.steps() & 0xFFFFu) << 8);
}

// The index of the action to play among `count` legal ones: the caller's action_idx[i] (clamped; or,
// with F_ACTION_FRACTION, a u32 fraction f -> floor(f * count / 2^32)), else Philox-uniform from rnd.
// word = action_idx[i] when the caller gave actions, else the Philox word of the turn
NHD uint32_t pick_from_word(const StepFullArgs& A, uint32_t word, uint32_t count) {
  if (count == 0) return 0;
  if (A.action_idx && !(A.flags & F_ACTION_FRACTION)) {
    int32_t v = (int32_t)word;
    if (v < 0) v = 0;
    if (v >= (int32_t)count) v = (int32_t)count - 1;
    return (uint32_t)v;
  }
  return mulhi32(word, count);
}
NHD uint32_t pick_action_index(const StepFullArgs& A, int64_t i, uint32_t rnd, uint32_t count) {
  return pick_from_word(A, A.action_idx ? (uint32_t)A.action_idx[i] : rnd, count);
}

struct StepFullLocal {  // per-env contributions to the stats vector
  int count;
  int finished, white_win, black_win, mars, ep_len, overflow;
  int clamped;  // the caller's action index was out of range (set by the kernels after complete_env)
  int result;   // bit 0 terminated, bit 1 truncated, bits 2-3 the reward (0, 1, 2): the NARDE_PACK_RESULT byte
};
// One env's contributions added to the stats vector: atomics on the device, plain adds on the host
NHD void stats_add_env(int64_t* stats, const StepFullLocal& L) {
  int v[6] = {L.finished, L.white_win, L.black_win, L.mars, L.ep_len, L.count};
#if defined(__CUDA_ARCH__)
  for (int k = 0; k < 6; k++)
    if (v[k]) atomicAdd(reinterpret_cast<unsigned long long*>(stats + k), (unsigned long long)v[k]);
  if (L.count) atomicMax(reinterpret_cast<long long*>(stats + NARDE_STAT_MAX_ACTIONS), (long long)L.count);
  if (L.overflow) atomicAdd(reinterpret_cast<unsigned long long*>(stats + NARDE_STAT_OVERFLOWS), 1ull);
  if (L.clamped) atomicAdd(reinterpret_cast<unsigned long long*>(stats + NARDE_STAT_CLAMPED_ACTIONS), 1ull);
#else
  for (int k = 0; k < 6; k++) stats[k] += v[k];
  if (L.count > stats[NARDE_STAT_MAX_ACTIONS]) stats[NARDE_STAT_MAX_ACTIONS] = L.count;
  stats[NARDE_STAT_OVERFLOWS] += L.overflow;
  stats[NARDE_STAT_CLAMPED_ACTIONS] += L.clamped;
#endif
}
// SURVEY 8b "Errors": an out-of-range index never raises (the reference's step forfeits silently, narde_env.py:63);
// it is clamped and counted
NHD int index_was_clamped(const StepFullArgs& A, uint32_t word, uint32_t count) {
  if (!A.action_idx || (A.flags & F_ACTION_FRACTION) || count == 0) return 0;
  const int32_t v = (int32_t)word;
  return (v < 0 || v >= (int32_t)count) ? 1 : 0;
}

NHD void step_full_env(State& s, int64_t i, const StepFullArgs& A, StepFullLocal& L) {
  L.count = 0;
  L.finished = L.white_win = L.black_win = L.mars = L.ep_len = L.overflow = L.clamped = 0;
  uint32_t env = (uint32_t)(A.env_base + i);
  if (s.flags() & FLAG_DONE) {  // only reachable without auto-reset: a finished env idles
    if (A.counts) A.counts[i] = 0;
    if (A.dice_out) A.dice_out[2 * i] = A.dice_out[2 * i + 1] = 0;
    if (A.chosen) A.chosen[i] = ACT_EMPTY;
    if (A.reward) A.reward[i] = 0.0f;
    if (A.done) A.done[i] = 1;
    if (A.truncated) A.truncated[i] = 0;
    return;
  }
  U4 rnd = turn_random(A.seed, env, A.step);
  int d1, d2;
  if (A.dice_in) {
    d1 = A.dice_in[2 * i];
    d2 = A.dice_in[2 * i + 1];
  } else {
    d1 = die_from_word(rnd.x);
    d2 = die_from_word(rnd.y);
  }
  int player = s.turn();
  bool first_turn = (s.flags() & (player == 1 ? FLAG_FIRST_W : FLAG_FIRST_B)) != 0;
  Pos P = decode_pos(s, player);

  int count;
  uint64_t* slice = A.actions ? A.actions + (int64_t)i * A.cap : nullptr;
  if (slice) {
    StoreSink sk = {slice, A.cap, 1, 0};
    count = enumerate_turn(P, d1, d2, first_turn, sk);
  } else {
    CountSink ck;
    count = enumerate_turn(P, d1, d2, first_turn, ck);
  }
  L.count = count;
  L.overflow = (slice && count > A.cap) ? 1 : 0;

  uint64_t act = ACT_EMPTY;
  if (count > 0) {
    int idx = (int)pick_action_index(A, i, rnd.z, (uint32_t)count);
    L.clamped = A.action_idx ? index_was_clamped(A, (uint32_t)A.action_idx[i], (uint32_t)count) : 0;
    if (slice && idx < A.cap) {
      act = slice[idx];
    } else {  // not stored: enumerate again and pick the idx-th
      PickSink pk = {idx, 0, ACT_EMPTY};
      enumerate_turn(P, d1, d2, first_turn, pk);
      act = pk.picked;
    }
    apply_action(s, player, act);
  }
  float rew;
  int dn;
  finish_turn(s, player, (A.flags & F_REWARD_MOVER12) ? 1 : 0, &rew, &dn);
  int bits = dn ? DONE_TERMINATED : 0;
  if (!dn && A.max_episode_steps > 0 && (int)s.steps() >= A.max_episode_steps) bits |= DONE_TRUNCATED;
  if (bits) {
    L.finished = 1;
    L.ep_len = (int)s.steps();
    if (dn) {
      if (player == 1)
        L.white_win = 1;
      else
        L.black_win = 1;
      int loser_off = player == 1 ? s.off_b() : s.off_w();
      L.mars = loser_off == 0 ? 1 : 0;
    }
    if (A.flags & F_AUTORESET) s = reset_env(A.seed, env, A.step);
  }
  if (A.counts) A.counts[i] = count;
  if (A.dice_out) {
    A.dice_out[2 * i] = (uint8_t)d1;
    A.dice_out[2 * i + 1] = (uint8_t)d2;
  }
  if (A.chosen) A.chosen[i] = act;
  if (A.reward) A.reward[i] = rew;
  if (A.done) A.done[i] = (bits & DONE_TERMINATED) ? 1 : 0;
  if (A.truncated) A.truncated[i] = (bits & DONE_TRUNCATED) ? 1 : 0;
}

// Outputs of a finished game without auto-reset, which stays as it is: no action, no reward, still terminated
// (under F_ENUMERATE_ONLY the "done" output carries the overflow flag: 0)
NHD void idle_outputs(int64_t i, const StepFullArgs& A) {
  if (A.counts) A.counts[i] = 0;
  if (A.dice_out) A.dice_out[2 * i] = A.dice_out[2 * i + 1] = 0;
  if (A.chosen) A.chosen[i] = ACT_EMPTY;
  if (A.reward) A.reward[i] = 0.0f;
  if (A.done) A.done[i] = (A.flags & F_ENUMERATE_ONLY) ? 0 : 1;
  if (A.truncated) A.truncated[i] = 0;
}

// End-of-turn completion shared by the kernels: apply, termination / reward / switch, auto-reset,
// outputs and per-env stats contributions.
// apply = false: the caller has applied `act` already (the exact kernel, with its rolled-up copy of apply_action)
NHD void complete_env(State& s, int64_t i, const StepFullArgs& A, int player, uint32_t count, uint64_t act, int d1, int d2,
                      StepFullLocal& L, bool apply = true) {
  uint64_t* slice = A.actions ? A.actions + (int64_t)i * A.cap : nullptr;
  L.count = (int)count;
  L.overflow = (slice && (int)count > A.cap) ? 1 : 0;
  L.finished = L.white_win = L.black_win = L.mars = L.ep_len = 0;
  L.result = 0;
  if (A.flags & F_ENUMERATE_ONLY) {  // get_valid_actions: the list and its length only, the state is not touched
    if (A.counts) A.counts[i] = (int32_t)count;
    if (A.chosen) A.chosen[i] = count ? act : ACT_EMPTY;
    if (A.done) A.done[i] = (uint8_t)L.overflow;  // the "done" output carries the overflow flag in this mode
    if (A.dice_out) {  // the turn's dice (Philox, or the caller's echoed): a later pass over the same turn needs them
      A.dice_out[2 * i] = (uint8_t)d1;
      A.dice_out[2 * i + 1] = (uint8_t)d2;
    }
    return;
  }
  if (count && apply) apply_action(s, player, act);
  float rew;
  int dn;
  finish_turn(s, player, (A.flags & F_REWARD_MOVER12) ? 1 : 0, &rew, &dn);
  int bits = dn ? DONE_TERMINATED : 0;
  if (!dn && A.max_episode_steps > 0 && (int)s.steps() >= A.max_episode_steps) bits |= DONE_TRUNCATED;
  if (bits) {
    L.finished = 1;
    L.ep_len = (int)s.steps();
    if (dn) {
      if (player == 1)
        L.white_win = 1;
      else
        L.black_win = 1;
      L.mars = (player == 1 ? s.off_b() : s.off_w()) == 0 ? 1 : 0;
    }
    if (A.flags & F_AUTORESET) s = reset_env(A.seed, (uint32_t)(A.env_base + i), A.step);
  }
  if (A.counts) A.counts[i] = (int32_t)count;
  if (A.dice_out) {
    A.dice_out[2 * i] = (uint8_t)d1;
    A.dice_out[2 * i + 1] = (uint8_t)d2;
  }
  if (A.chosen) A.chosen[i] = count ? act : ACT_EMPTY;
  L.result = bits | ((int)rew << 2);
  if (A.flags & F_PACK_RESULT) {  // one byte per env: bit 0 terminated, bit 1 truncated, bits 2-3 the reward (0, 1, 2)
    if (A.done) A.done[i] = (uint8_t)(bits | ((int)rew << 2));
    return;
  }
  if (A.reward) A.reward[i] = rew;
  if (A.done) A.done[i] = (bits & DONE_TERMINATED) ? 1 : 0;
  if (A.truncated) A.truncated[i] = (bits & DONE_TRUNCATED) ? 1 : 0;
}


// ---- narde_enumerate body -------------------------------------------------------------------
NHD int enumerate_env(const State& s, int d1, int d2, int cap, uint64_t* slice) {
  int player = s.turn();
  bool first_turn = (s.flags() & (player == 1 ? FLAG_FIRST_W : FLAG_FIRST_B)) != 0;
  Pos P = decode_pos(s, player);
  StoreSink sk = {slice, cap, 1, 0};
  return enumerate_turn(P, d1, d2, first_turn, sk);
}

// ---- narde_apply_actions body ---------------------------------------------------------------
NHD void apply_actions_env(State& s, uint64_t act, int flags, float* reward, int* done_bits) {
  if (s.flags() & FLAG_DONE) {
    *reward = 0.0f;
    *done_bits = DONE_TERMINATED;
    return;
  }
  int player = s.turn();
  apply_action(s, player, act);
  if (flags & F_HALF_MOVES_ONLY) {  // Narde.execute_rotated_move only (narde.py:36-56)
    *reward = 0.0f;
    *done_bits = 0;
    return;
  }
  int dn;
  finish_turn(s, player, (flags & F_REWARD_MOVER12) ? 1 : 0, reward, &dn);
  *done_bits = dn ? DONE_TERMINATED : 0;
}

}  // namespace narde
