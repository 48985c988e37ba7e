// hostsim.cpp -- TEST-ONLY host build of the device core (gym_narde_b200/csrc/narde_core.cuh).
//
// The CUDA path's per-environment arithmetic is written as __host__ __device__ functions; this
// file compiles the SAME source with g++ and wraps it in plain loops behind the C-ABI signatures
// of include/narde_b200.h (prefix hs_, HOST pointers), so the rules logic can be checked against
// the oracle in the GPU-less build container.  It is not a CPU fallback: the product package never
// loads it (gym_narde_b200/_cabi.py only opens libnarde_b200.so and fails loudly without CUDA).
#include <stdint.h>
#include <string.h>

#define NARDE_HOSTSIM_HOOKS 1
#include "../../gym_narde_b200/csrc/narde_block.cuh"
#include "../../gym_narde_b200/csrc/narde_deferred.cuh"
#include "../../gym_narde_b200/csrc/narde_env.cuh"

using namespace narde;
namespace narde { int g_hs_force_slow = 0; }
// bit 0: level-2 doubles items are not put in the item table; bit 1: no per-item offset table (recounting emit);
// bit 2: exact phases with a window of 8 candidates; bit 3: exact phases with a team of 128 threads instead of 32
extern "C" void hs_set_force_slow(int v) { narde::g_hs_force_slow = v; }
#ifdef NARDE_PROFILE
namespace narde { ProfCounters g_prof; }
extern "C" void hs_prof_get(long long* out) { memcpy(out, &narde::g_prof, sizeof(narde::g_prof)); }
extern "C" void hs_prof_reset() { memset(&narde::g_prof, 0, sizeof(narde::g_prof)); }
#endif

static State load_state(const void* lo, const void* hi, int64_t i) {
  State s;
  const uint32_t* l = (const uint32_t*)lo + 4 * i;
  const uint32_t* h = (const uint32_t*)hi + 4 * i;
  s.w[0] = l[0]; s.w[1] = l[1]; s.w[2] = l[2]; s.w[3] = l[3];
  s.w[4] = h[0]; s.w[5] = h[1]; s.meta = h[2]; s.aux = h[3];
  return s;
}
static void store_state(void* lo, void* hi, int64_t i, const State& s) {
  uint32_t* l = (uint32_t*)lo + 4 * i;
  uint32_t* h = (uint32_t*)hi + 4 * i;
  l[0] = s.w[0]; l[1] = s.w[1]; l[2] = s.w[2]; l[3] = s.w[3];
  h[0] = s.w[4]; h[1] = s.w[5]; h[2] = s.meta; h[3] = s.aux;
}

static void store_obs198(float* obs198, int64_t i, const State& s) {
  for (int k = 0; k < 99; k++) obs198_pair(s, k, obs198 + 198 * i + 2 * k, obs198 + 198 * i + 2 * k + 1);
}

extern "C" {

int hs_reset_masked(void* lo, void* hi, const uint8_t* mask, int64_t n, int64_t env_base, uint64_t seed,
                    uint64_t step, void*) {
  for (int64_t i = 0; i < n; i++) {
    if (mask && !mask[i]) continue;
    store_state(lo, hi, i, reset_env(seed, (uint32_t)(env_base + i), step));
  }
  return 0;
}
int hs_reset(void* lo, void* hi, int64_t n, int64_t env_base, uint64_t seed, uint64_t step, void* st) {
  return hs_reset_masked(lo, hi, nullptr, n, env_base, seed, step, st);
}

int hs_half_moves(const void* lo, const void* hi, const uint8_t* dice, int64_t n, int player_override,
                  uint8_t* moves, int32_t* counts, void*) {
  for (int64_t i = 0; i < n; i++) {
    State s = load_state(lo, hi, i);
    counts[i] = half_moves_env(s, dice + 4 * i, player_override, moves + i * 96 * 2);
  }
  return 0;
}

int hs_step_ref(void* lo, void* hi, const uint8_t* dice, const int32_t* codes, int64_t n,
                int32_t max_episode_steps, int32_t* o24, int32_t* reward, uint8_t* done, uint8_t* truncated, void*) {
  for (int64_t i = 0; i < n; i++) {
    State s = load_state(lo, hi, i);
    int r, d;
    step_ref_env(s, dice[2 * i], dice[2 * i + 1], codes[2 * i], codes[2 * i + 1], max_episode_steps, &r, &d);
    store_state(lo, hi, i, s);
    if (o24) obs24(s, s.turn(), o24 + 24 * i);
    if (reward) reward[i] = r;
    if (done) done[i] = (d & DONE_TERMINATED) ? 1 : 0;
    if (truncated) truncated[i] = (d & DONE_TRUNCATED) ? 1 : 0;
  }
  return 0;
}

int hs_enumerate(const void* lo, const void* hi, const uint8_t* dice, int64_t n, int32_t cap, uint64_t* actions,
                 int32_t* counts, uint8_t* overflow, void*) {
  for (int64_t i = 0; i < n; i++) {
    State s = load_state(lo, hi, i);
    int c = enumerate_env(s, dice[2 * i], dice[2 * i + 1], cap, actions + i * (int64_t)cap);
    counts[i] = c;
    if (overflow) overflow[i] = c > cap;
  }
  return 0;
}

int hs_obs198(const void* lo, const void* hi, int64_t n, float* obs, void*) {
  for (int64_t i = 0; i < n; i++) {
    State s = load_state(lo, hi, i);
    store_obs198(obs, i, s);
  }
  return 0;
}
int hs_obs24(const void* lo, const void* hi, int64_t n, int32_t* o, void*) {
  for (int64_t i = 0; i < n; i++) {
    State s = load_state(lo, hi, i);
    obs24(s, s.turn(), o + 24 * i);
  }
  return 0;
}

int hs_step_full(void* lo, void* hi, int64_t n, int64_t env_base, uint64_t seed, uint64_t step, const uint8_t* dice_in,
                 const int32_t* action_idx, int32_t cap, uint64_t* actions, int32_t* counts, uint8_t* dice_out,
                 uint64_t* chosen, float* obs198, float* reward, uint8_t* done, uint8_t* truncated, int64_t* stats,
                 int32_t flags, int32_t max_episode_steps, void*) {
  const StepFullArgs A = step_args(n, env_base, seed, step, dice_in, action_idx, cap, actions, counts, dice_out, chosen, reward,
                                   done, truncated, flags, max_episode_steps, nullptr);
  for (int64_t i = 0; i < n; i++) {
    State s = load_state(lo, hi, i);
    StepFullLocal L;
    step_full_env(s, i, A, L);
    store_state(lo, hi, i, s);
    if (stats) stats_add_env(stats, L);
    if (obs198) store_obs198(obs198, i, s);
  }
  return 0;
}

int hs_step_full_v2(void* lo, void* hi, int64_t n, int64_t env_base, uint64_t seed, uint64_t step, const uint8_t* dice_in,
                    const int32_t* action_idx, int32_t cap, uint64_t* actions, int32_t* counts, uint8_t* dice_out,
                    uint64_t* chosen, float* obs198, float* reward, uint8_t* done, uint8_t* truncated, int64_t* stats,
                    int32_t flags, int32_t max_episode_steps, int32_t* workspace, void*);
// narde_enumerate_fast: the fused-step phases in enumerate-only mode (flag 64)
int hs_enumerate_fast(const void* lo, const void* hi, const uint8_t* dice, int64_t n, int32_t cap, uint64_t* actions,
                      int32_t* counts, uint8_t* overflow, int32_t* workspace, void*) {
  return hs_step_full_v2(const_cast<void*>(lo), const_cast<void*>(hi), n, 0, 0, 0, dice, nullptr, cap, actions, counts, nullptr,
                         nullptr, nullptr, nullptr, overflow, nullptr, nullptr, 64, 0, workspace, nullptr);
}

}  // extern "C"

static int64_t g_small_batch = 16384;
extern "C" void hs_set_small_batch(int64_t v) { g_small_batch = v; }
static int g_tile = 128;   // large-batch tile, as in narde_kernels.cu: 128 envs on 128 threads (default) or 64 on 128
extern "C" void hs_set_tile(int v) { g_tile = v; }

// CTA-cooperative step (narde_block.cuh) emulated phase by phase: every phase runs for all tids
// of a block before the next one starts, which is what __syncthreads() guarantees on the GPU.
template <int BLK, bool DEFER, int NT = BLK>
static void step_full_v2_host(void* lo, void* hi, int64_t n, const StepFullArgs& A, float* obs198, int64_t* stats) {
  typedef BlockStep<BLK, DEFER, NT> BS;
  static BlockShared<BLK, NT> sh;
  for (int64_t row0 = 0; row0 < n; row0 += BLK) {
    for (int t = 0; t < NT; t++) {
      bool valid = t < BLK && row0 + t < n;
      State s;
      if (valid) s = load_state(lo, hi, row0 + t);
      BS::ph_load(t, sh, valid, s, row0 + t, A);
    }
    // NOTE: phases fused between two barriers on the GPU are emulated in DESCENDING tid order as
    // well as ascending elsewhere, so that a read-after-write hazard inside a fused pair shows up
    for (int t = 0; t < NT; t++) BS::ph_scan_serial(t, sh, 0x3u);
    for (int t = NT - 1; t >= 0; t--) BS::ph_item_bases(t, sh);
    for (int t = 0; t < NT; t++) BS::ph_rows(t, sh);
    for (int t = 0; t < NT; t++) BS::ph_scan_serial(t, sh, 0x2u);
    for (int t = 0; t < NT; t++) BS::ph_l2_bases(t, sh);
    for (int t = NT - 1; t >= 0; t--) BS::ph_count(t, sh);
    for (int t = 0; t < NT; t++) { BS::ph_env_totals(t, sh); if (DEFER) BS::ph_defer_push(t, sh, t < BLK && row0 + t < n, row0 + t, A); }
    for (int t = 0; t < NT; t++) BS::ph_scan_serial(t, sh, 0xFu);
    for (int t = NT - 1; t >= 0; t--) BS::ph_env_bases(t, sh);
    for (int t = 0; t < NT; t++) BS::ph_emit(t, sh, row0, A);
    for (int t = 0; t < BLK; t++) {
      bool valid = row0 + t < n;
      StepFullLocal L;
      BS::ph_finish(t, sh, valid, row0 + t, A, L);
      if (!valid || sh.defer[t]) continue;
      store_state(lo, hi, row0 + t, sh.st[t]);
      if (stats) stats_add_env(stats, L);
      if (obs198) store_obs198(obs198, row0 + t, sh.st[t]);
    }
  }
}

// CTA-per-env exact kernel (narde_deferred.cuh): the same driver, a phase = a loop over the team's tids
// (descending, so that a read-after-write hazard between the threads of one phase shows up)
template <int NT>
struct HostTeamExec {
  template <class F>
  void run(F&& f) {
    for (int t = NT - 1; t >= 0; t--) f(t);
  }
  void mark(int) {}
};
template <int NT>   // the device kernel's teams: the CTA (128 threads) for a short list, one warp per env for a long one
static void step_deferred_host(void* lo, void* hi, const StepFullArgs& A, float* obs198, int64_t* stats) {
  typedef ExactStep<NT> ES;
  static ExactSharedT<NT> sh;
  HostTeamExec<NT> ex;
  for (int q = 0; q < A.defer_count[0]; q++) {
    int64_t i = A.defer_list[q] - 1;   // entries are env index + 1 (0 = not published, narde_block.cuh ph_defer_push)
    State s = load_state(lo, hi, i);
    ES::solve(ex, sh, s, i, A);
    StepFullLocal L;
    State st = sh.st;
    ES::complete(sh, st, i, A, L);
    store_state(lo, hi, i, st);
    if (stats) stats_add_env(stats, L);
    if (obs198) store_obs198(obs198, i, st);
  }
}

extern "C" {
int hs_step_full_v2(void* lo, void* hi, int64_t n, int64_t env_base, uint64_t seed, uint64_t step, const uint8_t* dice_in,
                    const int32_t* action_idx, int32_t cap, uint64_t* actions, int32_t* counts, uint8_t* dice_out,
                    uint64_t* chosen, float* obs198, float* reward, uint8_t* done, uint8_t* truncated, int64_t* stats,
                    int32_t flags, int32_t max_episode_steps, int32_t* workspace, void*) {
  StepFullArgs A = step_args(n, env_base, seed, step, dice_in, action_idx, cap, actions, counts, dice_out, chosen, reward, done,
                             truncated, flags, max_episode_steps, nullptr);
  if (workspace) {
    for (int k = 0; k < 8; k++) workspace[k] = 0;   // NARDE_WORKSPACE_INTS layout (include/narde_b200.h)
    A.defer_count = workspace;
    A.defer_list = workspace + 8;
  }
  // same dispatch as narde_step_full: one-warp CTAs of 32 envs for small batches (g_small_batch can be
  // lowered by the tests so that both tile sizes are exercised on small inputs)
  if (n <= g_small_batch) {
    if (workspace)
      step_full_v2_host<32, true>(lo, hi, n, A, obs198, stats);
    else
      step_full_v2_host<32, false>(lo, hi, n, A, obs198, stats);
  } else if (g_tile == 64) {
    if (workspace)
      step_full_v2_host<64, true, 128>(lo, hi, n, A, obs198, stats);
    else
      step_full_v2_host<64, false, 128>(lo, hi, n, A, obs198, stats);
  } else if (workspace) {
    step_full_v2_host<128, true>(lo, hi, n, A, obs198, stats);
  } else {
    step_full_v2_host<128, false>(lo, hi, n, A, obs198, stats);
  }
  if (workspace) {
    if (g_hs_force_slow & 8) step_deferred_host<128>(lo, hi, A, obs198, stats);
    else step_deferred_host<32>(lo, hi, A, obs198, stats);
  }
  return 0;
}

int hs_apply_actions(void* lo, void* hi, const uint64_t* acts, int64_t n, int32_t flags, float* reward, uint8_t* done,
                     void*) {
  for (int64_t i = 0; i < n; i++) {
    State s = load_state(lo, hi, i);
    float r; int d;
    apply_actions_env(s, acts[i], flags, &r, &d);
    store_state(lo, hi, i, s);
    if (reward) reward[i] = r;
    if (done) done[i] = (uint8_t)d;
  }
  return 0;
}

// instrumentation for design decisions (tests/bench only)
int hs_block_irrelevant(const void* lo, const void* hi, const uint8_t* dice, int64_t n, uint8_t* out) {
  for (int64_t i = 0; i < n; i++) {
    State s = load_state(lo, hi, i);
    Pos P = decode_pos(s, s.turn());
    out[i] = block_rule_irrelevant(P, dice[2 * i], dice[2 * i + 1]);
  }
  return 0;
}
}
