// narde_kernels.cu -- sm_100a kernels + the C ABI of include/narde_b200.h.
//
// Layout in HBM: two SoA planes lo[N], hi[N] of 16-byte lanes (one uint4 per env per plane) so a
// warp loads/stores 512 contiguous bytes per plane.  One thread owns one environment for the
// integer rules work (registers only); Box(198) rows are written by the whole CTA from a
// shared-memory copy of the CTA's states so that global stores are contiguous 16-byte lanes.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "../../include/narde_b200.h"
// NARDE_DEBUG_HOOKS (tools only: `python -m gym_narde_b200.build --debug-hooks` -> libnarde_b200_debug.so) compiles
// in the A/B timing switches and the per-CTA phase clocks; the product library has neither.
#ifdef NARDE_DEBUG_HOOKS
namespace narde { __device__ int g_dbg_flags = 0; }
#endif
#include "narde_block.cuh"
#include "narde_deferred.cuh"
#include "narde_env.cuh"

using namespace narde;

namespace {

constexpr int kThreads = 128;
// envs (= threads) per CTA of the fused step: 128 for large batches; one-warp CTAs of 32 envs when the batch
// cannot fill the machine otherwise (4096 envs: 128 CTAs instead of 32; measured 0.081 -> 0.053 ms/step)
int g_variant = 0;
bool g_early = true;  // NARDE_LATE_TRIGGER=1 in the environment: the dependent is triggered after the count phase for every batch size (A/B timing)
int g_tile = 128;  // envs per CTA of the large-batch fused step: 128 (a thread per env) or 64 on 128 threads (NARDE_TILE=64 in the environment; measured equal within noise: the step is bound by the CTA's chain of phases, not by resident warps)
int64_t kSmallBatch = 16384;  // (NARDE_SMALL_BATCH in the environment overrides it: A/B timing of the two tiles)
constexpr int kDeferredThreads = 128;  // exact-doubles kernel: four warps per CTA, one env per warp at a time (7 KB of shared memory each)
constexpr int kDeferredGrid = 148 * 8;  // 8 CTAs per SM (64 registers, 27 KB)
constexpr int kDeferredGridEarly = 148 * 4;  // early-trigger launches: these CTAs sit beside the main kernel's last wave

__device__ __forceinline__ State ld_state(const uint4* __restrict__ lo, const uint4* __restrict__ hi, int64_t i) {
  uint4 a = lo[i], b = hi[i];
  State s;
  s.w[0] = a.x; s.w[1] = a.y; s.w[2] = a.z; s.w[3] = a.w;
  s.w[4] = b.x; s.w[5] = b.y; s.meta = b.z; s.aux = b.w;
  return s;
}
__device__ __forceinline__ void st_state(uint4* __restrict__ lo, uint4* __restrict__ hi, int64_t i, const State& s) {
  lo[i] = make_uint4(s.w[0], s.w[1], s.w[2], s.w[3]);
  hi[i] = make_uint4(s.w[4], s.w[5], s.meta, s.aux);
}

// CTA-cooperative Box(198) writer (README.md:44-102).  sm[] holds the CTA's states, rows
// [row0, row0+rows).  Work item = (env, point): one board byte gives the WHITE and the BLACK
// 4-float encodings of that point through a 16-entry shared-memory table (n -> [n>=1, n>=2, n>=3,
// (n-3)/2]); rows are 792 B, so 8-byte stores are always aligned.  lut must be filled
// (obs_lut_init) and the CTA synchronised before the call.
__device__ __forceinline__ void obs_lut_init(float4* lut) {
  if (threadIdx.x < 16) {
    int n = threadIdx.x;
    lut[n] = make_float4(n >= 1 ? 1.0f : 0.0f, n >= 2 ? 1.0f : 0.0f, n >= 3 ? 1.0f : 0.0f,
                         n > 3 ? (float)(n - 3) * 0.5f : 0.0f);
  }
}
__device__ __forceinline__ void write_obs198_cta(const State* sm, const float4* lut, int rows, int64_t row0,
                                                 float* __restrict__ obs, const uint32_t* skip = nullptr,
                                                 int tid = (int)threadIdx.x, int nthreads = (int)blockDim.x) {
  float* base = obs + row0 * 198;
  // rows are 792 B: in a 16-byte aligned row the WHITE block (4 floats per point from offset 0) is made of
  // aligned 16-byte lanes and the BLACK block (from offset 392 B) of 8-byte ones; in the next row it is the
  // other way round -- one 16-byte and two 8-byte stores per (env, point) instead of four 8-byte stores.
  // A thread keeps ONE point (24 threads per env; its state word and byte shift are loop constants) and takes, per
  // trip, one row of each alignment, so the warp never diverges on the store pattern and there is no division in
  // the loop (the item loop it replaces spent 51 instructions per (env, point): 17 % of the kernel's instructions).
  const int ngrp = nthreads / 24, grp = tid / 24, pt = tid - grp * 24;
  if (grp < ngrp) {
    const int wi = pt >> 2, shf = (pt & 3) * 8;
    const int pa = ((reinterpret_cast<uintptr_t>(base) & 15u) == 0) ? 0 : 1;  // parity of the 16-byte aligned rows
    for (int j = grp; 2 * j < rows; j += ngrp) {
      const int eA = 2 * j + pa, eB = 2 * j + 1 - pa;
      if (eA < rows && !(skip && skip[eA])) {  // (skip: row written by the deferred kernel)
        const int v = (int)(int8_t)(sm[eA].w[wi] >> shf);
        const float4 fw = lut[v > 0 ? v : 0], fb = lut[v < 0 ? -v : 0];
        float* rw = base + eA * 198 + 4 * pt;
        float* rb = rw + 98;
        *reinterpret_cast<float4*>(rw) = fw;
        reinterpret_cast<float2*>(rb)[0] = make_float2(fb.x, fb.y);
        reinterpret_cast<float2*>(rb)[1] = make_float2(fb.z, fb.w);
      }
      if (eB < rows && !(skip && skip[eB])) {
        const int v = (int)(int8_t)(sm[eB].w[wi] >> shf);
        const float4 fw = lut[v > 0 ? v : 0], fb = lut[v < 0 ? -v : 0];
        float* rw = base + eB * 198 + 4 * pt;
        float* rb = rw + 98;
        reinterpret_cast<float2*>(rw)[0] = make_float2(fw.x, fw.y);
        reinterpret_cast<float2*>(rw)[1] = make_float2(fw.z, fw.w);
        *reinterpret_cast<float4*>(rb) = fb;
      }
    }
  }
  for (int e = tid; e < rows; e += nthreads) {  // bars (always empty: no hitting, narde.py:71), off / 15, side to move
    if (skip && skip[e]) continue;
    const State& s = sm[e];
    float* r = base + e * 198;
    *reinterpret_cast<float2*>(r + 96) = make_float2(0.0f, off15(s.off_w()));
    *reinterpret_cast<float2*>(r + 194) = make_float2(0.0f, off15(s.off_b()));
    *reinterpret_cast<float2*>(r + 196) = s.turn() == 1 ? make_float2(1.0f, 0.0f) : make_float2(0.0f, 1.0f);
  }
}

__global__ void __launch_bounds__(kThreads) k_reset(uint4* lo, uint4* hi, const uint8_t* mask, int64_t n, int64_t env_base,
                                                   uint64_t seed, uint64_t step) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (mask && !mask[i]) return;
  st_state(lo, hi, i, reset_env(seed, (uint32_t)(env_base + i), step));
}

__global__ void __launch_bounds__(kThreads) k_half_moves(const uint4* lo, const uint4* hi, const uint8_t* dice, int64_t n,
                                                        int player_override, uint8_t* moves, int32_t* counts) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  State s = ld_state(lo, hi, i);
  uint32_t d4 = reinterpret_cast<const uint32_t*>(dice)[i];
  uint8_t dd[4] = {(uint8_t)(d4 & 0xFF), (uint8_t)((d4 >> 8) & 0xFF), (uint8_t)((d4 >> 16) & 0xFF), (uint8_t)(d4 >> 24)};
  counts[i] = half_moves_env(s, dd, player_override, moves + i * (NARDE_MAX_HALF_MOVES * 2));
}

__global__ void __launch_bounds__(kThreads) k_step_ref(uint4* lo, uint4* hi, const uint8_t* dice, const int32_t* codes, int64_t n,
                                                      int max_episode_steps, int32_t* o24, int32_t* reward, uint8_t* done,
                                                      uint8_t* truncated) {
  __shared__ State sm[kThreads];
  int64_t row0 = (int64_t)blockIdx.x * blockDim.x;
  int64_t i = row0 + threadIdx.x;
  if (i < n) {
    State s = ld_state(lo, hi, i);
    uint16_t d2 = reinterpret_cast<const uint16_t*>(dice)[i];
    int2 c = reinterpret_cast<const int2*>(codes)[i];
    int r, dn;
    step_ref_env(s, d2 & 0xFF, d2 >> 8, c.x, c.y, max_episode_steps, &r, &dn);
    st_state(lo, hi, i, s);
    if (reward) reward[i] = r;
    if (done) done[i] = (dn & DONE_TERMINATED) ? 1 : 0;
    if (truncated) truncated[i] = (dn & DONE_TRUNCATED) ? 1 : 0;
    sm[threadIdx.x] = s;
  }
  if (!o24) return;
  __syncthreads();
  int rows = (int)min((int64_t)blockDim.x, n - row0);
  // narde_env.py:24-25: 24 int32 per env, written as contiguous words by the CTA
  int32_t* base = o24 + row0 * 24;
  for (int j = threadIdx.x; j < rows * 24; j += blockDim.x) {
    int e = j / 24, k = j - e * 24;
    const State& s = sm[e];
    int v = s.turn() == 1 ? s.point(k) : -s.point(k < 12 ? k + 12 : k - 12);
    base[j] = v;
  }
}

__global__ void __launch_bounds__(kThreads) k_enumerate(const uint4* lo, const uint4* hi, const uint8_t* dice, int64_t n, int cap,
                                                       uint64_t* actions, int32_t* counts, uint8_t* overflow) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  State s = ld_state(lo, hi, i);
  uint16_t d2 = reinterpret_cast<const uint16_t*>(dice)[i];
  int c = 0;
  if (!(s.flags() & FLAG_DONE)) c = enumerate_env(s, d2 & 0xFF, d2 >> 8, cap, actions + i * (int64_t)cap);
  counts[i] = c;
  if (overflow) overflow[i] = c > cap ? 1 : 0;
}

__global__ void __launch_bounds__(kThreads) k_step_full(uint4* lo, uint4* hi, int64_t n, StepFullArgs A_in, float* obs198, int64_t* stats) {
  StepFullArgs A = A_in;
  if (A.step_dev) A.step = *A.step_dev;
  __shared__ State sm[kThreads];
  int64_t row0 = (int64_t)blockIdx.x * blockDim.x;
  int64_t i = row0 + threadIdx.x;
  StepFullLocal L;
  L.count = L.finished = L.white_win = L.black_win = L.mars = L.ep_len = L.overflow = L.clamped = L.result = 0;
  if (i < n) {
    State s = ld_state(lo, hi, i);
    step_full_env(s, i, A, L);
    st_state(lo, hi, i, s);
    if (A.mirror_lo) st_state((uint4*)A.mirror_lo, (uint4*)A.mirror_hi, i, s);
    sm[threadIdx.x] = s;
  }
  if (stats) {
    // warp-level reduction, one atomic per warp per slot that is non-zero
    unsigned full = 0xFFFFFFFFu;
    int v[6] = {L.finished, L.white_win, L.black_win, L.mars, L.ep_len, L.count};
    int mx = L.count, ov = L.overflow, cl = L.clamped;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
      for (int k = 0; k < 6; k++) v[k] += __shfl_xor_sync(full, v[k], o);
      mx = max(mx, __shfl_xor_sync(full, mx, o));
      ov += __shfl_xor_sync(full, ov, o);
      cl += __shfl_xor_sync(full, cl, o);
    }
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
      for (int k = 0; k < 6; k++)
        if (v[k]) atomicAdd(reinterpret_cast<unsigned long long*>(stats + k), (unsigned long long)v[k]);
      if (mx) atomicMax(reinterpret_cast<long long*>(stats + NARDE_STAT_MAX_ACTIONS), (long long)mx);
      if (ov) atomicAdd(reinterpret_cast<unsigned long long*>(stats + NARDE_STAT_OVERFLOWS), (unsigned long long)ov);
      if (cl) atomicAdd(reinterpret_cast<unsigned long long*>(stats + NARDE_STAT_CLAMPED_ACTIONS), (unsigned long long)cl);
    }
  }
  if (!obs198) return;
  __shared__ float4 lut[16];
  obs_lut_init(lut);
  __syncthreads();
  int rows = (int)min((int64_t)blockDim.x, n - row0);
  write_obs198_cta(sm, lut, rows, row0, obs198);
}

// The turn when the action is already known (the greedy actor: the lists were enumerated and scored a moment ago):
// apply choice[i] of the stored list -- or act_override[i] when it is not 0 (an action beyond the stored capacity,
// found by the side-batch pass; consumed and cleared here) -- then exactly the fused step's completion: termination,
// reward, player switch, truncation, auto-reset, outputs, statistics, Box(198).  A thread per env, no enumeration:
// the second full pass over the position that narde_step_full(action_idx) makes is not needed.
__global__ void __launch_bounds__(kThreads) k_step_chosen(uint4* lo, uint4* hi, int64_t n, StepFullArgs A_in,
                                                         const uint64_t* actions, const int32_t* counts, uint64_t* act_override,
                                                         float* obs198, int64_t* stats) {
  StepFullArgs A = A_in;
  if (A.step_dev) A.step = *A.step_dev;
  __shared__ State sm[kThreads];
  __shared__ float4 lut[16];
  obs_lut_init(lut);
  const int64_t row0 = (int64_t)blockIdx.x * blockDim.x, i = row0 + threadIdx.x;
  StepFullLocal L;
  L.count = L.finished = L.white_win = L.black_win = L.mars = L.ep_len = L.overflow = L.clamped = L.result = 0;
  if (i < n) {
    State s = ld_state(lo, hi, i);
    if (s.flags() & FLAG_DONE) {  // a finished game without auto-reset stays as it is (BlockStep::ph_finish, K_DONE)
      if (A.chosen) A.chosen[i] = ACT_EMPTY;
      if (A.reward) A.reward[i] = 0.0f;
      if (A.done) A.done[i] = 1;
      if (A.truncated) A.truncated[i] = 0;
    } else {
      const int count = counts[i];
      uint64_t act = ACT_EMPTY;
      if (count > 0) {
        int idx = A.action_idx[i];
        idx = idx < 0 ? 0 : idx < count ? idx : count - 1;
        const uint64_t over = act_override ? act_override[i] : 0ull;
        act = over ? over : actions[i * (int64_t)A.cap + (idx < A.cap ? idx : A.cap - 1)];
      }
      if (act_override && act_override[i]) act_override[i] = 0ull;
      const uint16_t d2 = reinterpret_cast<const uint16_t*>(A.dice_in)[i];
      // (A.counts / A.dice_out are NULL: counts, dice and lists are the enumeration's outputs and stay as they are)
      complete_env(s, i, A, s.turn(), (uint32_t)count, act, d2 & 0xFF, d2 >> 8, L);
      L.overflow = count > A.cap ? 1 : 0;
      L.clamped = index_was_clamped(A, (uint32_t)A.action_idx[i], (uint32_t)count);
      st_state(lo, hi, i, s);
    }
    sm[threadIdx.x] = s;
  }
  if (stats) {
    unsigned full = 0xFFFFFFFFu;
    int v[6] = {L.finished, L.white_win, L.black_win, L.mars, L.ep_len, L.count};
    int mx = L.count, ov = L.overflow, cl = L.clamped;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
      for (int k = 0; k < 6; k++) v[k] += __shfl_xor_sync(full, v[k], o);
      mx = max(mx, __shfl_xor_sync(full, mx, o));
      ov += __shfl_xor_sync(full, ov, o);
      cl += __shfl_xor_sync(full, cl, o);
    }
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
      for (int k = 0; k < 6; k++)
        if (v[k]) atomicAdd(reinterpret_cast<unsigned long long*>(stats + k), (unsigned long long)v[k]);
      if (mx) atomicMax(reinterpret_cast<long long*>(stats + NARDE_STAT_MAX_ACTIONS), (long long)mx);
      if (ov) atomicAdd(reinterpret_cast<unsigned long long*>(stats + NARDE_STAT_OVERFLOWS), (unsigned long long)ov);
      if (cl) atomicAdd(reinterpret_cast<unsigned long long*>(stats + NARDE_STAT_CLAMPED_ACTIONS), (unsigned long long)cl);
    }
  }
  if (!obs198) return;
  __syncthreads();
  const int rows = (int)min((int64_t)blockDim.x, n - row0);
  write_obs198_cta(sm, lut, rows, row0, obs198);
}

// Debug aid (NARDE_DEBUG_HOOKS builds only): per-CTA phase timestamps (clock64) when a buffer was registered
// through narde_debug_set_clock_buffer; [block][16] u64.
#ifdef NARDE_DEBUG_HOOKS
__device__ unsigned long long* g_dbg_clk = nullptr;
__device__ unsigned g_dbg_stagger_ns = 0;
#define PHASE_MARK(k)                                                                  \
  do {                                                                                 \
    if (g_dbg_clk && threadIdx.x == 0) g_dbg_clk[(size_t)blockIdx.x * 16 + (k)] = clock64(); \
  } while (0)
__device__ __forceinline__ unsigned long long dbg_globaltimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
// wall-clock (ns, one timer for the whole GPU) marks: rows [0, 2048) slots 10/11 = a main CTA's start / end,
// rows [3072 + block) slots 0..4 = a CTA of the exact kernel (tools/timeline_probe.py)
#define GT_MARK(row, k)                                                                          \
  do {                                                                                           \
    if (g_dbg_clk && threadIdx.x == 0) g_dbg_clk[(size_t)(row) * 16 + (k)] = dbg_globaltimer();  \
  } while (0)
#else
#define PHASE_MARK(k) do { } while (0)
#define GT_MARK(row, k) do { } while (0)
#endif

// Fused full-rules step, CTA-cooperative (narde_block.cuh): the phases run with a CTA barrier
// between them; everything between the state load and the Box(198) store stays in shared memory.
// BLK envs per CTA, NT threads.  <64, ., 128> is the large-batch tile: the kernel is latency-bound (a warp issues once
// in ~8 cycles) and shared memory holds ~350 B per env, so with a thread per env an SM tops out at 20 warps; two
// threads per env and a 64-register budget (8 CTAs of 128 threads) give it 32.
// MINB: CTAs per SM the register budget is cut for (65536 / (NT * MINB) registers per thread).
template <int BLK, bool DEFER, int NT, int MINB>
__global__ void __launch_bounds__(NT, MINB) k_step_full_v2(uint4* lo, uint4* hi, int64_t n, StepFullArgs A_in, float* obs198,
                                                           int64_t* stats) {
  typedef BlockStep<BLK, DEFER, NT> BS;
  StepFullArgs A = A_in;
  if (A.step_dev) A.step = *A.step_dev + ((A.flags & F_DEVICE_ADVANCE) ? 1u : 0u);
  __shared__ BlockShared<BLK, NT> sh;
  const int tid = threadIdx.x;
  const int64_t row0 = (int64_t)blockIdx.x * BLK;
  const int64_t i = row0 + tid;
  const bool valid = (NT == BLK || tid < BLK) && i < n;
  State s;
  PHASE_MARK(0);
  GT_MARK(blockIdx.x, 10);
  // Programmatic dependent launch, large batches: the exact kernel may become resident once every main CTA has
  // STARTED (it then warms its code up and waits for the list, see k_step_deferred)
  if (DEFER && A.early_trigger) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
#ifdef NARDE_DEBUG_HOOKS
  // timing experiment: de-phase the first wave (its CTAs start together and stay in lock-step: every phase of every CTA
  // hits the same unit at the same time); slot k of an SM starts k * g_dbg_stagger_ns later
  if (g_dbg_stagger_ns && blockIdx.x < 148 * 5) __nanosleep((blockIdx.x / 148) * g_dbg_stagger_ns);
#endif
  // The caller's action words of this CTA (BLK x 4 B, contiguous) come in as ONE bulk asynchronous copy into
  // shared memory.  When the buffer is pinned host memory (zero-copy step_host) that is one PCIe read of 512 B
  // per CTA instead of a 32-byte read per warp sector: the host step was bound by the NUMBER of small reads.
  const int cta_rows = (int)((n - row0) < (int64_t)BLK ? (n - row0) : (int64_t)BLK);
  const bool bulk_words = A.action_idx != nullptr && (cta_rows & 3) == 0 &&
                          ((reinterpret_cast<uintptr_t>(A.action_idx + row0) & 15u) == 0);
  if (bulk_words && tid == 0) {
    const uint32_t bar = (uint32_t)__cvta_generic_to_shared(&sh.rnd_bar);
    const uint32_t dst = (uint32_t)__cvta_generic_to_shared(sh.rnd);
    const uint32_t bytes = (uint32_t)cta_rows * 4u;
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(A.action_idx + row0), "r"(bytes), "r"(bar)
                 : "memory");
  }
  if (valid) s = ld_state(lo, hi, i);
  BS::ph_load(tid, sh, valid, s, i, A, bulk_words);
  __syncthreads();
  PHASE_MARK(1);
  BS::ph_scan_serial(tid, sh, 0x3u);
  __syncthreads();
  BS::ph_item_bases(tid, sh);
  __syncthreads();
  PHASE_MARK(2);
  BS::ph_rows(tid, sh);
  __syncthreads();
  PHASE_MARK(3);
  BS::ph_scan_serial(tid, sh, 0x2u);
  __syncthreads();
  BS::ph_l2_bases(tid, sh);
  __syncthreads();
  PHASE_MARK(4);
  BS::ph_count(tid, sh);
  __syncthreads();
  PHASE_MARK(5);
  BS::ph_env_totals(tid, sh);
  if (DEFER) {
    BS::ph_defer_push(tid, sh, valid, i, A);
    if (valid && sh.defer[tid]) __threadfence();  // (only a thread that pushed an entry: a fence per thread cost 1.8 % of the samples)
  }
  __syncthreads();
  // Publication of this CTA's list entries: the barrier above orders every thread's pushes before thread 0's
  // release-add; k_step_deferred acquires "all main CTAs have arrived" before it reads the list (the visibility
  // of a primary grid's writes is otherwise only guaranteed after griddepcontrol.wait, i.e. after its completion).
  if (DEFER && tid == 0) asm volatile("red.release.gpu.global.add.s32 [%0], 1;" ::"l"(A.arrivals) : "memory");
  // Programmatic dependent launch, small batches (one wave): k_step_deferred may start as soon as every CTA is past
  // this point, i.e. while the action lists and Box(198) rows of the other envs are still being written.
  if (!A.early_trigger) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  BS::ph_scan_serial(tid, sh, 0xFu);
  __syncthreads();
  BS::ph_env_bases(tid, sh);
  __syncthreads();
  PHASE_MARK(6);
  if (bulk_words) {  // the action words have landed (long ago): the wait makes the async-proxy writes visible
    const uint32_t bar = (uint32_t)__cvta_generic_to_shared(&sh.rnd_bar);
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAITW_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], 0;\n\t"
        "@p bra DONEW_%=;\n\t"
        "bra WAITW_%=;\n\t"
        "DONEW_%=:\n\t}" ::"r"(bar)
        : "memory");
  }
  BS::ph_emit(tid, sh, row0, A);
  __syncthreads();
  PHASE_MARK(7);
  StepFullLocal L;
  BS::ph_finish(tid, sh, valid, i, A, L);
  __syncthreads();
  PHASE_MARK(8);
  // deferred envs belong to k_step_deferred, which may already be running: never store their state here
  if (valid && !sh.defer[tid] && !(A.flags & F_ENUMERATE_ONLY)) {
    st_state(lo, hi, i, sh.st[tid]);
    if (A.mirror_lo) st_state((uint4*)A.mirror_lo, (uint4*)A.mirror_hi, i, sh.st[tid]);  // posted PCIe writes (zero-copy)
  }
  if (A.mirror_compact && !(A.flags & F_ENUMERATE_ONLY)) {
    // the 20-byte host records of this CTA, packed into shared memory (the scan scratch is dead by now) and written as
    // contiguous words: a warp's store is 128 contiguous bytes of (pinned host) memory; records of deferred envs are
    // the exact kernel's to write
    uint32_t* stg = &sh.part[0][0];
    static_assert(sizeof(sh.part) + sizeof(sh.base) >= 5 * BLK * sizeof(uint32_t), "staging area of the compact records");
    if (valid && !sh.defer[tid]) {
      uint32_t r[5];
      pack_compact(sh.st[tid], L.result, r);
#pragma unroll
      for (int k = 0; k < 5; k++) stg[tid * 5 + k] = r[k];
    }
    __syncthreads();
    const int nrec = (int)min((int64_t)BLK, n - row0);
    for (int w = tid; w < nrec * 5; w += NT)
      if (!sh.defer[w / 5]) A.mirror_compact[row0 * 5 + w] = stg[w];
  }
  if (stats) {
    unsigned full = 0xFFFFFFFFu;
    int v[6] = {L.finished, L.white_win, L.black_win, L.mars, L.ep_len, L.count};
    int mx = L.count, ov = L.overflow, cl = L.clamped;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
      for (int k = 0; k < 6; k++) v[k] += __shfl_xor_sync(full, v[k], o);
      mx = max(mx, __shfl_xor_sync(full, mx, o));
      ov += __shfl_xor_sync(full, ov, o);
      cl += __shfl_xor_sync(full, cl, o);
    }
    if ((tid & 31) == 0) {
#pragma unroll
      for (int k = 0; k < 6; k++)
        if (v[k]) atomicAdd(reinterpret_cast<unsigned long long*>(stats + k), (unsigned long long)v[k]);
      if (mx) atomicMax(reinterpret_cast<long long*>(stats + NARDE_STAT_MAX_ACTIONS), (long long)mx);
      if (ov) atomicAdd(reinterpret_cast<unsigned long long*>(stats + NARDE_STAT_OVERFLOWS), (unsigned long long)ov);
      if (cl) atomicAdd(reinterpret_cast<unsigned long long*>(stats + NARDE_STAT_CLAMPED_ACTIONS), (unsigned long long)cl);
    }
  }
  if (!obs198) return;
  __shared__ float4 lut[16];
  obs_lut_init(lut);
  __syncthreads();
  int rows = (int)min((int64_t)BLK, n - row0);
  write_obs198_cta(sh.st, lut, rows, row0, obs198, sh.defer);
  __syncthreads();
  PHASE_MARK(9);
  GT_MARK(blockIdx.x, 11);
}

// Exact doubles turns handed over by k_step_full_v2 (narde_deferred.cuh).  A short list (self-play: ~0.2 % of the envs,
// fewer entries than CTAs) is latency-bound -- the step ends when the slowest of these envs does -- so the whole CTA
// works on one env; a long list (the doubles-heavy microbench) is throughput-bound: one env per warp.
struct TeamExec {  // ExactStep's executor on the device: the calling thread runs the phase, then its team synchronises
  int tid;         // thread index inside the team
  bool cta;        // team = the CTA (else: the warp)
  template <class F>
  __device__ __forceinline__ void run(F&& f) {
    f(tid);
    if (cta) __syncthreads(); else __syncwarp();
  }
#ifdef NARDE_DEBUG_HOOKS
  unsigned long long* clk;  // phase marks of the env being solved (tools/phase_clock.py)
  __device__ __forceinline__ void mark(int k) {
    if (clk && tid == 0) clk[k] = clock64();
  }
#else
  __device__ __forceinline__ void mark(int) {}
#endif
};
template <int NT, class ShT>
__device__ __forceinline__ void exact_env(TeamExec& ex, ShT& sh, const float4* lut, uint4* lo, uint4* hi, int64_t i,
                                          const StepFullArgs& A, float* obs198, int64_t* stats) {
  State s;
  ex.mark(0);
  if (ex.tid == 0) s = ld_state(lo, hi, i);
#ifdef NARDE_DEBUG_HOOKS
  if (g_dbg_flags & 8) {  // timing experiment: solve twice, the marks show the second (warm) run
    ExactStep<NT>::solve(ex, sh, s, i, A);
    ex.mark(0);
  }
#endif
  ExactStep<NT>::solve(ex, sh, s, i, A);
  ex.mark(8);
  if (ex.tid == 0) {
    StepFullLocal L;
    State st = sh.st;
    if (sh.count && !(A.flags & F_ENUMERATE_ONLY)) {  // apply_action, rolled up (code size: see narde_deferred.cuh)
#pragma unroll 1
      for (int k = 0; k < 4; k++) {
        const uint32_t h = (uint32_t)(sh.chosen >> (16 * k)) & 0xFFFFu;
        if (h == 0xFFFFu) break;
        apply_half_move(st, sh.player, (int)(h & 0xFF), (h >> 8) == 255u ? -1 : (int)(h >> 8));
      }
    }
    complete_env(st, i, A, sh.player, sh.count, sh.chosen, sh.d1, sh.d2, L, false);
    L.clamped = A.action_idx ? index_was_clamped(A, (uint32_t)A.action_idx[i], sh.count) : 0;
    sh.st = st;
    if (!(A.flags & F_ENUMERATE_ONLY)) {
      st_state(lo, hi, i, st);
      if (A.mirror_lo) st_state((uint4*)A.mirror_lo, (uint4*)A.mirror_hi, i, st);
      if (A.mirror_compact) {
        uint32_t r[5];
        pack_compact(st, L.result, r);
        for (int k = 0; k < 5; k++) A.mirror_compact[i * 5 + k] = r[k];
      }
    }
    if (stats) {
      int v[6] = {L.finished, L.white_win, L.black_win, L.mars, L.ep_len, L.count};
      for (int k = 0; k < 6; k++)
        if (v[k]) atomicAdd(reinterpret_cast<unsigned long long*>(stats + k), (unsigned long long)v[k]);
      if (L.count) atomicMax(reinterpret_cast<long long*>(stats + NARDE_STAT_MAX_ACTIONS), (long long)L.count);
      if (L.overflow) atomicAdd(reinterpret_cast<unsigned long long*>(stats + NARDE_STAT_OVERFLOWS), 1ull);
      if (L.clamped) atomicAdd(reinterpret_cast<unsigned long long*>(stats + NARDE_STAT_CLAMPED_ACTIONS), 1ull);
    }
  }
  ex.run([](int) {});
  ex.mark(9);
  if (obs198) write_obs198_cta(&sh.st, lut, 1, i, obs198, nullptr, ex.tid, NT);
  ex.run([](int) {});
  ex.mark(10);
#ifdef NARDE_DEBUG_HOOKS
  if (ex.clk && ex.tid == 0) ex.clk[11] = sh.count | ((unsigned long long)sh.n_cand << 32);
#endif
}
template <int BLK>
__global__ void __launch_bounds__(BLK, 8) k_step_deferred(uint4* lo, uint4* hi, StepFullArgs A_in, float* obs198, int64_t* stats) {
  StepFullArgs A = A_in;
  if (A.step_dev) A.step = *A.step_dev + ((A.flags & F_DEVICE_ADVANCE) ? 1u : 0u);
  union Smem {
    ExactSharedT<32> warp[BLK / 32];
    ExactSharedT<BLK> cta;
  };
  __shared__ Smem sm;
  __shared__ float4 lut[16];
  __shared__ int32_t s_last, s_entry;
  obs_lut_init(lut);
  const int tid = threadIdx.x;
  GT_MARK(3072 + blockIdx.x, 0);
  // Launched as a programmatic dependent of k_step_full_v2: this grid starts once every main CTA has executed its
  // trigger -- at the CTA's start for large batches, after its release-add to `arrivals` (end of the count phase) for
  // one-wave batches -- while the main grid is still running.  "arrivals == n_primary" (acquire) means: every main CTA
  // has pushed its entries, the list is complete.
  // The list is consumed WHILE it is produced.  With the early trigger (large batches) this grid is resident as soon as
  // the last main CTA has been dispatched, most entries are already there (every main CTA of the earlier waves is past
  // its count phase) and the rest arrive while the last wave runs: CTA b takes entry b the moment it is published --
  // an entry is the env index + 1, a zero word means "not yet" -- instead of waiting for the complete list, so the
  // ~18 us an order-dependent turn takes (a latency-bound chain of ~4000 dependent instructions) overlap the main
  // kernel's last wave instead of following it.  Every consumed entry is zeroed again for the next call.
  volatile int32_t* list = reinterpret_cast<volatile int32_t*>(A.defer_list);
  TeamExec ex;
  ex.tid = tid;
  ex.cta = true;
  // (huge batches -- the 1 M-position enumeration -- have lists of tens of thousands of entries: throughput-bound, a warp
  // per env for all of them once the list is complete, no CTA-per-entry round first; decided by the batch size so that
  // every CTA decides the same)
  const bool stream_entries = A.list_cap <= 524288;
  if (stream_entries) {
    const int q = (int)blockIdx.x;
    if (tid == 0) {
      int32_t v = 0, seen = 0;
      while (q < A.list_cap) {
        v = list[q];
        if (v != 0) break;
        if (seen >= A.n_primary) break;  // the list was complete before that read of the entry: there is no entry q
        asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(seen) : "l"(A.arrivals) : "memory");
        if (seen < A.n_primary) __nanosleep(100);
      }
      if (v != 0) list[q] = 0;
      s_entry = v;
    }
    __syncthreads();
    const int32_t v = s_entry;
    GT_MARK(3072 + blockIdx.x, 1);
    if (v != 0) {
#ifdef NARDE_DEBUG_HOOKS
      ex.clk = (g_dbg_clk && q < 1024) ? g_dbg_clk + (size_t)(2048 + q) * 16 : nullptr;
      if (g_dbg_flags & 4) { /* timing experiment only (wrong results): the deferred envs are not solved */ } else
#endif
      exact_env<BLK>(ex, sm.cta, lut, lo, hi, (int64_t)v - 1, A, obs198, stats);
    }
  }
  // entries beyond the first gridDim.x (long lists: the doubles-heavy enumeration microbench) need the complete list
  if (tid == 0) {
    int32_t seen;
    for (;;) {
      asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(seen) : "l"(A.arrivals) : "memory");
      if (seen >= A.n_primary) break;
      __nanosleep(100);
    }
  }
  __syncthreads();
  int n_def = *reinterpret_cast<volatile const int32_t*>(A.defer_count);
  const int G = (int)gridDim.x;
  const int first = stream_entries ? G : 0;  // entries [0, first) were taken above
  if (n_def > first) {
    if (n_def <= first + 2 * G) {  // a few more: the CTA as a team again
      for (int q = first + (int)blockIdx.x; q < n_def; q += G) {
        const int32_t v = list[q];
        __syncthreads();
        if (tid == 0) list[q] = 0;
#ifdef NARDE_DEBUG_HOOKS
        ex.clk = (g_dbg_clk && q < 1024) ? g_dbg_clk + (size_t)(2048 + q) * 16 : nullptr;
#endif
        exact_env<BLK>(ex, sm.cta, lut, lo, hi, (int64_t)v - 1, A, obs198, stats);
      }
    } else {               // throughput-bound: one env per warp
      ex.tid = tid & 31;
      ex.cta = false;
      for (int q = first + (tid >> 5) * G + (int)blockIdx.x; q < n_def; q += G * (BLK / 32)) {
        const int32_t v = list[q];
        __syncwarp();
        if ((tid & 31) == 0) list[q] = 0;
#ifdef NARDE_DEBUG_HOOKS
        ex.clk = (g_dbg_clk && q < 1024) ? g_dbg_clk + (size_t)(2048 + q) * 16 : nullptr;
#endif
        exact_env<32>(ex, sm.warp[tid >> 5], lut, lo, hi, (int64_t)v - 1, A, obs198, stats);
      }
    }
  }
  GT_MARK(3072 + blockIdx.x, 2);
  // F_DEVICE_ADVANCE: the step's own bookkeeping instead of a memset and a counter kernel in front of every step
  // (each is a node of the step's CUDA graph, ~2 us).  Every CTA of this grid is done with the list when it arrives
  // here, and every main CTA has read the step index (first thing it does) and is past its last access to the list
  // header (arrivals == n_primary was observed above): the last arrival clears the header for the next step and
  // publishes the new step index -- while the main grid may still be writing its action lists and Box(198) rows.
  if (A.ticket) {
    __syncthreads();
    if (tid == 0) {
      __threadfence();
      s_last = atomicAdd(A.ticket, 1) == (int)gridDim.x - 1 ? 1 : 0;
    }
    __syncthreads();
    if (s_last) {
      if (tid == 0) {
        *A.last_count = n_def;
        *A.defer_count = 0;
        *A.ticket = 0;
        *A.arrivals = 0;
        *const_cast<uint64_t*>(A.step_dev) = A.step;
        __threadfence();
      }
    }
  }
  GT_MARK(3072 + blockIdx.x, 3);
  // stream order: this grid must not complete before its primary has (the next step follows it); nothing is left to
  // do after it
  asm volatile("griddepcontrol.wait;" ::: "memory");
  GT_MARK(3072 + blockIdx.x, 4);
}

__global__ void __launch_bounds__(kThreads) k_obs198(const uint4* lo, const uint4* hi, int64_t n, float* obs198) {
  __shared__ State sm[kThreads];
  int64_t row0 = (int64_t)blockIdx.x * blockDim.x;
  int64_t i = row0 + threadIdx.x;
  __shared__ float4 lut[16];
  obs_lut_init(lut);
  if (i < n) sm[threadIdx.x] = ld_state(lo, hi, i);
  __syncthreads();
  int rows = (int)min((int64_t)blockDim.x, n - row0);
  write_obs198_cta(sm, lut, rows, row0, obs198);
}

__global__ void __launch_bounds__(kThreads) k_obs24(const uint4* lo, const uint4* hi, int64_t n, int32_t* o24) {
  __shared__ State sm[kThreads];
  int64_t row0 = (int64_t)blockIdx.x * blockDim.x;
  int64_t i = row0 + threadIdx.x;
  if (i < n) sm[threadIdx.x] = ld_state(lo, hi, i);
  __syncthreads();
  int rows = (int)min((int64_t)blockDim.x, n - row0);
  int32_t* base = o24 + row0 * 24;
  for (int j = threadIdx.x; j < rows * 24; j += blockDim.x) {
    int e = j / 24, k = j - e * 24;
    const State& s = sm[e];
    base[j] = s.turn() == 1 ? s.point(k) : -s.point(k < 12 ? k + 12 : k - 12);
  }
}

__global__ void __launch_bounds__(kThreads) k_apply_actions(uint4* lo, uint4* hi, const uint64_t* acts, int64_t n, int flags,
                                                           float* reward, uint8_t* done) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  State s = ld_state(lo, hi, i);
  float r;
  int dn;
  apply_actions_env(s, acts[i], flags, &r, &dn);
  st_state(lo, hi, i, s);
  if (reward) reward[i] = r;
  if (done) done[i] = (uint8_t)dn;
}

// Afterstates of every stored legal action (README get_valid_actions list): row offsets[i] + k holds the
// state of env i after action k and the end-of-turn bookkeeping (player switched), as narde_apply_actions
// would leave it.  Thread per env; rows of neighbouring envs are neighbours in memory.
__global__ void __launch_bounds__(kThreads) k_afterstates(const uint4* lo, const uint4* hi, const uint64_t* actions,
                                                         const int32_t* counts, const int64_t* offsets, int64_t n, int cap,
                                                         uint4* as_lo, uint4* as_hi, int32_t* row_env) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const State s = ld_state(lo, hi, i);
  int c = counts[i];
  c = c < cap ? c : cap;
  const int64_t base = offsets[i];
  for (int k = 0; k < c; k++) {
    State t = s;
    float r;
    int dn;
    apply_actions_env(t, actions[i * (int64_t)cap + k], 0, &r, &dn);
    st_state(as_lo, as_hi, base + k, t);
    if (row_env) row_env[base + k] = (int32_t)i;
  }
}

// Afterstate rows in ONE pass (replaces a host-side clamp / cumsum / subtract / copy chain and the thread-per-env
// kernel above): a CTA owns a tile of 128 environments.  Row offsets are a device-wide exclusive scan of
// min(count, cap) done inside the kernel as a decoupled look-back: tiles are handed out by a ticket (so every tile with
// a smaller number is already running), a CTA publishes its tile total tagged with the launch epoch and then sums the
// totals of the tiles before it (warp 0, 32 tiles per trip).  Rows are then dealt to the threads one by one -- thread r
// finds its (env, action) by a search over the tile's 128 offsets in shared memory -- so neighbouring threads read
// neighbouring action words and write neighbouring 16-byte row halves, whatever the counts are.
// scratch (u64 words, zeroed once by the caller, restored by the last CTA of every launch):
//   [0] ticket  [1] finished CTAs  [2] launch epoch  [4 ..] one word per tile: epoch << 32 | rows of the tile.
__global__ void __launch_bounds__(kThreads) k_afterstates_scan(const uint4* lo, const uint4* hi, const uint64_t* actions,
                                                              const int32_t* counts, int64_t n, int cap, int64_t* offsets,
                                                              int64_t* rows_out, uint4* as_lo, uint4* as_hi, int32_t* row_env,
                                                              unsigned long long* scratch, int64_t rows_cap,
                                                              int32_t* counts_eff) {
  __shared__ State st[kThreads];
  __shared__ uint32_t excl[kThreads + 1];
  __shared__ uint32_t wtot[kThreads / 32];
  __shared__ unsigned long long s_base;
  __shared__ uint32_t s_tile;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) s_tile = (uint32_t)atomicAdd(&scratch[0], 1ull);
  __syncthreads();
  const uint32_t tile = s_tile, ntiles = gridDim.x;
  unsigned long long epoch = (*reinterpret_cast<volatile unsigned long long*>(&scratch[2]) + 1ull) & 0xFFFFFFFFull;
  if (epoch == 0ull) epoch = 1ull;  // 0 is the tag of a never-written word
  const int64_t row0 = (int64_t)tile * kThreads, i = row0 + tid;
  uint32_t c = 0;
  if (i < n) {
    st[tid] = ld_state(lo, hi, i);
    const int cc = counts[i];
    c = (uint32_t)(cc < 0 ? 0 : cc < cap ? cc : cap);
  }
  uint32_t incl = c;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) wtot[warp] = incl;
  __syncthreads();
  uint32_t before = 0, total = 0;
#pragma unroll
  for (int w = 0; w < kThreads / 32; w++) {
    if (w < warp) before += wtot[w];
    total += wtot[w];
  }
  excl[tid] = before + incl - c;
  if (tid == 0) {
    excl[kThreads] = total;
    atomicExch(&scratch[4 + tile], (epoch << 32) | (unsigned long long)total);  // publish before looking back
  }
  if (warp == 0) {  // look-back: rows of all tiles before this one
    unsigned long long sum = 0;
    for (int64_t j0 = (int64_t)tile - 1; j0 >= 0; j0 -= 32) {
      const int64_t j = j0 - lane;
      if (j >= 0) {
        unsigned long long v;
        do {
          v = *reinterpret_cast<volatile unsigned long long*>(&scratch[4 + j]);
        } while ((v >> 32) != epoch);
        sum += v & 0xFFFFFFFFull;
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xFFFFFFFFu, sum, o);
    if (lane == 0) {
      s_base = sum;
      if (tile == ntiles - 1 && rows_out) {
        const int64_t all = (int64_t)(sum + total);
        *rows_out = rows_cap > 0 && all > rows_cap ? rows_cap : all;
      }
    }
  }
  __syncthreads();
  const int64_t base = (int64_t)s_base;
  if (i < n && offsets) offsets[i] = base + excl[tid];
  // a bounded row pool (rows_cap > 0): an env whose rows do not all fit has no rows at all (counts_eff = 0)
  if (i < n && counts_eff) counts_eff[i] = (rows_cap <= 0 || base + excl[tid] + c <= rows_cap) ? (int32_t)c : 0;
  for (uint32_t r = (uint32_t)tid; r < total; r += kThreads) {
    if (rows_cap > 0 && base + r >= rows_cap) break;
    int a = 0, b = kThreads - 1;  // the last env whose first row is <= r (envs without rows share their successor's offset)
    while (a < b) {
      const int mid = (a + b + 1) >> 1;
      if (excl[mid] <= r) a = mid; else b = mid - 1;
    }
    const int e = a;
    const uint32_t k = r - excl[e];
    State t = st[e];
    float rw;
    int dn;
    apply_actions_env(t, actions[(row0 + e) * (int64_t)cap + k], 0, &rw, &dn);
    st_state(as_lo, as_hi, base + r, t);
    if (row_env) row_env[base + r] = (int32_t)(row0 + e);
  }
  __syncthreads();
  if (tid == 0) {
    __threadfence();
    if (atomicAdd(&scratch[1], 1ull) == (unsigned long long)ntiles - 1ull) {  // every CTA is past its look-back
      scratch[0] = 0ull;
      scratch[1] = 0ull;
      scratch[2] = epoch;
      __threadfence();
    }
  }
}

// Second pass of the greedy actor for environments whose legal list exceeds the stored capacity (0.5-1 % of the envs
// in self-play, up to ~1300 actions): their states and dice are gathered into a small side batch that is enumerated
// with a large capacity, scored and arg-maxed like the main batch; k_scatter_choice puts the results back.
// ctrl: [0] overflowing envs seen (all of them, also beyond m), [1] finished CTAs, [2] envs not covered so far (total).
// Slots beyond the gathered ones are marked finished games (no legal action, no afterstate rows) by the last CTA.
// act_override (optional): zeroed for every env, so that the turn starts without an override that an earlier choice left
// unconsumed (k_scatter_choice writes this turn's overrides after this kernel).
__global__ void __launch_bounds__(kThreads) k_gather_overflow(const uint4* lo, const uint4* hi, const uint8_t* dice,
                                                             const uint8_t* overflow, int64_t n, int m, uint4* sub_lo,
                                                             uint4* sub_hi, uint8_t* sub_dice, int32_t* sub_idx, int32_t* ctrl,
                                                             uint64_t* act_override) {
  __shared__ int s_last;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  // The k-th gathered env goes to slot (k mod T) * 32 + k / T, T = m / 32: consecutive entries land in different 32-slot
  // tiles, so the few hundred long lists are spread over all CTAs of the side batch's kernels instead of filling the
  // first ones (contiguous slots: 136 + 140 us for the side enumeration and its afterstate rows; spread: see DESIGN 9).
  const int T = m >> 5;
  if (i < n && act_override) act_override[i] = 0ull;
  if (i < n && overflow[i]) {
    const int seq = atomicAdd(&ctrl[0], 1);
    if (seq < m) {
      const int slot = (seq % T) * 32 + seq / T;
      sub_lo[slot] = lo[i];
      sub_hi[slot] = hi[i];
      reinterpret_cast<uint16_t*>(sub_dice)[slot] = reinterpret_cast<const uint16_t*>(dice)[i];
      sub_idx[slot] = (int32_t)i;
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    s_last = atomicAdd(&ctrl[1], 1) == (int)gridDim.x - 1;
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  const int seen = *reinterpret_cast<volatile int32_t*>(&ctrl[0]);
  State fin;
  for (int k = 0; k < 6; k++) fin.w[k] = 0;
  fin.set_meta(15, 0, 1, FLAG_DONE);
  fin.aux = 0;
  for (int sl = (int)threadIdx.x; sl < m; sl += (int)blockDim.x) {
    if ((sl & 31) * T + (sl >> 5) < seen) continue;  // a gathered env sits here
    st_state(sub_lo, sub_hi, sl, fin);
    reinterpret_cast<uint16_t*>(sub_dice)[sl] = 0x0101;
    sub_idx[sl] = -1;
  }
  if (threadIdx.x == 0) {
    ctrl[1] = 0;
    if (seen > m) ctrl[2] += seen - m;
  }
}
__global__ void __launch_bounds__(256) k_scatter_choice(const int32_t* sub_choice, const float* sub_value, const int32_t* sub_idx,
                                                        const int32_t* sub_counts_eff, const int32_t* sub_counts, int m, int cap,
                                                        int32_t* choice, float* value, int32_t* ctrl,
                                                        const uint64_t* sub_actions, uint64_t* act_out) {
  int missed = 0;
  for (int sl = blockIdx.x * blockDim.x + threadIdx.x; sl < m; sl += gridDim.x * blockDim.x) {
    const int32_t i = sub_idx[sl];
    if (i < 0) continue;  // an unused slot (a finished game put there by the gather)
    if (sub_counts_eff && sub_counts_eff[sl] == 0) {  // its rows did not fit the row pool: the first pass's choice stands
      missed++;
      continue;
    }
    if (sub_counts && sub_counts[sl] > cap) missed++;  // longer than the side batch's capacity: best of the first `cap`
    choice[i] = sub_choice[sl];
    if (value && sub_value) value[i] = sub_value[sl];
    // the action itself, for narde_step_chosen: an index beyond the main batch's stored list cannot be looked up there
    if (act_out && sub_actions) act_out[i] = sub_actions[(int64_t)sl * cap + sub_choice[sl]];
  }
  if (missed) atomicAdd(&ctrl[2], missed);
  if (blockIdx.x == 0 && threadIdx.x == 0) ctrl[0] = 0;  // ready for the next turn's gather (nothing here reads it)
}

// Exploration of narde_segment_sample (the Philox streams and the rule: include/narde_b200.h).  The parameters are read
// from device memory, so a captured CUDA graph picks up new values without a recapture.
struct SampleArgs {
  const float* params;      // {epsilon, inv_temperature}
  const int32_t* env_idx;   // slot -> env index (NULL: slot i is env i); a slot of -1 is skipped
  int64_t env_base;
  uint64_t seed, step;
  const uint64_t* step_dev;  // the turn number on the device (overrides step), as in StepFullArgs
};

// Per env: its global id, the turn number and 1 / temperature; returns the explored index (the env's own uniform
// policy over its c actions, pick_from_word), -1 when the env does not explore, -2 for a skipped slot.
__device__ __forceinline__ int sample_prologue(const SampleArgs& S, int64_t i, int c, uint32_t* env, uint64_t* step,
                                               float* inv_tau) {
  int64_t e = i;
  if (S.env_idx) {
    e = S.env_idx[i];
    if (e < 0) return -2;
  }
  *env = (uint32_t)(S.env_base + e);
  *step = S.step_dev ? *S.step_dev : S.step;
  *inv_tau = S.params[1];
  if (c == 0) return -1;
  const uint32_t below = (uint32_t)(S.params[0] * 16777216.0f);  // floor(eps * 2^24), exact for eps in [0, 1]
  if ((stream_random(S.seed, *env, *step, 2u).x >> 8) >= below) return -1;
  return (int)mulhi32(turn_random(S.seed, *env, *step).z, (uint32_t)c);
}
// Gumbel noise of action k: u = ((w >> 9) + 1/2) / 2^23 lies strictly inside (0, 1) in float32, so G is finite
__device__ __forceinline__ float gumbel(uint64_t seed, uint32_t env, uint64_t step, int k) {
  const float u = ((float)(stream_random(seed, env, step, 3u + ((uint32_t)k << 8)).x >> 9) + 0.5f) * 0x1p-23f;
  return -logf(-logf(u));
}

// The same for long segments (the side batch: lists of hundreds to thousands of actions): a warp per env, lanes stride over
// the segment (coalesced), the (value, index) pairs reduced by shuffles -- a thread per env walks such a segment alone.
// kSample: narde_segment_sample (each lane draws the noise of its own actions); otherwise greedy.
template <bool kSample>
__global__ void __launch_bounds__(kThreads) k_segment_argmax_warp(const float* score, const int64_t* offsets, const int32_t* counts,
                                                                 const uint4* hi, int64_t n, int cap, int mode, int32_t* idx_out,
                                                                 float* best_out, SampleArgs S) {
  const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (i >= n) return;  // (whole warps leave together)
  int c = counts[i];
  c = c < cap ? c : cap;
  const int64_t base = offsets[i];
  float sign = 1.0f;
  if (mode == 1) {
    const uint32_t meta = hi[i].z;
    if ((int)(int8_t)((meta >> 16) & 0xFF) != 1) sign = -1.0f;
  }
  uint32_t env = 0;
  uint64_t step = 0;
  float inv_tau = 0.0f;
  if constexpr (kSample) {
    const int x = sample_prologue(S, i, c, &env, &step, &inv_tau);  // (the same for every lane)
    if (x == -2) return;
    if (x >= 0) {
      if (lane == 0) {
        idx_out[i] = x;
        if (best_out) best_out[i] = score[base + x];
      }
      return;
    }
  }
  float best = 0.0f;
  int best_k = 0x7FFFFFFF;
  for (int k = lane; k < c; k += 32) {
    float v = sign * score[base + k];
    if constexpr (kSample) {
      if (inv_tau > 0.0f) v = v * inv_tau + gumbel(S.seed, env, step, k);
    }
    if (best_k == 0x7FFFFFFF || v > best) {  // strictly greater: the lowest index of a lane's maximum stays
      best = v;
      best_k = k;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_down_sync(0xFFFFFFFFu, best, o);
    const int ok = __shfl_down_sync(0xFFFFFFFFu, best_k, o);
    if (ok != 0x7FFFFFFF && (best_k == 0x7FFFFFFF || ov > best || (ov == best && ok < best_k))) {
      best = ov;
      best_k = ok;
    }
  }
  if (lane == 0) {
    idx_out[i] = c ? best_k : 0;
    if (best_out) best_out[i] = c ? (kSample ? score[base + best_k] : sign * best) : 0.0f;
  }
}

// Greedy choice per env over its segment of afterstate scores: mode 0 = maximise; mode 1 = WHITE
// maximises, BLACK minimises (a value net that scores positions for WHITE).  Ties -> lowest index.
// kSample: narde_segment_sample's epsilon-greedy / Gumbel-max choice instead.
template <bool kSample>
__global__ void __launch_bounds__(kThreads) k_segment_argmax(const float* score, const int64_t* offsets, const int32_t* counts,
                                                            const uint4* hi, int64_t n, int cap, int mode, int32_t* idx_out,
                                                            float* best_out, SampleArgs S) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int c = counts[i];
  c = c < cap ? c : cap;
  const int64_t base = offsets[i];
  float sign = 1.0f;
  if (mode == 1) {
    const uint32_t meta = hi[i].z;
    if ((int)(int8_t)((meta >> 16) & 0xFF) != 1) sign = -1.0f;
  }
  uint32_t env = 0;
  uint64_t step = 0;
  float inv_tau = 0.0f;
  if constexpr (kSample) {
    const int x = sample_prologue(S, i, c, &env, &step, &inv_tau);
    if (x == -2) return;
    if (x >= 0) {
      idx_out[i] = x;
      if (best_out) best_out[i] = score[base + x];
      return;
    }
  }
  int best_k = 0;
  float best = 0.0f;
  for (int k = 0; k < c; k++) {
    float v = sign * score[base + k];
    if constexpr (kSample) {
      if (inv_tau > 0.0f) v = v * inv_tau + gumbel(S.seed, env, step, k);
    }
    if (k == 0 || v > best) {
      best = v;
      best_k = k;
    }
  }
  idx_out[i] = best_k;
  if (best_out) best_out[i] = c ? (kSample ? score[base + best_k] : sign * best) : 0.0f;
}

// Trainer-compatible action codes (train_deepq_pytorch.py:432-437,495-507,752-761): for every stored legal
// turn action the reference's (move1_code, move2_code) pair, code = from*24 + to with to = 0 for a bear-off
// and move2_code = 0 when the turn has one half-move.  Only the first two half-moves are representable in
// the reference's pair space; codes[.., 2] = number of half-moves of the turn (3 or 4 for doubles).
__global__ void __launch_bounds__(kThreads) k_action_codes(const uint64_t* actions, const int32_t* counts, int64_t n, int cap,
                                                          int32_t* codes) {
  int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n * (int64_t)cap) return;
  const int64_t i = g / cap;
  const int k = (int)(g - i * cap);
  int32_t c1 = 0, c2 = 0, nh = 0;
  if (k < counts[i]) {
    const uint64_t a = actions[g];
#pragma unroll
    for (int h = 0; h < 4; h++) {
      const uint32_t hm = (uint32_t)(a >> (16 * h)) & 0xFFFFu;
      if (hm == 0xFFFFu) break;
      const int from = (int)(hm & 0xFF), to = (int)(hm >> 8);
      const int code = from * 24 + (to == 255 ? 0 : to);
      if (h == 0) c1 = code;
      if (h == 1) c2 = code;
      nh++;
    }
  }
  codes[3 * g] = c1;
  codes[3 * g + 1] = c2;
  codes[3 * g + 2] = nh;
}

// Trajectory record of one env turn (SURVEY 8(f) rank 3), 48 bytes:
//   [0,16) lo lane | [16,32) hi lane (state AFTER the turn = state before the next one) | u64 action played
//   | f32 reward | u8 die 1, u8 die 2, u8 done (1 terminated, 2 truncated), u8 reserved
__global__ void __launch_bounds__(kThreads) k_trajectory_append(const uint4* lo, const uint4* hi, const uint8_t* dice,
                                                               const uint64_t* chosen, const float* reward, const uint8_t* done,
                                                               const uint8_t* truncated, int64_t n, uint4* records) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint64_t a = chosen ? chosen[i] : ~0ull;
  const uint32_t d = dice ? (uint32_t)reinterpret_cast<const uint16_t*>(dice)[i] : 0u;
  const uint32_t dn = (done && done[i] ? 1u : 0u) | (truncated && truncated[i] ? 2u : 0u);
  records[3 * i] = lo[i];
  records[3 * i + 1] = hi[i];
  records[3 * i + 2] = make_uint4((uint32_t)a, (uint32_t)(a >> 32), reward ? __float_as_uint(reward[i]) : 0u, d | (dn << 16));
}

__global__ void __launch_bounds__(kThreads) k_roll_dice(int64_t n, int64_t env_base, uint64_t seed, uint64_t step, uint8_t* dice) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  U4 r = turn_random(seed, (uint32_t)(env_base + i), step);
  reinterpret_cast<uint16_t*>(dice)[i] = (uint16_t)(die_from_word(r.x) | (die_from_word(r.y) << 8));
}

__global__ void __launch_bounds__(kThreads) k_block_rule(const int8_t* boards, int64_t n, uint8_t* out) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t own = 0, opp = 0;
  for (int k = 0; k < 24; k++) {
    int v = boards[i * 24 + k];
    own |= (v > 0 ? 1u : 0u) << k;
    opp |= (v < 0 ? 1u : 0u) << k;
  }
  out[i] = violates_block(own, opp) ? 1 : 0;
}

// programmatic dependent launch of the exact kernel (NARDE_NO_PDL=1 in the environment disables it: A/B timing)
bool g_use_pdl = true;

__global__ void k_advance_counter(uint64_t* ctr) { *ctr += 1; }

inline int grid_for(int64_t n) { return (int)((n + kThreads - 1) / kThreads); }
inline int launch_status() { return (int)cudaGetLastError(); }

template <bool kSample>
int launch_segment(const float* score, const int64_t* offsets, const int32_t* counts, const void* hi, int64_t n, int cap, int mode,
                   int32_t* idx_out, float* best_out, const SampleArgs& S, void* stream) {
  if (cap > 128)  // long segments: a warp per env
    k_segment_argmax_warp<kSample><<<grid_for(n * 32), kThreads, 0, (cudaStream_t)stream>>>(score, offsets, counts, (const uint4*)hi,
                                                                                             n, cap, mode, idx_out, best_out, S);
  else
    k_segment_argmax<kSample><<<grid_for(n), kThreads, 0, (cudaStream_t)stream>>>(score, offsets, counts, (const uint4*)hi, n, cap,
                                                                                  mode, idx_out, best_out, S);
  return launch_status();
}
inline bool aligned16(const void* p) { return (((uintptr_t)p) & 15u) == 0; }

}  // namespace

extern "C" {

int narde_abi_version(void) {
  static bool env_read = false;
  if (!env_read) {
    const char* v = getenv("NARDE_NO_PDL");
    if (v && v[0] == '1') g_use_pdl = false;
    v = getenv("NARDE_SMALL_BATCH");
    if (v) kSmallBatch = atoll(v);
    v = getenv("NARDE_TILE");
    if (v && (atoi(v) == 128 || atoi(v) == 64)) g_tile = atoi(v);
    v = getenv("NARDE_LATE_TRIGGER");
    if (v && v[0] == '1') g_early = false;
    v = getenv("NARDE_VARIANT");
    if (v) g_variant = atoi(v);
    env_read = true;
  }
  // one-time function attributes are set here (outside any stream capture)
  return NARDE_ABI_VERSION;
}
const char* narde_build_arch(void) { return "sm_100a"; }

int narde_reset_masked(void* lo, void* hi, const uint8_t* mask, int64_t n, int64_t env_base, uint64_t seed, uint64_t step,
                       void* stream) {
  if (n == 0) return 0;
  if (n < 0 || !lo || !hi || !aligned16(lo) || !aligned16(hi)) return -1;
  k_reset<<<grid_for(n), kThreads, 0, (cudaStream_t)stream>>>((uint4*)lo, (uint4*)hi, mask, n, env_base, seed, step);
  return launch_status();
}

int narde_reset(void* lo, void* hi, int64_t n, int64_t env_base, uint64_t seed, uint64_t step, void* stream) {
  return narde_reset_masked(lo, hi, nullptr, n, env_base, seed, step, stream);
}

int narde_half_moves(const void* lo, const void* hi, const uint8_t* dice, int64_t n, int player_override, uint8_t* moves,
                     int32_t* counts, void* stream) {
  if (n == 0) return 0;
  if (n < 0 || !lo || !hi || !dice || !moves || !counts || !aligned16(lo) || !aligned16(hi)) return -1;
  if ((((uintptr_t)dice) & 3u) != 0) return -1;
  k_half_moves<<<grid_for(n), kThreads, 0, (cudaStream_t)stream>>>((const uint4*)lo, (const uint4*)hi, dice, n,
                                                                   player_override, moves, counts);
  return launch_status();
}

int narde_step_ref(void* lo, void* hi, const uint8_t* dice, const int32_t* codes, int64_t n, int32_t max_episode_steps,
                   int32_t* obs24, int32_t* reward, uint8_t* done, uint8_t* truncated, void* stream) {
  if (n == 0) return 0;
  if (n < 0 || !lo || !hi || !dice || !codes || !aligned16(lo) || !aligned16(hi)) return -1;
  if ((((uintptr_t)dice) & 1u) != 0 || (((uintptr_t)codes) & 7u) != 0) return -1;
  k_step_ref<<<grid_for(n), kThreads, 0, (cudaStream_t)stream>>>((uint4*)lo, (uint4*)hi, dice, codes, n,
                                                                 max_episode_steps, obs24, reward, done, truncated);
  return launch_status();
}

int narde_enumerate(const void* lo, const void* hi, const uint8_t* dice, int64_t n, int32_t cap, uint64_t* actions,
                    int32_t* counts, uint8_t* overflow, void* stream) {
  if (n == 0) return 0;
  if (n < 0 || cap < 0 || !lo || !hi || !dice || !counts || (cap > 0 && !actions) || !aligned16(lo) || !aligned16(hi))
    return -1;
  if ((((uintptr_t)dice) & 1u) != 0) return -1;
  k_enumerate<<<grid_for(n), kThreads, 0, (cudaStream_t)stream>>>((const uint4*)lo, (const uint4*)hi, dice, n, cap,
                                                                  actions, counts, overflow);
  return launch_status();
}

int narde_step_full(void* lo, void* hi, int64_t n, int64_t env_base, uint64_t seed, uint64_t step, const uint8_t* dice_in,
                    const int32_t* action_idx, int32_t cap, uint64_t* actions, int32_t* counts, uint8_t* dice_out,
                    uint64_t* chosen, float* obs198, float* reward, uint8_t* done, uint8_t* truncated, int64_t* stats,
                    int32_t flags, int32_t max_episode_steps, int32_t* workspace, const uint64_t* step_dev, void* stream);

int narde_enumerate_fast(const void* lo, const void* hi, const uint8_t* dice, int64_t n, int32_t cap, uint64_t* actions,
                         int32_t* counts, uint8_t* overflow, int32_t* workspace, void* stream) {
  if (n == 0) return 0;
  if (n < 0 || cap < 0 || !lo || !hi || !dice || !counts || (cap > 0 && !actions)) return -1;
  return narde_step_full(const_cast<void*>(lo), const_cast<void*>(hi), n, 0, 0, 0, dice, nullptr, cap, actions, counts, nullptr,
                         nullptr, nullptr, nullptr, overflow, nullptr, nullptr, NARDE_ENUMERATE_ONLY, 0, workspace, nullptr,
                         stream);
}

int narde_step_full(void* lo, void* hi, int64_t n, int64_t env_base, uint64_t seed, uint64_t step, const uint8_t* dice_in,
                    const int32_t* action_idx, int32_t cap, uint64_t* actions, int32_t* counts, uint8_t* dice_out,
                    uint64_t* chosen, float* obs198, float* reward, uint8_t* done, uint8_t* truncated, int64_t* stats,
                    int32_t flags, int32_t max_episode_steps, int32_t* workspace, const uint64_t* step_dev, void* stream) {
  return narde_step_full_mirror(lo, hi, n, env_base, seed, step, dice_in, action_idx, cap, actions, counts, dice_out, chosen,
                                obs198, reward, done, truncated, stats, flags, max_episode_steps, workspace, step_dev, nullptr,
                                nullptr, stream);
}

int narde_step_full_mirror(void* lo, void* hi, int64_t n, int64_t env_base, uint64_t seed, uint64_t step,
                           const uint8_t* dice_in, const int32_t* action_idx, int32_t cap, uint64_t* actions, int32_t* counts,
                           uint8_t* dice_out, uint64_t* chosen, float* obs198, float* reward, uint8_t* done,
                           uint8_t* truncated, int64_t* stats, int32_t flags, int32_t max_episode_steps, int32_t* workspace,
                           const uint64_t* step_dev, void* mirror_lo, void* mirror_hi, void* stream) {
  if (n == 0) return 0;
  // mirror_lo with mirror_hi: the two state planes; mirror_lo alone: the compact 20-byte records
  if ((mirror_hi && !mirror_lo) || !aligned16(mirror_lo) || !aligned16(mirror_hi)) return -1;
  if (mirror_lo && (flags & NARDE_ENUMERATE_ONLY)) return -1;
  const bool compact = mirror_lo && !mirror_hi;
  if (compact && (flags & NARDE_PER_THREAD_KERNEL)) return -1;
  if (n < 0 || cap < 0 || !lo || !hi || !aligned16(lo) || !aligned16(hi)) return -1;
  if (obs198 && (((uintptr_t)obs198) & 7u) != 0) return -1;
  if (n == 0) return 0;
  StepFullArgs A;
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
  A.defer_count = nullptr;
  A.defer_list = nullptr;
  A.step_dev = step_dev;
  A.ticket = nullptr;
  A.arrivals = nullptr;
  A.n_primary = 0;
  A.early_trigger = 0;
  A.list_cap = n;
  A.last_count = nullptr;
  A.mirror_lo = compact ? nullptr : mirror_lo;
  A.mirror_hi = mirror_hi;
  A.mirror_compact = compact ? reinterpret_cast<uint32_t*>(mirror_lo) : nullptr;
  const bool dev_advance = (flags & NARDE_DEVICE_ADVANCE) != 0;
  if (dev_advance && (!workspace || !step_dev || (flags & (NARDE_PER_THREAD_KERNEL | NARDE_ENUMERATE_ONLY)))) return -1;
  if (flags & NARDE_PER_THREAD_KERNEL) {
    if (flags & NARDE_ENUMERATE_ONLY) return -1;
    k_step_full<<<grid_for(n), kThreads, 0, (cudaStream_t)stream>>>((uint4*)lo, (uint4*)hi, n, A, obs198, stats);
    return launch_status();
  }
  // Workspace (NARDE_WORKSPACE_INTS(n) words, layout in include/narde_b200.h): header [0] number of deferred envs,
  // [1] arrival counter of the exact kernel's CTAs (DEVICE_ADVANCE), [2] arrival counter of the main kernel's CTAs,
  // [3] deferred envs of the last completed DEVICE_ADVANCE call; [NARDE_WORKSPACE_HEADER..] the deferred indices.
  if (workspace) {
    if ((((uintptr_t)workspace) & 3u) != 0) return -1;
    A.defer_count = workspace;
    A.arrivals = workspace + 2;
    A.last_count = workspace + 3;
    A.defer_list = workspace + NARDE_WORKSPACE_HEADER;
    A.n_primary = (int32_t)(n <= kSmallBatch ? (n + 31) / 32 : (n + g_tile - 1) / g_tile);
    A.early_trigger = (g_use_pdl && g_early && n > kSmallBatch) ? 1 : 0;
    if (dev_advance) {  // the three counters are zero on entry and again on exit
      A.ticket = workspace + 1;
    } else {
      cudaError_t e = cudaMemsetAsync(workspace, 0, 3 * sizeof(int32_t), (cudaStream_t)stream);
      if (e != cudaSuccess) return (int)e;
    }
  }
  const cudaStream_t st = (cudaStream_t)stream;
  uint4 *plo = (uint4*)lo, *phi = (uint4*)hi;
  if (n <= kSmallBatch) {
    const int g = (int)((n + 31) / 32);
    if (workspace)
      k_step_full_v2<32, true, 32, 1><<<g, 32, 0, st>>>(plo, phi, n, A, obs198, stats);
    else
      k_step_full_v2<32, false, 32, 1><<<g, 32, 0, st>>>(plo, phi, n, A, obs198, stats);
  } else if (g_tile == 64) {
    const int g = (int)((n + 63) / 64);
    if (!workspace)
      k_step_full_v2<64, false, 128, 8><<<g, 128, 0, st>>>(plo, phi, n, A, obs198, stats);
#ifdef NARDE_DEBUG_HOOKS  // A/B variants of the tile (NARDE_VARIANT): register budget / threads per env
    else if (g_variant == 1)
      k_step_full_v2<64, true, 128, 5><<<g, 128, 0, st>>>(plo, phi, n, A, obs198, stats);
    else if (g_variant == 2)
      k_step_full_v2<64, true, 128, 6><<<g, 128, 0, st>>>(plo, phi, n, A, obs198, stats);
    else if (g_variant == 3)
      k_step_full_v2<64, true, 64, 10><<<g, 64, 0, st>>>(plo, phi, n, A, obs198, stats);
#endif
    else
      k_step_full_v2<64, true, 128, 8><<<g, 128, 0, st>>>(plo, phi, n, A, obs198, stats);
  } else {
    const int g = (int)((n + 127) / 128);
    if (!workspace)
      k_step_full_v2<128, false, 128, 5><<<g, 128, 0, st>>>(plo, phi, n, A, obs198, stats);
#ifdef NARDE_DEBUG_HOOKS
    else if (g_variant == 1)
      k_step_full_v2<128, true, 128, 8><<<g, 128, 0, st>>>(plo, phi, n, A, obs198, stats);
    else if (g_variant == 2)
      k_step_full_v2<128, true, 256, 4><<<g, 256, 0, st>>>(plo, phi, n, A, obs198, stats);
    else if (g_variant == 3)  // 128-register budget (110-113 used), 4 CTAs per SM: 1 us faster in the timeline probe, 7 us SLOWER in bench.py
      k_step_full_v2<128, true, 128, 4><<<g, 128, 0, st>>>(plo, phi, n, A, obs198, stats);
#endif
    else
      k_step_full_v2<128, true, 128, 5><<<g, 128, 0, st>>>(plo, phi, n, A, obs198, stats);
  }
  if (workspace) {
    if (g_use_pdl) {
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3(A.early_trigger && n <= 524288 ? kDeferredGridEarly : kDeferredGrid);
      cfg.blockDim = dim3(kDeferredThreads);
      cfg.dynamicSmemBytes = 0;
      cfg.stream = (cudaStream_t)stream;
      cudaLaunchAttribute at[1];
      at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
      at[0].val.programmaticStreamSerializationAllowed = 1;
      cfg.attrs = at;
      cfg.numAttrs = 1;
      cudaError_t e = cudaLaunchKernelEx(&cfg, k_step_deferred<kDeferredThreads>, (uint4*)lo, (uint4*)hi, A, obs198, stats);
      if (e != cudaSuccess) return (int)e;
    } else {
      k_step_deferred<kDeferredThreads><<<kDeferredGrid, kDeferredThreads, 0, (cudaStream_t)stream>>>((uint4*)lo, (uint4*)hi, A, obs198, stats);
    }
  }
  return launch_status();
}

int narde_obs198(const void* lo, const void* hi, int64_t n, float* obs198, void* stream) {
  if (n == 0) return 0;
  if (n < 0 || !lo || !hi || !obs198 || !aligned16(lo) || !aligned16(hi) || (((uintptr_t)obs198) & 7u) != 0) return -1;
  k_obs198<<<grid_for(n), kThreads, 0, (cudaStream_t)stream>>>((const uint4*)lo, (const uint4*)hi, n, obs198);
  return launch_status();
}

int narde_obs24(const void* lo, const void* hi, int64_t n, int32_t* obs24, void* stream) {
  if (n == 0) return 0;
  if (n < 0 || !lo || !hi || !obs24 || !aligned16(lo) || !aligned16(hi)) return -1;
  k_obs24<<<grid_for(n), kThreads, 0, (cudaStream_t)stream>>>((const uint4*)lo, (const uint4*)hi, n, obs24);
  return launch_status();
}

int narde_apply_actions(void* lo, void* hi, const uint64_t* acts, int64_t n, int32_t flags, float* reward, uint8_t* done,
                        void* stream) {
  if (n == 0) return 0;
  if (n < 0 || !lo || !hi || !acts || !aligned16(lo) || !aligned16(hi)) return -1;
  k_apply_actions<<<grid_for(n), kThreads, 0, (cudaStream_t)stream>>>((uint4*)lo, (uint4*)hi, acts, n, flags, reward, done);
  return launch_status();
}

int narde_afterstates(const void* lo, const void* hi, const uint64_t* actions, const int32_t* counts, const int64_t* offsets,
                      int64_t n, int32_t cap, void* as_lo, void* as_hi, int32_t* row_env, void* stream) {
  if (n == 0) return 0;
  if (n < 0 || cap <= 0 || !lo || !hi || !actions || !counts || !offsets || !as_lo || !as_hi) return -1;
  if (!aligned16(lo) || !aligned16(hi) || !aligned16(as_lo) || !aligned16(as_hi)) return -1;
  k_afterstates<<<grid_for(n), kThreads, 0, (cudaStream_t)stream>>>((const uint4*)lo, (const uint4*)hi, actions, counts, offsets, n,
                                                                    cap, (uint4*)as_lo, (uint4*)as_hi, row_env);
  return launch_status();
}

int narde_afterstates_scan(const void* lo, const void* hi, const uint64_t* actions, const int32_t* counts, int64_t n,
                           int32_t cap, int64_t* offsets, int64_t* rows_out, void* as_lo, void* as_hi, int32_t* row_env,
                           uint64_t* scratch, int64_t rows_cap, int32_t* counts_eff, void* stream) {
  if (n == 0) return 0;
  if (n < 0 || cap <= 0 || !lo || !hi || !actions || !counts || !as_lo || !as_hi || !scratch) return -1;
  if (!aligned16(lo) || !aligned16(hi) || !aligned16(as_lo) || !aligned16(as_hi) || (((uintptr_t)scratch) & 7u) != 0) return -1;
  k_afterstates_scan<<<grid_for(n), kThreads, 0, (cudaStream_t)stream>>>((const uint4*)lo, (const uint4*)hi, actions, counts, n, cap,
                                                                         offsets, rows_out, (uint4*)as_lo, (uint4*)as_hi, row_env,
                                                                         reinterpret_cast<unsigned long long*>(scratch), rows_cap,
                                                                         counts_eff);
  return launch_status();
}

int narde_gather_overflow_clear(const void* lo, const void* hi, const uint8_t* dice, const uint8_t* overflow, int64_t n,
                                int32_t m, void* sub_lo, void* sub_hi, uint8_t* sub_dice, int32_t* sub_idx, int32_t* ctrl,
                                uint64_t* act_override, void* stream) {
  if (n == 0) return 0;
  if (n < 0 || m <= 0 || (m & 31) != 0 || !lo || !hi || !dice || !overflow || !sub_lo || !sub_hi || !sub_dice || !sub_idx || !ctrl) return -1;
  if (!aligned16(lo) || !aligned16(hi) || !aligned16(sub_lo) || !aligned16(sub_hi)) return -1;
  if ((((uintptr_t)dice) & 1u) != 0 || (((uintptr_t)sub_dice) & 1u) != 0) return -1;
  k_gather_overflow<<<grid_for(n), kThreads, 0, (cudaStream_t)stream>>>((const uint4*)lo, (const uint4*)hi, dice, overflow, n, m,
                                                                        (uint4*)sub_lo, (uint4*)sub_hi, sub_dice, sub_idx, ctrl,
                                                                        act_override);
  return launch_status();
}

int narde_gather_overflow(const void* lo, const void* hi, const uint8_t* dice, const uint8_t* overflow, int64_t n, int32_t m,
                          void* sub_lo, void* sub_hi, uint8_t* sub_dice, int32_t* sub_idx, int32_t* ctrl, void* stream) {
  return narde_gather_overflow_clear(lo, hi, dice, overflow, n, m, sub_lo, sub_hi, sub_dice, sub_idx, ctrl, nullptr, stream);
}

int narde_scatter_choice(const int32_t* sub_choice, const float* sub_value, const int32_t* sub_idx, const int32_t* sub_counts_eff,
                         const int32_t* sub_counts, int32_t m, int32_t cap, int32_t* choice, float* value, int32_t* ctrl,
                         const uint64_t* sub_actions, uint64_t* act_out, void* stream) {
  if (m <= 0 || !sub_choice || !sub_idx || !choice || !ctrl) return -1;
  k_scatter_choice<<<(m + 255) / 256, 256, 0, (cudaStream_t)stream>>>(sub_choice, sub_value, sub_idx, sub_counts_eff, sub_counts, m,
                                                                      cap, choice, value, ctrl, sub_actions, act_out);
  return launch_status();
}

int narde_step_chosen(void* lo, void* hi, int64_t n, int64_t env_base, uint64_t seed, uint64_t step, const uint8_t* dice,
                      const int32_t* choice, const uint64_t* actions, int32_t cap, const int32_t* counts, uint64_t* act_override,
                      uint64_t* chosen, float* obs198, float* reward, uint8_t* done, uint8_t* truncated, int64_t* stats,
                      int32_t flags, int32_t max_episode_steps, const uint64_t* step_dev, void* stream) {
  if (n == 0) return 0;
  if (n < 0 || cap <= 0 || !lo || !hi || !dice || !choice || !actions || !counts || !aligned16(lo) || !aligned16(hi)) return -1;
  if ((((uintptr_t)dice) & 1u) != 0 || (obs198 && (((uintptr_t)obs198) & 7u) != 0)) return -1;
  if (flags & ~(NARDE_REWARD_MOVER12 | NARDE_AUTORESET)) return -1;
  StepFullArgs A = {};
  A.env_base = env_base;
  A.seed = seed;
  A.step = step;
  A.dice_in = dice;
  A.action_idx = choice;
  A.cap = cap;
  A.chosen = chosen;
  A.reward = reward;
  A.done = done;
  A.truncated = truncated;
  A.flags = flags;
  A.max_episode_steps = max_episode_steps;
  A.step_dev = step_dev;
  k_step_chosen<<<grid_for(n), kThreads, 0, (cudaStream_t)stream>>>((uint4*)lo, (uint4*)hi, n, A, actions, counts, act_override,
                                                                   obs198, stats);
  return launch_status();
}

int narde_segment_argmax(const float* score, const int64_t* offsets, const int32_t* counts, const void* hi, int64_t n,
                         int32_t cap, int32_t mode, int32_t* idx_out, float* best_out, void* stream) {
  if (n == 0) return 0;
  if (n < 0 || cap <= 0 || !score || !offsets || !counts || !hi || !idx_out || !aligned16(hi)) return -1;
  return launch_segment<false>(score, offsets, counts, hi, n, cap, mode, idx_out, best_out, SampleArgs{}, stream);
}

int narde_segment_sample(const float* score, const int64_t* offsets, const int32_t* counts, const void* hi, int64_t n,
                         int32_t cap, int32_t mode, const int32_t* env_idx, int64_t env_base, uint64_t seed, uint64_t step,
                         const uint64_t* step_dev, const float* params, int32_t* idx_out, float* value_out, void* stream) {
  if (n == 0) return 0;
  if (n < 0 || cap <= 0 || !score || !offsets || !counts || !hi || !params || !idx_out || !aligned16(hi)) return -1;
  const SampleArgs S = {params, env_idx, env_base, seed, step, step_dev};
  return launch_segment<true>(score, offsets, counts, hi, n, cap, mode, idx_out, value_out, S, stream);
}

int narde_action_codes(const uint64_t* actions, const int32_t* counts, int64_t n, int32_t cap, int32_t* codes, void* stream) {
  if (n == 0 || cap == 0) return 0;
  if (n < 0 || cap < 0 || !actions || !counts || !codes) return -1;
  k_action_codes<<<grid_for(n * (int64_t)cap), kThreads, 0, (cudaStream_t)stream>>>(actions, counts, n, cap, codes);
  return launch_status();
}

int narde_trajectory_append(const void* lo, const void* hi, const uint8_t* dice, const uint64_t* chosen, const float* reward,
                            const uint8_t* done, const uint8_t* truncated, int64_t n, void* records, void* stream) {
  if (n == 0) return 0;
  if (n < 0 || !lo || !hi || !records || !aligned16(lo) || !aligned16(hi) || !aligned16(records)) return -1;
  if (dice && (((uintptr_t)dice) & 1u) != 0) return -1;
  k_trajectory_append<<<grid_for(n), kThreads, 0, (cudaStream_t)stream>>>((const uint4*)lo, (const uint4*)hi, dice, chosen, reward,
                                                                          done, truncated, n, (uint4*)records);
  return launch_status();
}

int narde_roll_dice(int64_t n, int64_t env_base, uint64_t seed, uint64_t step, uint8_t* dice, void* stream) {
  if (n == 0) return 0;
  if (n < 0 || !dice || (((uintptr_t)dice) & 1u) != 0) return -1;
  k_roll_dice<<<grid_for(n), kThreads, 0, (cudaStream_t)stream>>>(n, env_base, seed, step, dice);
  return launch_status();
}

int narde_violates_block_rule(const int8_t* boards, int64_t n, uint8_t* out, void* stream) {
  if (n == 0) return 0;
  if (n < 0 || !boards || !out) return -1;
  k_block_rule<<<grid_for(n), kThreads, 0, (cudaStream_t)stream>>>(boards, n, out);
  return launch_status();
}

int narde_advance_counter(uint64_t* counter, void* stream) {
  if (!counter) return -1;
  k_advance_counter<<<1, 1, 0, (cudaStream_t)stream>>>(counter);
  return launch_status();
}

#ifdef NARDE_DEBUG_HOOKS
int narde_debug_set_flags(int flags) { return (int)cudaMemcpyToSymbol(narde::g_dbg_flags, &flags, sizeof(flags)); }

int narde_debug_set_stagger(unsigned ns) { return (int)cudaMemcpyToSymbol(g_dbg_stagger_ns, &ns, sizeof(ns)); }

int narde_debug_set_clock_buffer(void* devptr) {
  unsigned long long* p = (unsigned long long*)devptr;
  return (int)cudaMemcpyToSymbol(g_dbg_clk, &p, sizeof(p));
}
#endif

}  // extern "C"
