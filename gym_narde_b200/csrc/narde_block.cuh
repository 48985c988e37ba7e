// narde_block.cuh -- the fused full-rules step, CTA-cooperative version.
//
// One CTA of BLK threads owns BLK environments.  Instead of one thread walking one environment's
// whole move tree (badly divergent: doubles vs non-doubles, 1 vs 1000 legal turns), the CTA
// flattens the enumeration into uniform work items that are dealt out evenly to its threads:
//   non-doubles : item = (env, p)       "source p plays the higher die"            (~9 per env)
//   doubles     : item = (env, s1, s2)  "the two highest sources played"           (~7 per env)
// Items are counted, prefix-summed in shared memory, and every thread takes a contiguous chunk of
// ceil(items / BLK).  Legal-action counts per chunk / per env are prefix-summed again to give
// every item its slot in the env's canonical action list, so the list is written in order
// without sorting.  Positions where the 6-prime block rule could matter (~4%) run the exact
// (board-testing) arithmetic inside the same items; only doubles turns that cannot use all four
// dice (~3%) fall back to a sequential per-thread walk.
//
// The code is written as PHASES: plain functions of (tid, shared block state) that only read what
// earlier phases wrote (shared-memory atomics aside).  The kernel runs them with __syncthreads()
// in between; the test-only host harness runs "for tid in 0..BLK" per phase, which is the same
// thing, so this file is verified against the oracle on the CPU before it reaches the GPU.
#pragma once
#include "narde_env.cuh"

namespace narde {

enum : uint8_t { K_NONE = 0, K_DONE = 1, K_ND = 2, K_D = 3 };

#if defined(NARDE_HOSTSIM_HOOKS) && !defined(__CUDA_ARCH__)
extern int g_hs_force_slow;  // defined by the test-only host harness (tests/hostsim/hostsim.cpp)
#endif

NHD void sm_add(uint32_t* p, uint32_t v) {
#if defined(__CUDA_ARCH__)
  atomicAdd(p, v);
#else
  *p += v;
#endif
}
NHD int32_t gl_fetch_add(int32_t* p, int32_t v) {  // global-memory counter
#if defined(__CUDA_ARCH__)
  return atomicAdd(p, v);
#else
  int32_t o = *p;
  *p += v;
  return o;
#endif
}
NHD void sm_max(uint32_t* p, uint32_t v) {
#if defined(__CUDA_ARCH__)
  atomicMax(p, v);
#else
  if (v > *p) *p = v;
#endif
}

// One sink for the rare per-thread walks (stores the first `cap`, remembers ordinal `want`), and the
// walk itself out of line: the code exists once instead of once per (sink, variant) combination.
struct WalkSink {
  uint64_t* out;
  int cap, want, n;
  uint64_t picked;
  NHD void operator()(uint64_t a) {
    if (n < cap) out[n] = a;
    if (n == want) picked = a;
    n++;
  }
};
NHD_NOINLINE int walk_short_double(const Pos& P, int d, bool first_turn, int H, int target, bool known, WalkSink& sink) {
  if (known) return enum_double_at(P, d, H, target, sink);
  int depth;
  return enum_double(P, d, first_turn, !block_rule_irrelevant(P, d, d), sink, &depth);
}

constexpr int kL1PerEnv = 5;  // level-1 doubles items a CTA can hold per env (all-doubles CTAs with > 8 sources per env overflow to the sequential walk; never observed)

// BLK = environments per CTA, NT = threads per CTA (NT >= BLK, both multiples of 32).  NT = BLK: a thread per env.
// NT = 2 BLK: the same work items dealt to twice the threads -- shared memory is what limits the number of
// environments resident on an SM, so this is how the SM gets more warps (the kernel is latency-bound).
template <int BLK, int NT = BLK>
struct BlockShared {
  static constexpr int kL1Cap = kL1PerEnv * BLK;
  State st[BLK];
  // per-env position in the mover frame
  uint32_t own[BLK], opp[BLK], ones[BLK];
  uint32_t nlo0[BLK], nlo1[BLK], nhi[BLK];
  uint32_t Ca[BLK], S[BLK], qhome[BLK];  // non-doubles: candidates of die a, die b; "q makes all home"
  alignas(16) uint32_t rnd[BLK];         // the policy word of the turn (bulk-copied from the caller's buffer, or Philox)
  alignas(8) unsigned long long rnd_bar; // mbarrier of that bulk copy
  uint64_t chosen[BLK];
  uint8_t a[BLK], b[BLK], kind[BLK], first[BLK], d1[BLK], d2[BLK], blk[BLK];
  uint32_t maxd[BLK];                    // doubles: deepest playable level seen
  uint32_t defer[BLK];                   // doubles: a reachable-looking board violates the block rule -> exact kernel
  uint32_t etotal[BLK], ebase[BLK];      // legal actions of the env / start of its list in item space
  // work items: ND rows, doubles level-1 sources, doubles level-2 sources
  uint32_t rowmask[BLK], dmask[BLK];
  uint32_t ibase[BLK + 1], dbase[BLK + 1];
  uint32_t pres[BLK * 24];               // ND: pairs (p, q) legal in some order, one mask per row
  uint32_t d2mask[kL1Cap];
  uint32_t d2base[kL1Cap + 1];
  uint8_t l1env[kL1Cap], l1src[kL1Cap];
  uint16_t itab[BLK * 24];               // ND work items in canonical order: env << 5 | source point
  uint32_t n_l1, n_l2;                   // level-1 / level-2 doubles items of the CTA
  // scan scratch (4 lanes)
  uint32_t part[4][NT], base[4][NT], ws[4][36];
};

template <class BaseT>
struct ItemIter {  // items (parent e, bit p) over masks[e], parents ascending, bits descending
  int e, j, j1;
  uint32_t rem;
  NHD void init(const uint32_t* masks, const BaseT* base, int nparent, int j0, int j1_) {
    j = j0;
    j1 = j1_;
    e = 0;
    rem = 0;
    if (j >= j1) return;
    int lo = 0, hi = nparent - 1;
    while (lo < hi) {
      int mid = (lo + hi + 1) >> 1;
      if ((int)base[mid] <= j0)
        lo = mid;
      else
        hi = mid - 1;
    }
    e = lo;
    rem = masks[e];
    for (int k = j0 - (int)base[e]; k > 0; k--) rem &= ~(1u << fls32(rem));
  }
  NHD bool next(const uint32_t* masks, int* eo, int* po) {
    if (j >= j1) return false;
    while (rem == 0u) {
      e++;
      rem = masks[e];
    }
    int p = fls32(rem);
    rem &= ~(1u << p);
    *eo = e;
    *po = p;
    j++;
    return true;
  }
};

// DEFER = true: order-dependent doubles turns are handed to the exact CTA-per-env kernel (the caller
// gave a workspace) and the inline exact walk is not even compiled into the kernel (smaller code).
template <int BLK, bool DEFER = true, int NT = BLK>
struct BlockStep {
  typedef BlockShared<BLK, NT> Sh;
  static_assert(NT >= BLK && NT % 32 == 0 && BLK % 32 == 0, "threads per CTA: a multiple of 32, at least one per env");
  static constexpr int PER = NT / 32;  // partial sums per scan lane

  static NHD Pos pos_of(const Sh& sh, int e) {
    Pos P;
    P.lo = (uint64_t)sh.nlo0[e] | ((uint64_t)sh.nlo1[e] << 32);
    P.hi = sh.nhi[e];
    P.own = sh.own[e];
    P.opp = sh.opp[e];
    return P;
  }
  static NHD int head_budget(const Sh& sh, int e) {
    int d = sh.a[e];
    return (sh.first[e] && (d == 3 || d == 4 || d == 6)) ? 2 : 1;  // narde.py:100-103, per turn
  }
  static NHD void chunk(int total, int tid, int* j0, int* j1) {
    int c = (total + NT - 1) / NT;
    int a = tid * c, b = a + c;
    *j0 = a < total ? a : total;
    *j1 = b < total ? b : total;
  }

  // ---- phase 1: load, dice, decode, classify, item masks --------------------------------
  // bulk_words: the CTA's action words are arriving in sh.rnd through a bulk asynchronous copy (see the kernel)
  static NHD void ph_load(int tid, Sh& sh, bool valid, const State& s_in, int64_t i, const StepFullArgs& A,
                          bool bulk_words = false) {
    // the policy's choice may live in pinned HOST memory (zero-copy step_host): issue that load first and consume
    // it last, so that the microseconds of PCIe latency overlap everything else this phase does
    uint32_t policy_word = 0;
    if (valid && A.action_idx && !bulk_words) policy_word = (uint32_t)A.action_idx[i];
    for (int l = 0; l < 4; l++) sh.part[l][tid] = 0;
    if (NT > BLK && tid >= BLK) return;  // threads beyond the envs only take part in the item phases
    sh.rowmask[tid] = 0;
    sh.dmask[tid] = 0;
    sh.chosen[tid] = ACT_EMPTY;
    sh.etotal[tid] = 0;
    sh.ebase[tid] = 0;
    sh.maxd[tid] = 0;
    sh.defer[tid] = 0;
    sh.kind[tid] = K_NONE;
    if (!valid) return;
    sh.st[tid] = s_in;
    if (s_in.flags() & FLAG_DONE) {
      sh.kind[tid] = K_DONE;
      return;
    }
    uint32_t env = (uint32_t)(A.env_base + i);
    U4 rnd = turn_random(A.seed, env, A.step);
    int d1, d2;
    if (A.dice_in) {
      d1 = A.dice_in[2 * i];
      d2 = A.dice_in[2 * i + 1];
    } else {
      d1 = die_from_word(rnd.x);
      d2 = die_from_word(rnd.y);
    }
    sh.d1[tid] = (uint8_t)d1;
    sh.d2[tid] = (uint8_t)d2;
    int player = s_in.turn();
    bool first_turn = (s_in.flags() & (player == 1 ? FLAG_FIRST_W : FLAG_FIRST_B)) != 0;
    uint32_t ones;
    Pos P = decode_pos(s_in, player, &ones);
    int a = d1 > d2 ? d1 : d2, b = d1 > d2 ? d2 : d1;
    sh.a[tid] = (uint8_t)a;
    sh.b[tid] = (uint8_t)b;
    sh.first[tid] = first_turn ? 1 : 0;
    sh.own[tid] = P.own;
    sh.opp[tid] = P.opp;
    sh.ones[tid] = ones;
    sh.nlo0[tid] = (uint32_t)P.lo;
    sh.nlo1[tid] = (uint32_t)(P.lo >> 32);
    sh.nhi[tid] = P.hi;
    // the 6-prime block rule can only matter for ~4% of positions; those take the exact
    // (nibble-board) arithmetic, everything else the mask-only fast path
    bool blk = !block_rule_irrelevant(P, d1, d2);
#if defined(__CUDA_ARCH__) && defined(NARDE_DEBUG_HOOKS)
    if (g_dbg_flags & 1) blk = false;  // timing experiment only (wrong results when the rule matters)
#endif
    sh.blk[tid] = blk ? 1 : 0;
    if (a != b) {
      sh.kind[tid] = K_ND;
      uint32_t Ca = cand_mask(P.own, P.opp, a, true);
      uint32_t S = cand_mask(P.own, P.opp, b, true);
      if (blk) {
        Ca = block_filter(P, Ca, a);
        S = block_filter(P, S, b);
      }
      uint32_t q_home = 0, outside = P.own & ~0x3Fu;
      if (outside == 0u) {
        q_home = S;
      } else if ((outside & (outside - 1u)) == 0u) {
        int qo = ctz32(outside);
        if ((ones & outside) && qo - b < 6) q_home = S & outside;
      }
      sh.Ca[tid] = Ca;
      sh.S[tid] = S;
      sh.qhome[tid] = q_home;
      uint32_t rows = (P.own | (S >> b)) & 0xFFFFFFu;
      sh.rowmask[tid] = rows;
      sh.part[0][tid] = (uint32_t)popc32(rows);
    } else {
      sh.kind[tid] = K_D;
      uint32_t m = cand_mask(P.own, P.opp, a, true);
      sh.dmask[tid] = m;
      sh.part[1][tid] = (uint32_t)popc32(m);
    }
    if (!bulk_words) sh.rnd[tid] = A.action_idx ? policy_word : rnd.z;  // the policy's choice, or the turn's uniform word
  }

  // ---- block exclusive scan of part[l] -> base[l], totals in ws[l][32] ----------------------
  // One phase.  On the device warp l scans lane l with shuffles (BLK = 128: four
  // warps, four lanes); the host harness runs the plain serial scan.  lanes: bit mask of the lanes needed.
  static NHD void ph_scan_serial(int tid, Sh& sh, uint32_t lanes) {
#if defined(__CUDA_ARCH__)
    const int lane = tid & 31;
    for (int l = tid >> 5; l < 4; l += NT / 32) {  // a warp per scan lane (NT = 128), fewer warps take several
      if (!((lanes >> l) & 1u)) continue;
      uint32_t v[PER], sum = 0;
#pragma unroll
      for (int k = 0; k < PER; k++) {
        v[k] = sh.part[l][lane * PER + k];
        sum += v[k];
      }
      uint32_t incl = sum;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
        if (lane >= o) incl += t;
      }
      uint32_t r = incl - sum;
#pragma unroll
      for (int k = 0; k < PER; k++) {
        sh.base[l][lane * PER + k] = r;
        r += v[k];
      }
      if (lane == 31) sh.ws[l][32] = incl;
    }
#else
    if (tid >= 4 || !((lanes >> tid) & 1u)) return;
    const int l = tid;
    uint32_t r = 0;
    for (int k = 0; k < NT; k++) {
      uint32_t t = sh.part[l][k];
      sh.base[l][k] = r;
      r += t;
    }
    sh.ws[l][32] = r;
#endif
  }
  // after the first scan: bases of the ND row items and of the doubles level-1 items
  static NHD void ph_item_bases(int tid, Sh& sh) {
    if (NT > BLK && tid >= BLK) return;
    sh.ibase[tid] = sh.base[0][tid];
    sh.dbase[tid] = sh.base[1][tid];
    // item table of the pair rows: every later phase deals out [j0, j1) and reads (env, point) from here
    // instead of searching the per-env bases and walking bit masks (17 % of the warp samples before)
    uint32_t j = sh.base[0][tid];
    for (uint32_t m = sh.rowmask[tid]; m;) {
      int p = fls32(m);
      m &= ~(1u << p);
      sh.itab[j++] = (uint16_t)((tid << 5) | p);
    }
    // doubles level-1 items (env, first source): same idea, straight into the l1env / l1src tables
    uint32_t jd = sh.base[1][tid];
    if (sh.ws[1][32] <= (uint32_t)Sh::kL1Cap) {
      for (uint32_t m = sh.dmask[tid]; m;) {
        int p = fls32(m);
        m &= ~(1u << p);
        sh.l1env[jd] = (uint8_t)tid;
        sh.l1src[jd] = (uint8_t)p;
        jd++;
      }
    }
    if (tid == 0) {
      sh.ibase[BLK] = sh.ws[0][32];
      sh.dbase[BLK] = sh.ws[1][32];
      uint32_t n1 = sh.ws[1][32];
      sh.n_l1 = n1 <= (uint32_t)Sh::kL1Cap ? n1 : 0u;  // overflow: doubles envs fall back to the sequential walk
    }
  }

  // ---- non-doubles row arithmetic -----------------------------------------------------------
  static NHD void nd_row(const Sh& sh, int e, int p, uint32_t* m1_out, uint32_t* m2_out) {
    uint32_t own = sh.own[e], opp = sh.opp[e], ones = sh.ones[e], S = sh.S[e];
    int a = sh.a[e], b = sh.b[e];
    uint32_t bp = 1u << p;
    int ta = p - a;
    uint32_t m1 = 0;
    if (sh.Ca[e] & bp) {  // p moves a first, then q moves b on the resulting board
      uint32_t own1 = (own & ~(ones & bp)) | (ta >= 0 ? (1u << ta) : 0u);
      m1 = cand_mask(own1, opp, b, p != 23);
    }
    uint32_t m2;  // q in S moves b first, then p moves a
    if (own & bp) {
      m2 = S & ~(ones & bp);
    } else {
      m2 = p + b < 24 ? (S & (1u << (p + b))) : 0u;
    }
    if (ta >= 0) {
      if ((opp >> ta) & 1u) m2 = 0;
    } else {
      m2 &= sh.qhome[e];
    }
    if (p == 23) m2 &= ~(1u << 23);
    if (sh.blk[e]) {  // exact path: every intermediate and final board is tested (narde.py:78-89)
      Pos P = pos_of(sh, e);
      m1 = 0;
      if (sh.Ca[e] & bp) {
        Pos P1 = P;
        P1.move(p, ta);
        m1 = block_filter(P1, cand_mask(P1.own, P1.opp, b, p != 23), b);
      }
      uint32_t keep = 0;
      for (uint32_t mm = m2 & ~m1; mm; mm &= mm - 1) {
        int q = ctz32(mm);
        Pos Q = P;
        Q.move(q, q - b);
        if (!violates_block(after_mask(Q, p, ta), Q.opp)) keep |= 1u << q;
      }
      m2 = keep | (m2 & m1);
    }
    *m1_out = m1;
    *m2_out = m2;
  }
  // the m1 half of nd_row alone (which pairs can be played with p's higher-die move first): all the emit
  // phase needs to order a pair's two half-moves
  static NHD uint32_t nd_m1(const Sh& sh, int e, int p) {
    const uint32_t bp = 1u << p;
    if (!(sh.Ca[e] & bp)) return 0u;
    const int b = sh.b[e], ta = p - sh.a[e];
    if (sh.blk[e]) {
      Pos P1 = pos_of(sh, e);
      P1.move(p, ta);
      return block_filter(P1, cand_mask(P1.own, P1.opp, b, p != 23), b);
    }
    uint32_t own1 = (sh.own[e] & ~(sh.ones[e] & bp)) | (ta >= 0 ? (1u << ta) : 0u);
    return cand_mask(own1, sh.opp[e], b, p != 23);
  }
  // pairs of row p that duplicate a pair of a higher row (see enum_nondouble)
  static NHD uint32_t nd_dups(const Sh& sh, int e, int p) {
    int a = sh.a[e], b = sh.b[e];
    uint32_t dup = 0;
    int x = p + b;
    if (x < 24 && x - a >= 0 && ((sh.pres[e * 24 + x] >> (x - a)) & 1u)) dup |= 1u << x;
    if (p < b)
      for (int q = p + 1; q < b; q++)
        if ((sh.pres[e * 24 + q] >> p) & 1u) dup |= 1u << q;
    return dup;
  }

  // ---- doubles sub-tree below the two highest sources (s1 >= s2) ----------------------------
  // fast variant (block rule irrelevant): count the 4-move leaves; *deep = 3 if a third move exists
  // detect = true (block rule may matter): also test every board on the way; *taint is set when one
  // violates -- then orderings matter and the env is handed to the exact CTA-per-env kernel.  When no
  // board of the tree violates, highest-source-first play is legal for every multiset and the rule
  // changes nothing, so the fast result is exact.
  static NHD uint32_t dbl_count2(const Pos& P, int d, int H, int s1, int s2, uint32_t* deep, bool detect = false,
                                 uint32_t* taint = nullptr) {
    Pos P2 = P;
    P2.move(s1, s1 - d);
    if (detect && violates_block(P2.own, P2.opp)) {
      *taint = 1;
      return 0;
    }
    P2.move(s2, s2 - d);
    if (detect && violates_block(P2.own, P2.opp)) {
      *taint = 1;
      return 0;
    }
    int h2 = (s1 == 23) + (s2 == 23);
    uint32_t leaves = 0;
    uint32_t m3 = cand_mask(P2.own, P2.opp, d, h2 < H) & ((2u << s2) - 1u);
    *deep = m3 ? 3u : 2u;
    while (m3) {
      int s3 = fls32(m3);
      m3 &= ~(1u << s3);
      Pos P3 = P2;
      P3.move(s3, s3 - d);
      int h3 = h2 + (s3 == 23);
      uint32_t m4 = cand_mask(P3.own, P3.opp, d, h3 < H) & ((2u << s3) - 1u);
      if (detect) {
        if (violates_block(P3.own, P3.opp)) {
          *taint = 1;
          return 0;
        }
        for (uint32_t r = m4 & (completing_points(P3.own, P3.opp) << d); r; r &= r - 1) {
          int s4 = ctz32(r);
          if (violates_block(after_mask(P3, s4, s4 - d), P3.opp)) {
            *taint = 1;
            return 0;
          }
        }
      }
      leaves += (uint32_t)popc32(m4);
    }
    return leaves;
  }
  static NHD uint32_t dbl_emit2(const Pos& P, int d, int H, int s1, int s2, uint32_t off, uint64_t* slice, int cap,
                                uint32_t idx, uint64_t* chosen) {
    Pos P2 = P;
    P2.move(s1, s1 - d);
    P2.move(s2, s2 - d);
    int h2 = (s1 == 23) + (s2 == 23);
    uint64_t a2 = act_set(act_set(ACT_EMPTY, 0, s1, s1 - d), 1, s2, s2 - d);
    uint32_t k = off;
    uint32_t m3 = cand_mask(P2.own, P2.opp, d, h2 < H) & ((2u << s2) - 1u);
    while (m3) {
      int s3 = fls32(m3);
      m3 &= ~(1u << s3);
      Pos P3 = P2;
      P3.move(s3, s3 - d);
      int h3 = h2 + (s3 == 23);
      uint64_t a3 = act_set(a2, 2, s3, s3 - d);
      uint32_t m4 = cand_mask(P3.own, P3.opp, d, h3 < H) & ((2u << s3) - 1u);
      while (m4) {
        int s4 = fls32(m4);
        m4 &= ~(1u << s4);
        uint64_t a4 = act_set(a3, 3, s4, s4 - d);
        if (slice && (int)k < cap) slice[k] = a4;
        if (k == idx) *chosen = a4;
        k++;
      }
    }
    return k - off;
  }
  // exact variant (the block rule may matter, narde.py:78-89,139-184): same walk, but every board on
  // the way is tested.  A multiset is legal iff SOME ordering keeps all intermediate boards legal;
  // highest-source-first is tried implicitly (desc), any other ordering by dbl_order_search, which
  // is only reached below a violating prefix.  Leaves are tested on occupancy masks only.
  // EMIT = false: returns the number of legal 4-move leaves.  EMIT = true: also writes them.
  static NHD bool order_search_dbg(const Pos& P, const int* src, int k, int d, int H, int* order) {
#if defined(__CUDA_ARCH__) && defined(NARDE_DEBUG_HOOKS)
    if (g_dbg_flags & 2) {  // timing experiment only
      for (int i = 0; i < k; i++) order[i] = src[i];
      return false;
    }
#endif
    return dbl_order_search(P, src, k, d, H, order);
  }
  template <bool EMIT>
  static NHD uint32_t dbl_exact2(const Pos& P, int d, int H, int s1, int s2, uint32_t off, uint64_t* slice, int cap,
                                 uint32_t idx, uint64_t* chosen) {
    int src[4], order[4];
    src[0] = s1;
    src[1] = s2;
    Pos P1 = P;
    P1.move(s1, s1 - d);
    bool v1 = violates_block(P1.own, P1.opp);
    Pos P2 = P1;
    P2.move(s2, s2 - d);
    if (violates_block(P2.own, P2.opp)) {
      // (s1, s2) itself is not a legal pair in any order, but longer multisets containing it may be
      // reachable through other sub-multisets: handled per node by the ordering search below
    }
    bool v2 = violates_block(P2.own, P2.opp);
    bool desc2 = !v1 && !v2;
    bool reach2 = !v2 && (!v1 || order_search_dbg(P, src, 2, d, H, order));
    int h2 = (s1 == 23) + (s2 == 23);
    uint32_t k = off;
    uint32_t m3 = cand_mask(P2.own, P2.opp, d, h2 < H) & ((2u << s2) - 1u);
    while (m3) {
      int s3 = fls32(m3);
      m3 &= ~(1u << s3);
      src[2] = s3;
      Pos P3 = P2;
      P3.move(s3, s3 - d);
      bool v3 = violates_block(P3.own, P3.opp);
      bool desc3 = desc2 && !v3;
      bool reach3 = !v3 && (reach2 || order_search_dbg(P, src, 3, d, H, order));
      int h3 = h2 + (s3 == 23);
      uint32_t m4 = cand_mask(P3.own, P3.opp, d, h3 < H) & ((2u << s3) - 1u);
      // leaves that cannot violate: the board is legal and the move does not land on a completing point
      uint32_t risky = v3 ? m4 : (m4 & (completing_points(P3.own, P3.opp) << d));
      if (!EMIT && reach3) {  // counting below a reachable node: only the risky leaves need a look
        k += (uint32_t)popc32(m4 & ~risky);
        m4 = risky;
      }
      while (m4) {
        int s4 = fls32(m4);
        m4 &= ~(1u << s4);
        if (((risky >> s4) & 1u) && violates_block(after_mask(P3, s4, s4 - d), P3.opp)) continue;
        src[3] = s4;
        bool searched = false;
        if (!reach3) {
          if (!order_search_dbg(P, src, 4, d, H, order)) continue;
          searched = true;
        }
        if (EMIT) {
          bool hit = k == idx;
          if (hit || (slice && (int)k < cap)) {
            uint64_t act = ACT_EMPTY;
            if (desc3) {
              for (int i = 0; i < 4; i++) act = act_set(act, i, src[i], src[i] - d);
            } else {  // representative = first legal ordering, higher sources tried first
              if (!searched) order_search_dbg(P, src, 4, d, H, order);
              for (int i = 0; i < 4; i++) act = act_set(act, i, order[i], order[i] - d);
            }
            if (slice && (int)k < cap) slice[k] = act;
            if (hit) *chosen = act;
          }
        }
        k++;
      }
    }
    return k - off;
  }
  static NHD uint32_t dbl_count2_exact(const Pos& P, int d, int H, int s1, int s2) {
    return dbl_exact2<false>(P, d, H, s1, s2, 0, nullptr, 0, 0xFFFFFFFFu, nullptr);
  }

  // ---- phase 3: ND rows -> pres ; doubles level-1 items -> second-source masks -------------
  static NHD void ph_rows(int tid, Sh& sh) {
    constexpr bool deferral = DEFER;
    int j0, j1, e, p;
    chunk((int)sh.ibase[BLK], tid, &j0, &j1);
    for (int jj = j0; jj < j1; jj++) {
      const uint32_t v = sh.itab[jj];
      e = (int)(v >> 5);
      p = (int)(v & 31u);
      uint32_t m1, m2;
      nd_row(sh, e, p, &m1, &m2);
      sh.pres[e * 24 + p] = m1 | m2;
    }
    chunk((int)sh.n_l1, tid, &j0, &j1);
    uint32_t sum = 0;
    for (int j = j0; j < j1; j++) {
      e = sh.l1env[j];
      p = sh.l1src[j];
      int d = sh.a[e];
      Pos P1 = pos_of(sh, e);
      P1.move(p, p - d);
      uint32_t m2 = cand_mask(P1.own, P1.opp, d, (p == 23) < head_budget(sh, e)) & ((2u << p) - 1u);
      sh.d2mask[j] = m2;
      if (!sh.blk[e] || deferral) sm_max(&sh.maxd[e], m2 ? 2u : 1u);
      if (sh.blk[e] && deferral && violates_block(P1.own, P1.opp)) sm_max(&sh.defer[e], 1u);
      sum += (uint32_t)popc32(m2);
    }
    sh.part[1][tid] = sum;
  }
  // level-2 doubles items share the item table with the pair rows when both fit (they practically always do;
  // otherwise the phases fall back to the searching iterator)
  static NHD bool l2_in_table(const Sh& sh, uint32_t n_l2) {
#if defined(NARDE_HOSTSIM_HOOKS) && !defined(__CUDA_ARCH__)
    if (g_hs_force_slow & 1) return false;  // test-only (tests/hostsim): exercise the searching iterator
#endif
    return sh.n_l1 > 0 && sh.n_l1 < 1024u && sh.ibase[BLK] + n_l2 <= (uint32_t)(BLK * 24);
  }
  // Per level-2 item, 16 bits: its action count (written by ph_count), then its offset inside the env's list
  // (ph_env_bases).  The array lives on top of d2mask / d2base, which nobody reads once the items are in the table.
  // With it the emit phase deals the items round-robin (a heavy env's items spread over all warps instead of
  // sitting in one thread's contiguous chunk) and skips, without recounting, every item that lies beyond the
  // stored capacity and does not hold the chosen action.
  static constexpr uint32_t kL2OffCap = (uint32_t)((sizeof(uint32_t) * (2 * Sh::kL1Cap + 1)) / sizeof(uint16_t));
  static NHD bool l2_fast(const Sh& sh) {
#if defined(NARDE_HOSTSIM_HOOKS) && !defined(__CUDA_ARCH__)
    if (g_hs_force_slow & 2) return false;  // test-only (tests/hostsim): exercise the recounting emit
#endif
    return l2_in_table(sh, sh.n_l2) && sh.n_l2 <= kL2OffCap;
  }
  static NHD uint16_t* l2_off(Sh& sh) { return reinterpret_cast<uint16_t*>(sh.d2mask); }
  struct L2Iter {  // items (level-1 item j, second source p) of [j0, j1): from the table, else by searching
    bool tab;
    int jj, j1;
    uint32_t t0;
    ItemIter<uint32_t> it;
    NHD void init(const Sh& sh, int j0, int j1_) {
      const int n1 = (int)sh.n_l1;
      tab = l2_in_table(sh, sh.n_l2);
      jj = j0;
      j1 = j1_;
      t0 = sh.ibase[BLK];
      if (!tab) it.init(sh.d2mask, sh.d2base, n1, j0, j1_);
    }
    NHD bool next(const Sh& sh, int* j, int* p) {
      if (!tab) return it.next(sh.d2mask, j, p);
      if (jj >= j1) return false;
      const uint32_t v = sh.itab[t0 + (uint32_t)jj++];
      *j = (int)(v >> 5);
      *p = (int)(v & 31u);
      return true;
    }
  };
  // after the scan of level-2 counts: per level-1 item bases
  static NHD void ph_l2_bases(int tid, Sh& sh) {
    int j0, j1;
    chunk((int)sh.n_l1, tid, &j0, &j1);
    uint32_t r = sh.base[1][tid];
    // level-2 items (level-1 item, second source) go into the free tail of the item table when they fit
    const uint32_t t0 = sh.ibase[BLK];
    const bool tab = l2_in_table(sh, sh.ws[1][32]);
    for (int j = j0; j < j1; j++) {
      sh.d2base[j] = r;
      uint32_t m = sh.d2mask[j];
      if (tab) {
        uint32_t k = t0 + r;
        for (uint32_t mm = m; mm;) {
          int p = fls32(mm);
          mm &= ~(1u << p);
          sh.itab[k++] = (uint16_t)((j << 5) | p);
        }
      }
      r += (uint32_t)popc32(m);
    }
    if (tid == 0) {
      sh.d2base[sh.n_l1] = sh.ws[1][32];
      sh.n_l2 = sh.ws[1][32];
    }
  }
  // ---- phase 5: counts per item -> chunk sums (lanes 0/1) and per-env totals ----------------
  static NHD void ph_count(int tid, Sh& sh) {
    constexpr bool deferral = DEFER;
    int j0, j1, e, p;
    chunk((int)sh.ibase[BLK], tid, &j0, &j1);
    uint32_t sum = 0;
    for (int jj = j0; jj < j1; jj++) {
      const uint32_t v = sh.itab[jj];
      e = (int)(v >> 5);
      p = (int)(v & 31u);
      // De-duplicate IN PLACE so that the emit phase reads the final mask.  This is race-free although other
      // threads test bits of this row in nd_dups at the same time: only bits ABOVE the row index are ever
      // removed from a row (bit p+b, bits q in (p, b)), and only bits BELOW the row index are ever tested
      // (row x bit x-a, row q bit p < q), so a tested bit has the same value before and after.
      uint32_t nd = sh.pres[e * 24 + p] & ~nd_dups(sh, e, p);
      sh.pres[e * 24 + p] = nd;
      uint32_t c = (uint32_t)popc32(nd);
      if (c) sm_add(&sh.etotal[e], c);
      sum += c;
    }
    sh.part[0][tid] = sum;
    int n1 = (int)sh.n_l1;
    sum = 0;
    if (n1 > 0) {
      chunk((int)sh.n_l2, tid, &j0, &j1);
      const bool fast = l2_fast(sh);
      uint16_t* cnt16 = l2_off(sh);
      L2Iter it2;
      it2.init(sh, j0, j1);
      int j, t = j0;
      while (it2.next(sh, &j, &p)) {
        e = sh.l1env[j];
        int s1 = sh.l1src[j];
        uint32_t c;
        if (!deferral && sh.blk[e]) {
          if constexpr (!DEFER) c = dbl_count2_exact(pos_of(sh, e), sh.a[e], head_budget(sh, e), s1, p);
        } else {
          uint32_t deep = 0, taint = 0;
          c = dbl_count2(pos_of(sh, e), sh.a[e], head_budget(sh, e), s1, p, &deep, sh.blk[e] != 0, &taint);
          if (taint) sm_max(&sh.defer[e], 1u);
          if (c == 0) sm_max(&sh.maxd[e], deep);
        }
        if (c) sm_add(&sh.etotal[e], c);
        if (fast) cnt16[t] = (uint16_t)c;  // <= 24 * 24 leaves per item
        t++;
        sum += c;
      }
    }
    sh.part[1][tid] = sum;
  }
  // the same count again, without side effects (emit phase of the rare CTA whose items did not fit the tables)
  static NHD_NOINLINE uint32_t recount_item(const Sh& sh, int e, int s1, int p) {
    if (!DEFER && sh.blk[e]) {
      if constexpr (!DEFER) return dbl_count2_exact(pos_of(sh, e), sh.a[e], head_budget(sh, e), s1, p);
    }
    uint32_t deep = 0, taint = 0;
    return dbl_count2(pos_of(sh, e), sh.a[e], head_budget(sh, e), s1, p, &deep, sh.blk[e] != 0, &taint);
  }
  // per-env totals into scan lanes 2 (ND) / 3 (doubles): list starts in item space
  static NHD void ph_env_totals(int tid, Sh& sh) {
    if (NT > BLK && tid >= BLK) return;  // part[2], part[3] of those threads stay 0 (ph_load)
    uint8_t k = sh.kind[tid];
    sh.part[2][tid] = k == K_ND ? sh.etotal[tid] : 0u;
    sh.part[3][tid] = k == K_D ? sh.etotal[tid] : 0u;
  }
  // hand-over of order-dependent doubles turns: the list is complete once every CTA is past this
  // phase, which is when the exact kernel (a programmatic dependent launch) may start
  static NHD void ph_defer_push(int tid, const Sh& sh, bool valid, int64_t i, const StepFullArgs& A) {
    // entry = env index + 1: a zero word is "not published yet" (the exact kernel consumes entries while the main
    // kernel is still producing them and puts the zero back)
    if (valid && sh.defer[tid]) {
#if defined(__CUDA_ARCH__)
      *reinterpret_cast<volatile int32_t*>(A.defer_list + gl_fetch_add(A.defer_count, 1)) = (int32_t)i + 1;
#else
      A.defer_list[gl_fetch_add(A.defer_count, 1)] = (int32_t)i + 1;
#endif
    }
  }
  static NHD void ph_env_bases(int tid, Sh& sh) {
    if (NT == BLK || tid < BLK) sh.ebase[tid] = sh.kind[tid] == K_ND ? sh.base[2][tid] : sh.base[3][tid];
    {  // pair rows: the row's offset inside its env's list goes into the free top byte of its mask (a non-doubles
       // turn has < 15 x 17 legal pairs), so the emit phase can deal the rows round-robin
      int j0, j1;
      chunk((int)sh.ibase[BLK], tid, &j0, &j1);
      uint32_t G = sh.base[0][tid];
      for (int jj = j0; jj < j1; jj++) {
        const uint32_t v = sh.itab[jj];
        const int e = (int)(v >> 5), p = (int)(v & 31u);
        const uint32_t nd = sh.pres[e * 24 + p];
        sh.pres[e * 24 + p] = nd | ((G - sh.base[2][e]) << 24);
        G += (uint32_t)popc32(nd);
      }
    }
    if (sh.n_l1 > 0 && l2_fast(sh)) {  // level-2 item counts -> offsets inside the env's list (lane 3 = doubles env starts)
      int j0, j1;
      chunk((int)sh.n_l2, tid, &j0, &j1);
      uint16_t* off16 = l2_off(sh);
      const uint32_t t0 = sh.ibase[BLK];
      uint32_t G = sh.base[1][tid];
      for (int t = j0; t < j1; t++) {
        const int e = sh.l1env[sh.itab[t0 + (uint32_t)t] >> 5];
        const uint32_t c = off16[t];
        off16[t] = (uint16_t)(G - sh.base[3][e]);
        G += c;
      }
    }
  }
  static NHD uint32_t pick_index(const Sh& sh, int e, int64_t i, uint32_t count, const StepFullArgs& A) {
    return pick_from_word(A, sh.rnd[e], count);
  }
  // ---- phase 7: write the action lists in canonical order, capture the chosen action ------
  static NHD void ph_emit(int tid, Sh& sh, int64_t row0, const StepFullArgs& A) {
    int j0, j1, e, p;
    uint32_t G = 0;
    const int n_nd = (int)sh.ibase[BLK];
    for (int jj = tid; jj < n_nd; jj += NT) {  // round-robin: neighbouring threads write neighbouring list slots
      const uint32_t v = sh.itab[jj];
      e = (int)(v >> 5);
      p = (int)(v & 31u);
      const uint32_t w = sh.pres[e * 24 + p];  // de-duplicated by ph_count, offset added by ph_env_bases
      uint32_t nd = w & 0xFFFFFFu;
      uint32_t cnt = (uint32_t)popc32(nd);
      uint32_t off = w >> 24;
      if (cnt == 0) continue;
      uint32_t idx = pick_index(sh, e, row0 + e, sh.etotal[e], A);
      uint64_t* slice = A.actions ? A.actions + (row0 + e) * (int64_t)A.cap : nullptr;
      bool want = idx >= off && idx < off + cnt;
      if (!want && (!slice || (int)off >= A.cap)) continue;
      const uint32_t m1 = nd_m1(sh, e, p);  // pairs playable "p with the higher die first"
      int a = sh.a[e], b = sh.b[e], ta = p - a;
      uint32_t k = off;
      const uint32_t hp = (uint32_t)p | ((ta < 0 ? 255u : (uint32_t)ta) << 8);  // half-move of the higher die
      while (nd) {
        int q = fls32(nd);
        nd &= ~(1u << q);
        int tb = q - b;
        uint32_t hq = (uint32_t)q | ((tb < 0 ? 255u : (uint32_t)tb) << 8);
        // two half-moves in slots 0,1 (played in that order), slots 2,3 unused (0xFFFF)
        uint32_t lo32 = ((m1 >> q) & 1u) ? (hp | (hq << 16)) : (hq | (hp << 16));
        uint64_t act = 0xFFFFFFFF00000000ull | lo32;
        if (slice && (int)k < A.cap) slice[k] = act;
        if (k == idx) sh.chosen[e] = act;
        k++;
      }
    }
    int n1 = (int)sh.n_l1;
    if (n1 > 0) {
      // level-2 doubles items.  Normal case: dealt round-robin, offset and count of an item read from the table
      // ph_env_bases left (an item beyond the stored capacity that does not hold the chosen action costs
      // nothing).  Fallback (tables did not fit): contiguous chunks, running offset, every item counted again.
      const bool fast = l2_fast(sh);
      const int n2 = (int)sh.n_l2;
      const uint16_t* off16 = l2_off(sh);
      const uint32_t t0 = sh.ibase[BLK];
      L2Iter it2;
      int t = tid, t1 = n2, dt = NT;
      if (!fast) {
        chunk(n2, tid, &j0, &j1);
        it2.init(sh, j0, j1);
        G = sh.base[1][tid];
        t = j0;
        t1 = j1;
        dt = 1;
      }
      for (; t < t1; t += dt) {
        int j;
        uint32_t off, cnt;
        if (fast) {
          const uint32_t v = sh.itab[t0 + (uint32_t)t];
          j = (int)(v >> 5);
          p = (int)(v & 31u);
        } else {
          it2.next(sh, &j, &p);
        }
        e = sh.l1env[j];
        const int s1 = sh.l1src[j];
        const uint32_t total = sh.etotal[e];
        if (fast) {
          if (total == 0 || sh.defer[e]) continue;  // cannot use four dice (ph_finish) / deferred to the exact kernel
          off = off16[t];
          uint32_t nxt = total;                     // the next item of the same env starts where this one ends
          if (t + 1 < n2 && sh.l1env[sh.itab[t0 + (uint32_t)t + 1u] >> 5] == e) nxt = off16[t + 1];
          cnt = nxt - off;
        } else {
          cnt = total ? recount_item(sh, e, s1, p) : 0u;  // what ph_count added for this item
          off = G - sh.ebase[e];
          G += cnt;
          if (total == 0 || sh.defer[e]) continue;
        }
        if (cnt == 0) continue;
        const uint32_t idx = pick_index(sh, e, row0 + e, total, A);
        uint64_t* slice = A.actions ? A.actions + (row0 + e) * (int64_t)A.cap : nullptr;
        if (!(slice && (int)off < A.cap)) {
          slice = nullptr;                          // nothing to store: walk only if the chosen index is inside
          if (!(idx >= off && idx < off + cnt)) continue;
        }
        const Pos P = pos_of(sh, e);
        const int d = sh.a[e], H = head_budget(sh, e);
        if (!DEFER && sh.blk[e] != 0) {
          if constexpr (!DEFER) dbl_exact2<true>(P, d, H, s1, p, off, slice, A.cap, idx, &sh.chosen[e]);
        } else {
          dbl_emit2(P, d, H, s1, p, off, slice, A.cap, idx, &sh.chosen[e]);
        }
      }
    }
  }

  // ---- phase 8: per-env completion: rare sequential cases, apply, outputs ------------------
  static NHD void ph_finish(int tid, Sh& sh, bool valid, int64_t i, const StepFullArgs& A, StepFullLocal& L) {
    L.count = 0;
    L.finished = L.white_win = L.black_win = L.mars = L.ep_len = L.overflow = L.clamped = L.result = 0;
    if (!valid) return;
    uint8_t kind = sh.kind[tid];
    if (kind == K_DONE) {
      idle_outputs(i, A);
      L.result = DONE_TERMINATED;  // a finished game without auto-reset stays terminated
      return;
    }
    if (sh.defer[tid]) return;  // handed to the exact CTA-per-env kernel (ph_defer_push); left untouched here
    State s = sh.st[tid];
    int player = s.turn();
    int a = sh.a[tid], b = sh.b[tid];
    uint64_t* slice = A.actions ? A.actions + (int64_t)i * A.cap : nullptr;
    uint32_t count = sh.etotal[tid];
    uint64_t act = sh.chosen[tid];
    if (kind == K_ND && count == 0) {
      // maximal length 1: the higher die if it can be played (narde.py:6 rule 4), else the lower
      uint32_t m = sh.Ca[tid] ? sh.Ca[tid] : sh.S[tid];
      int d = sh.Ca[tid] ? a : b;
      count = (uint32_t)popc32(m);
      uint32_t idx = pick_index(sh, tid, i, count, A);
      uint32_t k = 0;
      while (m) {
        int sp = fls32(m);
        m &= ~(1u << sp);
        uint64_t one = act_set(ACT_EMPTY, 0, sp, sp - d);
        if (slice && (int)k < A.cap) slice[k] = one;
        if (k == idx) act = one;
        k++;
      }
    } else if (kind == K_D && count == 0) {
      // a doubles turn that cannot use all four dice (~3% of turns): per-thread walk of a small tree
      Pos P = pos_of(sh, tid);
      bool ft = sh.first[tid] != 0;
      int target = (int)sh.maxd[tid];
      bool known = (!sh.blk[tid] || DEFER) && sh.n_l1 > 0;  // depth found by the item phases
      act = ACT_EMPTY;
      if (sh.dmask[tid] == 0u || (known && target == 0)) {
        count = 0;  // no playable die: the turn is passed
      } else {
        // store + count pass; a second (pick) pass only when the chosen action was not stored.  The
        // common case (depth known) is inlined once inside this two-trip loop, the rest out of line.
        WalkSink sk = {slice, slice ? A.cap : 0, -1, 0, ACT_EMPTY};
        const int H = head_budget(sh, tid);
#pragma unroll 1
        for (int pass = 0; pass < 2; pass++) {
          int n = known ? enum_double_at(P, a, H, target, sk) : walk_short_double(P, a, ft, H, target, false, sk);
          if (pass == 1) {
            act = sk.picked;
            break;
          }
          count = (uint32_t)n;
          if (n == 0) break;
          uint32_t idx = pick_index(sh, tid, i, count, A);
          if (slice && (int)idx < A.cap) {
            act = slice[idx];
            break;
          }
          sk.out = nullptr;
          sk.cap = 0;
          sk.want = (int)idx;
          sk.n = 0;
        }
      }
    }
    complete_env(s, i, A, player, count, act, sh.d1[tid], sh.d2[tid], L);
    L.clamped = index_was_clamped(A, sh.rnd[tid], count);  // (sh.rnd holds the caller's word when action_idx was given)
    sh.st[tid] = s;
  }
};

}  // namespace narde
