// narde_deferred.cuh -- exact doubles turns when the 6-prime block rule bites (one small CTA per env).
//
// The block kernel (narde_block.cuh) hands over the rare doubles turns (~0.2% of env steps in self-play, 2% of
// the doubles-heavy microbench) in which some board of the move tree violates the block rule
// (narde.py:139-184): there the set of playable source multisets depends on the ORDER of the half-moves.
//
// What the rule text says (narde.py:64-89, max-dice rule narde.py:4-6): a multiset of j sources is playable
// iff SOME ordering of it is a sequence of legal half-moves through legal boards; the turn's actions are the
// playable multisets of the deepest level that has any.  Two facts make this cheap:
//   * without the block rule, playing a multiset highest source first is legal whenever any order is
//     (arrivals precede departures, checkers are home as early as possible), so the multisets the FAST walk
//     finds (cand_mask on highest-first boards, no board test) are a superset of the playable ones at every
//     depth, and the walk yields them once each, already in canonical order;
//   * whether one candidate is playable is an independent, bounded question: the final board must be legal,
//     then highest-first is tried, else a depth-first search over its orderings (higher sources first -> the
//     representative ordering) that remembers dead sub-multisets (a board depends only on the sub-multiset,
//     so at most 2^4 of them are ever expanded).
// So a team of NT threads owns one environment: the candidates of the deepest fast level are written into
// shared memory (thread-parallel over the (s1, s2) items), tested one per thread with no barrier in between,
// the survivors ranked by one block scan, the first `cap` actions and the chosen one stored.  No survivor at
// that depth -> the next shallower level.
// (Round 1 ran a level-synchronous breadth-first search over multiset bitmaps with one 256-thread CTA per
// env: 40-48 k cycles per env behind 25 CTA barriers, most lanes idle.  Typical trees have tens of leaves.)
//
// Written as phases like narde_block.cuh: `ex.run(f)` runs f(tid) for the NT threads of the team and then
// synchronises them; everything that crosses threads goes through the team's shared-memory record.  The
// test-only host harness runs the same driver with a loop over tids.
#pragma once
#include "narde_block.cuh"

namespace narde {

constexpr int kExItems = 300;    // (s1, s2) items: 2-multisets of 24 sources
constexpr int kExWindow = 1024;  // candidates tested per pass over the tree (more -> several windows)
NHD uint32_t ex_window() {
#if defined(NARDE_HOSTSIM_HOOKS) && !defined(__CUDA_ARCH__)
  if (g_hs_force_slow & 4) return 8u;  // test-only (tests/hostsim): several windows per level on ordinary positions
#endif
  return (uint32_t)kExWindow;
}

NHD uint32_t sm_fetch_or(uint32_t* p, uint32_t v) {
#if defined(__CUDA_ARCH__)
  return atomicOr(p, v);
#else
  uint32_t o = *p;
  *p |= v;
  return o;
#endif
}

template <int NT>
struct ExactSharedT {
  State st;
  uint32_t own, opp, nlo0, nlo1, nhi;
  int32_t d, H, player, d1, d2;
  uint32_t rnd;
  uint32_t m1;                   // level-1 candidate sources
  uint32_t n_items;              // (s1, s2) items
  uint32_t deep;                 // bit j: the fast tree has a level j+1
  uint32_t n_cand;               // candidates of the level being tested
  uint32_t run;                  // playable multisets found so far in the pass over the level
  uint32_t count, idx;           // playable multisets of the final level; the one to play
  uint32_t found;                // the chosen action has been captured
  uint64_t chosen;
  uint32_t part[NT];
  uint32_t wsum[NT / 32 + 1];    // survivors per warp of a round (teams of several warps)
  uint16_t item[kExItems];       // s1 << 5 | s2, canonical order
  uint16_t c3[kExItems], c4[kExItems];  // per item: candidates at depth 3 / 4
  uint16_t ioff[kExItems + 1];   // exclusive scan of the tested level's per-item counts
  uint32_t cand[kExWindow];      // window of candidates (sources descending, 5 bits each) -> test results in place
};

template <int NT>
struct ExactStep {
  typedef ExactSharedT<NT> Sh;
  static constexpr uint32_t kPlayable = 0x80000000u;

  static NHD Pos base_pos(const Sh& sh) {
    Pos P;
    P.lo = (uint64_t)sh.nlo0 | ((uint64_t)sh.nlo1 << 32);
    P.hi = sh.nhi;
    P.own = sh.own;
    P.opp = sh.opp;
    return P;
  }
  static NHD_NOINLINE void ex_move(Pos& P, int s, int t) { P.move(s, t); }  // one copy of the half-move (code size)
  static NHD uint64_t action_of(uint32_t orderp, int j, int d) {
    uint64_t act = ACT_EMPTY;
#pragma unroll 1
    for (int t = 0; t < j; t++) {
      const int s = (int)((orderp >> (5 * t)) & 31u);
      act = act_set(act, t, s, s - d);
    }
    return act;
  }

  // ---- thread 0: load, decode; thread NT-1: the turn's random words ------------------------------------
  static NHD void ph_init(int tid, Sh& sh, const State& s_in, int64_t i, const StepFullArgs& A) {
    if (tid == NT - 1) {
      U4 rnd = turn_random(A.seed, (uint32_t)(A.env_base + i), A.step);
      int d1, d2;
      if (A.dice_in) {
        d1 = A.dice_in[2 * i];
        d2 = A.dice_in[2 * i + 1];
      } else {
        d1 = die_from_word(rnd.x);
        d2 = die_from_word(rnd.y);
      }
      sh.rnd = rnd.z;
      sh.d1 = d1;
      sh.d2 = d2;
      sh.d = d1;  // doubles: d1 == d2
    }
    if (tid != 0) return;
    sh.st = s_in;
    int player = s_in.turn();
    Pos P = decode_pos(s_in, player);
    sh.player = player;
    sh.own = P.own;
    sh.opp = P.opp;
    sh.nlo0 = (uint32_t)P.lo;
    sh.nlo1 = (uint32_t)(P.lo >> 32);
    sh.nhi = P.hi;
    sh.n_items = 0;
    sh.n_cand = 0;
    sh.run = 0;
    sh.count = 0;
    sh.idx = 0;
    sh.found = 0;
    sh.chosen = ACT_EMPTY;
  }
  static NHD void ph_init2(int tid, Sh& sh) {
    if (tid != 0) return;
    const int d = sh.d, player = sh.player;
    const bool first_turn = (sh.st.flags() & (player == 1 ? FLAG_FIRST_W : FLAG_FIRST_B)) != 0;
    sh.H = (first_turn && (d == 3 || d == 4 || d == 6)) ? 2 : 1;  // narde.py:100-103, per turn
    sh.m1 = cand_mask(sh.own, sh.opp, d, true);
    sh.deep = sh.m1 ? 1u : 0u;
  }
  // ---- (s1, s2) items: thread = first source ----------------------------------------------------------
  static NHD uint32_t second_mask(const Sh& sh, int s1) {
    Pos P1 = base_pos(sh);
    ex_move(P1, s1, s1 - sh.d);
    return cand_mask(P1.own, P1.opp, sh.d, (s1 == 23) < sh.H) & ((2u << s1) - 1u);
  }
  static NHD void ph_items_count(int tid, Sh& sh) {
    if (tid < 32) sh.part[tid] = (tid < 24 && ((sh.m1 >> tid) & 1u)) ? second_mask(sh, tid) : 0u;
  }
  static NHD void ph_items_fill(int tid, Sh& sh) {
    if (tid >= 32) return;
    const uint32_t m2 = sh.part[tid];  // 0 for tid >= 24
    uint32_t j;                        // items of the higher first sources come first: sum over the lanes above
#if defined(__CUDA_ARCH__)
    const uint32_t c = (uint32_t)__popc(m2);
    uint32_t incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_down_sync(0xFFFFFFFFu, incl, o);
      if (tid + o < 32) incl += t;
    }
    j = incl - c;
#else
    j = 0;
    for (int l = tid + 1; l < 24; l++) j += (uint32_t)popc32(sh.part[l]);
#endif
    for (uint32_t m = m2; m;) {
      int s2 = fls32(m);
      m &= ~(1u << s2);
      sh.item[j++] = (uint16_t)((tid << 5) | s2);
    }
    if (tid == 0) {
      sh.n_items = j;
      if (j) sh.deep |= 2u;
    }
  }
  // ---- the fast sub-tree below one item (no board tests), depth 3 or 4 --------------------------------
  template <class F>
  static NHD void walk_item(const Sh& sh, uint32_t it, int depth, F&& f) {
    const int d = sh.d, H = sh.H;
    const int s1 = (int)(it >> 5), s2 = (int)(it & 31u);
    Pos P2 = base_pos(sh);
    ex_move(P2, s1, s1 - d);
    ex_move(P2, s2, s2 - d);
    const int h2 = (s1 == 23) + (s2 == 23);
    const uint32_t c2 = (uint32_t)s1 | ((uint32_t)s2 << 5);
    uint32_t m3 = cand_mask(P2.own, P2.opp, d, h2 < H) & ((2u << s2) - 1u);
    while (m3) {
      const int s3 = fls32(m3);
      m3 &= ~(1u << s3);
      const uint32_t c3 = c2 | ((uint32_t)s3 << 10);
      if (depth == 3) {
        f(c3);
        continue;
      }
      Pos P3 = P2;
      ex_move(P3, s3, s3 - d);
      uint32_t m4 = cand_mask(P3.own, P3.opp, d, h2 + (s3 == 23) < H) & ((2u << s3) - 1u);
      while (m4) {
        const int s4 = fls32(m4);
        m4 &= ~(1u << s4);
        f(c3 | ((uint32_t)s4 << 15));
      }
    }
  }
  static NHD void ph_item_counts(int tid, Sh& sh) {
    uint32_t deep = 0;
    for (uint32_t t = (uint32_t)tid; t < sh.n_items; t += (uint32_t)NT) {
      const int d = sh.d, H = sh.H;
      const uint32_t it = sh.item[t];
      const int s1 = (int)(it >> 5), s2 = (int)(it & 31u);
      Pos P2 = base_pos(sh);
      ex_move(P2, s1, s1 - d);
      ex_move(P2, s2, s2 - d);
      const int h2 = (s1 == 23) + (s2 == 23);
      uint32_t m3 = cand_mask(P2.own, P2.opp, d, h2 < H) & ((2u << s2) - 1u);
      uint32_t n3 = (uint32_t)popc32(m3), n4 = 0;
      while (m3) {
        const int s3 = fls32(m3);
        m3 &= ~(1u << s3);
        Pos P3 = P2;
        ex_move(P3, s3, s3 - d);
        n4 += (uint32_t)popc32(cand_mask(P3.own, P3.opp, d, h2 + (s3 == 23) < H) & ((2u << s3) - 1u));
      }
      sh.c3[t] = (uint16_t)n3;  // <= 24
      sh.c4[t] = (uint16_t)n4;  // <= 300
      if (n3) deep |= 4u;
      if (n4) deep |= 8u;
    }
    if (deep) sm_fetch_or(&sh.deep, deep);
  }
  // ---- block exclusive scan of per-thread chunk sums: part[] -> part[] (exclusive), returns nothing -------
  static NHD void chunk_of(uint32_t n, int tid, uint32_t* t0, uint32_t* t1) {
    const uint32_t per = (n + (uint32_t)NT - 1u) / (uint32_t)NT;
    const uint32_t a = (uint32_t)tid * per, b = a + per;
    *t0 = a < n ? a : n;
    *t1 = b < n ? b : n;
  }
  // Exclusive prefix / total of part[] over the team.  On the device every thread of the team calls these
  // convergently (warp shuffles; the sums of the preceding warps are recomputed per warp, so no barrier is needed).
  static NHD uint32_t prefix_before(const Sh& sh, int tid) {  // sum of part[0 .. tid)
#if defined(__CUDA_ARCH__)
    const int lane = tid & 31, w = tid >> 5;
    const uint32_t v = sh.part[tid];
    uint32_t pre = 0;
    for (int k = 0; k < w; k++) pre += sh.part[lane + 32 * k];
    if (NT > 32) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) pre += __shfl_xor_sync(0xFFFFFFFFu, pre, o);
    }
    uint32_t incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
      if (lane >= o) incl += t;
    }
    return pre + incl - v;
#else
    uint32_t r = 0;
    for (int l = 0; l < tid; l++) r += sh.part[l];
    return r;
#endif
  }
  static NHD uint32_t part_total(const Sh& sh, int tid) {
#if defined(__CUDA_ARCH__)
    uint32_t t = 0;
    for (int k = 0; k < NT / 32; k++) t += sh.part[(tid & 31) + 32 * k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xFFFFFFFFu, t, o);
    return t;
#else
    (void)tid;
    uint32_t r = 0;
    for (int l = 0; l < NT; l++) r += sh.part[l];
    return r;
#endif
  }
  // ---- candidates per item at `depth` -> exclusive offsets --------------------------------------------
  static NHD uint32_t item_cands(const Sh& sh, uint32_t t, int depth) {
    return depth == 4 ? sh.c4[t] : depth == 3 ? sh.c3[t] : 1u;
  }
  static NHD void ph_scan_a(int tid, Sh& sh, int depth) {
    uint32_t t0, t1, s = 0;
    chunk_of(sh.n_items, tid, &t0, &t1);
    for (uint32_t t = t0; t < t1; t++) s += item_cands(sh, t, depth);
    sh.part[tid] = s;
  }
  static NHD void ph_scan_b(int tid, Sh& sh, int depth) {
    uint32_t t0, t1;
    chunk_of(sh.n_items, tid, &t0, &t1);
    uint32_t r = prefix_before(sh, tid);
    for (uint32_t t = t0; t < t1; t++) {
      sh.ioff[t] = (uint16_t)r;  // <= 17550
      r += item_cands(sh, t, depth);
    }
    if (tid == NT - 1) {
      sh.ioff[sh.n_items] = (uint16_t)r;
      sh.n_cand = r;
    }
  }
  static NHD void ph_level1(int tid, Sh& sh) {  // depth 1: the candidates are the level-1 sources
    if (tid == 0) sh.n_cand = (uint32_t)popc32(sh.m1);
  }
  // ---- write the candidates [w0, w0 + kExWindow) of `depth` into the window ---------------------------
  static NHD void ph_materialise(int tid, Sh& sh, int depth, uint32_t w0) {
    const uint32_t w1 = w0 + ex_window();
    if (depth == 1) {
      if (tid == 0) {
        uint32_t k = 0;
        for (uint32_t m = sh.m1; m; k++) {
          int s = fls32(m);
          m &= ~(1u << s);
          if (k >= w0 && k < w1) sh.cand[k - w0] = (uint32_t)s;
        }
      }
      return;
    }
    for (uint32_t t = (uint32_t)tid; t < sh.n_items; t += (uint32_t)NT) {
      const uint32_t it = sh.item[t];
      if (depth == 2) {
        if (t >= w0 && t < w1) sh.cand[t - w0] = (it >> 5) | ((it & 31u) << 5);
        continue;
      }
      uint32_t o = sh.ioff[t];
      const uint32_t o1 = sh.ioff[t + 1];
      if (o1 <= w0 || o >= w1 || o == o1) continue;
      walk_item(sh, it, depth, [&](uint32_t code) {
        if (o >= w0 && o < w1) sh.cand[o - w0] = code;
        o++;
      });
    }
  }
  // ---- is the multiset playable, and in which order?  (narde.py:64-89 along one ordering) ----------------
  // The board after a sub-multiset does not depend on the order it was played in, so the orderings of a candidate
  // live on the 2^J subsets S of its (descending) sources: ok(S) = the board exists and is legal, an edge
  // S -> S + {c} = a legal half-move of source c on board(S); the candidate is playable iff the full set can be
  // reached from the empty one through ok subsets (bounded work: no walk over the J! orderings).
  // Only the <= J source points can lose their last checker and only the <= J destinations can gain one, so a
  // subset's board is: the untouched part of the own mask, the destinations that are not source points (OR), and
  // the source points still occupied -- their checker counts sit in the four bytes of one word (biased by 32, so
  // that a missing checker shows without a borrow between bytes).  board(S) exists iff no count is negative: the
  // arrivals a departure may need come from higher sources, which a descending order plays first.
  // Whether the moves of a candidate respect the head budget does not depend on their order (the fast walk never
  // uses more head moves than allowed), and the opponent never moves: what depends on S is the block rule, the
  // checker on the source (implied by "board(S + {c}) exists") and "every checker home" for a bear-off.
  template <int J>
  struct Sub {
    uint32_t own[1 << J];       // own-occupancy mask of board(S)
    uint32_t ok;                // bit S: board(S) exists and does not violate the block rule
    uint32_t dec[J], inc[J], arrbit[J], ptbit[J];
    uint32_t rest, opp;
    NHD uint32_t mask_of(uint32_t cn, uint32_t arr) const {
      const uint32_t t = (cn + 0x5F5F5F5Fu) & 0x80808080u;  // byte >= 33: at least one checker left on that source point
      uint32_t m = rest | arr;
#pragma unroll
      for (int k = 0; k < J; k++)
        if (t & (0x80u << (8 * k))) m |= ptbit[k];
      return m;
    }
    NHD static bool exists(uint32_t cn) { return (cn & 0x20202020u) == 0x20202020u; }  // every byte >= 32: no count negative
    // node (counts cn, arrivals arr) of subset S: its child S + {C}, that child's children (indices above C), the next sibling
    template <int C, uint32_t S>
    NHD void kids(uint32_t cn, uint32_t arr) {
      if constexpr (C < J) {
        constexpr uint32_t T = S | (1u << C);
        const uint32_t cn2 = cn - dec[C] + inc[C], arr2 = arr | arrbit[C];
        const uint32_t m = mask_of(cn2, arr2);
        own[T] = m;
        if (exists(cn2) && !violates_block(m, opp)) ok |= 1u << T;
        kids<C + 1, T>(cn2, arr2);
        kids<C + 1, S>(cn, arr);
      }
    }
  };
  template <int J>
  static NHD bool playable_j(const Sh& sh, uint32_t srcp, uint32_t* orderp) {
    const int d = sh.d;
    const Pos base = base_pos(sh);
    constexpr uint32_t FULL = (1u << J) - 1u;
    Sub<J> sub;
    int src[J];
    uint32_t srcpts = 0, cn0 = 0x20202020u, dest_free = 0;
    bool bear = false;
#pragma unroll
    for (int c = 0; c < J; c++) {
      src[c] = (int)((srcp >> (5 * c)) & 31u);
      srcpts |= 1u << src[c];
    }
#pragma unroll
    for (int c = 0; c < J; c++) {
      // equal sources share the count of the first of them (sources are sorted: equal ones are neighbours)
      int slot = c;
#pragma unroll
      for (int a = c - 1; a >= 0; a--)
        if (src[a] == src[c]) slot = a;
      sub.dec[c] = 1u << (8 * slot);
      sub.ptbit[c] = slot == c ? 1u << src[c] : 0u;
      if (slot == c) cn0 += base.cnt(src[c]) << (8 * c);
      const int t = src[c] - d;
      uint32_t inc = 0;
#pragma unroll
      for (int k = J - 1; k > c; k--)  // a destination that is itself a source point: the count of its first index
        if (src[k] == t) inc = 1u << (8 * k);
      sub.inc[c] = inc;
      sub.arrbit[c] = (t >= 0 && !((srcpts >> t) & 1u)) ? 1u << t : 0u;
      if (t >= 0 ? !((base.opp >> t) & 1u) : true) dest_free |= 1u << c;  // narde.py:69-72 (a bear-off has no destination)
      if (t < 0) bear = true;
    }
    sub.rest = base.own & ~srcpts;
    sub.opp = base.opp;
    {  // highest source first: legal up to the block rule (that is how the fast walk found the candidate), the
       // representative whenever its boards are legal; the last board is the same in every order
      uint32_t cn = cn0, arr = 0, bad = 0;
#pragma unroll
      for (int t = 0; t < J; t++) {
        cn = cn - sub.dec[t] + sub.inc[t];
        arr |= sub.arrbit[t];
        if (violates_block(sub.mask_of(cn, arr), base.opp)) bad |= 1u << t;
      }
      if ((bad >> (J - 1)) & 1u) return false;
      if (bad == 0u) {
        *orderp = srcp;
        return true;
      }
    }
    if constexpr (J == 1) {
      return false;  // (unreachable: one move, its board was tested above)
    } else {
      sub.own[0] = base.own;
      sub.ok = 1u;  // the start board counts as legal (narde.py tests the boards AFTER a move)
      sub.template kids<0, 0u>(cn0, 0u);
      if (!((sub.ok >> FULL) & 1u)) return false;
      uint32_t allhome = 0xFFFFu;
      if (bear) {  // narde.py:73-77: a bear-off needs every checker home on the board it is played from
        allhome = 0;
#pragma unroll
        for (uint32_t S = 0; S <= FULL; S++)
          if ((sub.own[S] >> 6) == 0u) allhome |= 1u << S;
      }
      // legal[c]: bit S (c not in S) = the half-move of source c is legal on board(S), given that board(S + {c}) exists
      constexpr uint32_t kClear[4] = {0x5555u, 0x3333u, 0x0F0Fu, 0x00FFu};
      uint32_t legal[J];
#pragma unroll
      for (int c = 0; c < J; c++)
        legal[c] = kClear[c] & (src[c] - d >= 0 ? (((dest_free >> c) & 1u) ? 0xFFFFu : 0u) : allhome);
      // good: bit S = the turn can be completed from board(S), all subsets at once, one level per trip
      uint32_t good = 1u << FULL;
#pragma unroll
      for (int level = 0; level < J; level++) {
        uint32_t reach = 0;
#pragma unroll
        for (int c = 0; c < J; c++) reach |= legal[c] & (good >> (1u << c));
        good |= sub.ok & reach;
      }
      if (!(good & 1u)) return false;
      // the lexicographically first legal ordering, higher sources first (equal sources are the same move)
      uint32_t S = 0, o = 0;
#pragma unroll
      for (int step = 0; step < J; step++) {
        bool placed = false;
#pragma unroll
        for (int c = 0; c < J; c++) {
          if (!placed && !((S >> c) & 1u) && ((legal[c] >> S) & 1u) && ((good >> (S | (1u << c))) & 1u)) {
            o |= (uint32_t)src[c] << (5 * step);
            S |= 1u << c;
            placed = true;
          }
        }
      }
      *orderp = o;
      return true;
    }
  }
  static NHD_NOINLINE bool playable(const Sh& sh, uint32_t srcp, int j, uint32_t* orderp) {
    switch (j) {
      case 1: return playable_j<1>(sh, srcp, orderp);
      case 2: return playable_j<2>(sh, srcp, orderp);
      case 3: return playable_j<3>(sh, srcp, orderp);
      default: return playable_j<4>(sh, srcp, orderp);
    }
  }
  // one round: candidate c0 + tid of the window is tested; the result goes to the team's scratch
  static NHD void ph_test(int tid, Sh& sh, int depth, uint32_t c, uint32_t n_win) {
    uint32_t r = 0, o;
    if (c < n_win && playable(sh, sh.cand[c], depth, &o)) r = kPlayable | o;
    sh.part[tid] = r;
  }
  // ... and its survivors are ranked (survivors before this round = `before`).  mode 0: the first `cap` actions are
  // stored; a level that fits one window keeps its survivors compacted at the front of the window (a survivor's
  // rank never exceeds its own index, and every candidate at or below that index has been read), so the chosen one
  // is there when the count is known.  mode 1: capture the survivor of rank sh.idx (second pass over a multi-window level).
  static NHD void ph_rank_a(int tid, Sh& sh) {  // teams of several warps: survivors per warp
#if defined(__CUDA_ARCH__)
    const uint32_t b = __ballot_sync(0xFFFFFFFFu, (sh.part[tid] >> 31) != 0u);
    if ((tid & 31) == 0) sh.wsum[tid >> 5] = (uint32_t)__popc(b);
#else
    (void)tid;
    (void)sh;
#endif
  }
  static NHD void ph_rank(int tid, Sh& sh, int depth, uint32_t before, bool keep, int mode, int64_t i, const StepFullArgs& A) {
    const uint32_t mine = sh.part[tid];
    uint32_t below, total;
#if defined(__CUDA_ARCH__)
    const uint32_t b = __ballot_sync(0xFFFFFFFFu, (mine >> 31) != 0u);
    below = (uint32_t)__popc(b & ((1u << (tid & 31)) - 1u));
    total = (uint32_t)__popc(b);
    if (NT > 32) {
      total = 0;
      for (int w = 0; w < NT / 32; w++) {
        const uint32_t t = sh.wsum[w];
        if (w < (tid >> 5)) below += t;
        total += t;
      }
    }
#else
    below = total = 0;
    for (int l = 0; l < NT; l++) {
      const uint32_t v = sh.part[l] >> 31;
      if (l < tid) below += v;
      total += v;
    }
#endif
    if (mine >> 31) {
      const uint32_t r = before + below, o = mine & ~kPlayable;
      if (mode == 0) {
        if (A.actions && r < (uint32_t)A.cap) A.actions[i * (int64_t)A.cap + r] = action_of(o, depth, sh.d);
        if (keep) sh.cand[r] = o;
      } else if (r == sh.idx) {
        sh.chosen = action_of(o, depth, sh.d);
        sh.found = 1;
      }
    }
    if (tid == 0) sh.run = before + total;
  }
  // the level is complete with n playable multisets: the action to play
  static NHD void ph_pick(int tid, Sh& sh, int depth, uint32_t n, bool kept, int64_t i, const StepFullArgs& A) {
    if (tid != 0) return;
    sh.count = n;
    sh.idx = pick_action_index(A, i, sh.rnd, n);
    if (n == 0) return;
    if (kept) {
      sh.chosen = action_of(sh.cand[sh.idx], depth, sh.d);
      sh.found = 1;
    } else if (A.actions && sh.idx < (uint32_t)A.cap) {
      // stored by ph_rank (the team has synchronised since)
      sh.chosen = *reinterpret_cast<volatile const uint64_t*>(A.actions + i * (int64_t)A.cap + sh.idx);
      sh.found = 1;
    }
  }

  // ---- the whole turn of one env; `ex.run(f)` = f(tid) on the NT threads, then a barrier -----------------
  template <class Exec>
  static NHD void solve(Exec& ex, Sh& sh, const State& s_in, int64_t i, const StepFullArgs& A) {
    ex.run([&](int tid) { ph_init(tid, sh, s_in, i, A); });
    ex.run([&](int tid) { ph_init2(tid, sh); });
    ex.mark(1);
    if (sh.m1) {
      ex.run([&](int tid) { ph_items_count(tid, sh); });
      ex.run([&](int tid) { ph_items_fill(tid, sh); });
      ex.mark(2);
      if (sh.n_items) ex.run([&](int tid) { ph_item_counts(tid, sh); });
    }
    ex.mark(3);
    int depth = sh.deep & 8u ? 4 : sh.deep & 4u ? 3 : sh.deep & 2u ? 2 : sh.deep & 1u ? 1 : 0;
    for (; depth > 0; depth--) {  // max-dice rule: the deepest level with a playable multiset
      if (depth >= 2) {
        ex.run([&](int tid) { ph_scan_a(tid, sh, depth); });
        ex.run([&](int tid) { ph_scan_b(tid, sh, depth); });
      } else {
        ex.run([&](int tid) { ph_level1(tid, sh); });
      }
      ex.mark(4);
      const uint32_t n_cand = sh.n_cand;
      const bool single = n_cand <= ex_window();
      uint32_t survivors = 0;
      for (int mode = 0; mode < 2; mode++) {
        uint32_t before = 0;
        bool stop = false;
        for (uint32_t w0 = 0; w0 < n_cand && !stop; w0 += ex_window()) {
          const uint32_t n_win = n_cand - w0 < ex_window() ? n_cand - w0 : ex_window();
          ex.run([&](int tid) { ph_materialise(tid, sh, depth, w0); });
          ex.mark(5);
          for (uint32_t c0 = 0; c0 < n_win && !stop; c0 += (uint32_t)NT) {
            ex.run([&](int tid) { ph_test(tid, sh, depth, c0 + (uint32_t)tid, n_win); });
            if (NT > 32) ex.run([&](int tid) { ph_rank_a(tid, sh); });
            ex.run([&](int tid) { ph_rank(tid, sh, depth, before, single, mode, i, A); });
            before = sh.run;
            stop = mode == 1 && sh.found != 0u;
          }
          ex.mark(6);
        }
        if (mode == 1) break;
        survivors = before;
        if (survivors == 0u) break;
        ex.run([&](int tid) { ph_pick(tid, sh, depth, survivors, single, i, A); });
        ex.mark(7);
        if (sh.found) break;  // else: the chosen action lies beyond the stored capacity -> find it (mode 1)
      }
      if (survivors) break;
    }
  }
  // ---- after solve, one thread: the chosen action played on st (a copy of sh.st), then the turn's completion ---------
  static NHD void complete(const Sh& sh, State& st, int64_t i, const StepFullArgs& A, StepFullLocal& L) {
    if (sh.count && !(A.flags & F_ENUMERATE_ONLY)) {  // apply_action, rolled up (code size)
#pragma unroll 1
      for (int k = 0; k < 4; k++) {
        const uint32_t h = (uint32_t)(sh.chosen >> (16 * k)) & 0xFFFFu;
        if (h == 0xFFFFu) break;
        apply_half_move(st, sh.player, (int)(h & 0xFF), (h >> 8) == 255u ? -1 : (int)(h >> 8));
      }
    }
    complete_env(st, i, A, sh.player, sh.count, sh.chosen, sh.d1, sh.d2, L, false);
    L.clamped = A.action_idx ? index_was_clamped(A, (uint32_t)A.action_idx[i], sh.count) : 0;
  }
};

}  // namespace narde
