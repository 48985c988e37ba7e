// narde_core.cuh -- per-environment rules arithmetic of the B200 Narde path.
//
// Everything here is integer bit arithmetic on ONE environment held in registers; the kernels in
// narde_kernels.cu run it thread-per-environment.  The functions are __host__ __device__ so that
// the identical source can be compiled by g++ into the host simulation harness under
// tests/hostsim/ (test-only) and checked against the oracle without a GPU.
//
// What it reproduces (reference = /root/reference, cited file:line):
//   * mover-perspective view            gym_narde/envs/narde.py:16-17,31-34
//   * single half-move candidates       gym_narde/envs/narde.py:64-77
//   * 6-prime "block" filter            gym_narde/envs/narde.py:78-89,139-184
//   * list-level head filter            gym_narde/envs/narde.py:94-106,127-137
//   * move application                  gym_narde/envs/narde.py:36-56,108-125
//   * env step / termination / reward   gym_narde/envs/narde_env.py:27-103,134-141
//   * README contract (Tier N): full-turn enumeration with max-dice / higher-die / per-turn head
//     rule (README.md:30, narde.py:4-6), Box(198) observation (README.md:44-102), +1/0 WHITE
//     reward (README.md:107-108)
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define NHD __host__ __device__ __forceinline__
#define NHD_NOINLINE __host__ __device__ __noinline__
#else
#define NHD inline
#define NHD_NOINLINE inline
#endif

namespace narde {

// Host-only work counters for design studies (tests/hostsim with -DNARDE_PROFILE); no-ops otherwise.
#if defined(NARDE_PROFILE) && !defined(__CUDA_ARCH__)
struct ProfCounters {
  long long nd_env, nd_rows, nd_pairs, nd_block_env, dbl_env, dbl_nodes[4], dbl_block_env, dbl_order_search, dbl_second_pass;
};
extern ProfCounters g_prof;
#define NPROF(x) (g_prof.x)
#else
#define NPROF(x) ((void)0)
#endif

// ------------------------------------------------------------------------------------------
// bit helpers
// ------------------------------------------------------------------------------------------
NHD int popc32(uint32_t x) {
#if defined(__CUDA_ARCH__)
  return __popc(x);
#else
  return __builtin_popcount(x);
#endif
}
NHD int ctz32(uint32_t x) {  // x != 0
#if defined(__CUDA_ARCH__)
  return __ffs((int)x) - 1;
#else
  return __builtin_ctz(x);
#endif
}
NHD int fls32(uint32_t x) {  // index of highest set bit, x != 0
#if defined(__CUDA_ARCH__)
  return 31 - __clz((int)x);
#else
  return 31 - __builtin_clz(x);
#endif
}
NHD uint32_t mulhi32(uint32_t a, uint32_t b) {
#if defined(__CUDA_ARCH__)
  return __umulhi(a, b);
#else
  return (uint32_t)(((uint64_t)a * b) >> 32);
#endif
}

// ------------------------------------------------------------------------------------------
// HBM state record: two 16-byte lanes per environment (SoA planes lo[N], hi[N]).
//   lo : int8 points 0..15                    (absolute / White frame, +white -black)
//   hi : int8 points 16..23 | off_w | off_b | turn(+1/-1) | flags | u16 episode_steps | u16 rsvd
// ------------------------------------------------------------------------------------------
enum : uint32_t {
  FLAG_FIRST_W = 1u,   // narde.py:28
  FLAG_FIRST_B = 2u,   // narde.py:29
  FLAG_DONE = 4u,      // episode terminated (sticky until reset)
};

struct State {
  uint32_t w[6];  // 24 signed bytes
  uint32_t meta;  // off_w | off_b<<8 | turn<<16 | flags<<24
  uint32_t aux;   // episode_steps (u16) | reserved<<16

  NHD int off_w() const { return (int)(meta & 0xFF); }
  NHD int off_b() const { return (int)((meta >> 8) & 0xFF); }
  NHD int turn() const { return (int)(int8_t)((meta >> 16) & 0xFF); }
  NHD uint32_t flags() const { return meta >> 24; }
  NHD uint32_t steps() const { return aux & 0xFFFF; }
  NHD void set_meta(int ow, int ob, int turn, uint32_t flags) {
    meta = (uint32_t)ow | ((uint32_t)ob << 8) | (((uint32_t)turn & 0xFF) << 16) | (flags << 24);
  }
  NHD void set_steps(uint32_t s) { aux = (aux & 0xFFFF0000u) | (s & 0xFFFF); }
  NHD int point(int i) const { return (int)(int8_t)((w[i >> 2] >> ((i & 3) * 8)) & 0xFF); }
};

NHD State initial_state(int turn) {  // narde.py:21-29
  State s;
  s.w[0] = s.w[1] = s.w[3] = s.w[4] = 0;
  s.w[2] = 0xF1000000u;  // point 11 = -15
  s.w[5] = 0x0F000000u;  // point 23 = +15
  s.set_meta(0, 0, turn, FLAG_FIRST_W | FLAG_FIRST_B);
  s.aux = 0;
  return s;
}

// per-byte add without carries between bytes
NHD uint32_t vadd4(uint32_t a, uint32_t b) {
#if defined(__CUDA_ARCH__)
  return __vadd4(a, b);
#else
  return ((a & 0x7F7F7F7Fu) + (b & 0x7F7F7F7Fu)) ^ ((a ^ b) & 0x80808080u);
#endif
}

// add delta (+1/-1) to absolute point idx of the byte board
NHD void state_add(State& s, int idx, int delta) {
  uint32_t d = ((uint32_t)delta & 0xFFu) << ((idx & 3) * 8);
  int wi = idx >> 2;
#pragma unroll
  for (int k = 0; k < 6; k++) s.w[k] = vadd4(s.w[k], k == wi ? d : 0u);
}

// ------------------------------------------------------------------------------------------
// Mover-frame working position: own counts nibble-packed (24 x 4 bit), occupancy masks.
// Mover frame = narde.py:60 (White: board as is; Black: rotate_board, narde.py:16-17), i.e. the
// mover's checkers are positive, its head is index 23, it moves towards index 0.
// ------------------------------------------------------------------------------------------
struct Pos {
  uint64_t lo;   // own counts, points 0..15
  uint32_t hi;   // own counts, points 16..23
  uint32_t own;  // bit p: mover has >= 1 checker on p
  uint32_t opp;  // bit p: opponent has >= 1 checker on p

  NHD uint32_t cnt(int p) const {
    return p < 16 ? (uint32_t)(lo >> (4 * p)) & 15u : (hi >> (4 * (p - 16))) & 15u;
  }
  NHD void dec(int p) {
    if (p < 16)
      lo -= 1ull << (4 * p);
    else
      hi -= 1u << (4 * (p - 16));
  }
  NHD void inc(int p) {
    if (p < 16)
      lo += 1ull << (4 * p);
    else
      hi += 1u << (4 * (p - 16));
  }
  // one half-move s -> t (t < 0: bear off); narde.py:108-125 in the mover frame
  NHD void move(int s, int t) {
    if (cnt(s) == 1) own &= ~(1u << s);
    dec(s);
    if (t >= 0) {
      inc(t);
      own |= 1u << t;
    }
  }
  NHD bool all_home() const { return (own >> 6) == 0; }  // narde.py:75
};

NHD uint32_t nib16(uint32_t x) {  // 4 bytes (each <= 15) -> 4 nibbles
  uint32_t c = (x & 0x000F000Fu) | ((x >> 4) & 0x00F000F0u);
  return (c & 0xFFu) | ((c >> 8) & 0xFF00u);
}
NHD uint32_t msb4(uint32_t m) {  // bits 7,15,23,31 -> bits 0..3
  return (((m >> 7) & 0x01010101u) * 0x01020408u) >> 24 & 0xFu;
}

// Decode the byte board into the mover frame of `player` (+1 / -1).
// *ones (optional) receives the mask of points holding exactly one mover checker.
NHD Pos decode_pos(const State& s, int player, uint32_t* ones = nullptr) {
  uint32_t own16[6], ownb[6], oppb[6], oneb[6];
#pragma unroll
  for (int k = 0; k < 6; k++) {
    uint32_t w = s.w[k];
    uint32_t neg = w & 0x80808080u;
    uint32_t negmask = (neg >> 7) * 0xFFu;
    uint32_t posb = w & ~negmask;                                      // max(v, 0)
    uint32_t negb = ((~w) & negmask) + (0x01010101u & negmask);        // max(-v, 0)
    uint32_t mine = player == 1 ? posb : negb;
    uint32_t theirs = player == 1 ? negb : posb;
    own16[k] = nib16(mine);
    ownb[k] = msb4((mine + 0x7F7F7F7Fu) & 0x80808080u);
    oppb[k] = msb4((theirs + 0x7F7F7F7Fu) & 0x80808080u);
    oneb[k] = msb4(~((mine ^ 0x01010101u) + 0x7F7F7F7Fu) & 0x80808080u);  // byte == 1
  }
  if (ones) {
    uint32_t o = oneb[0] | (oneb[1] << 4) | (oneb[2] << 8) | (oneb[3] << 12) | (oneb[4] << 16) | (oneb[5] << 20);
    *ones = player == 1 ? o : (((o >> 12) | (o << 12)) & 0xFFFFFFu);
  }
  // rotation by 12 points = 3 words (narde.py:16-17)
  Pos p;
  if (player == 1) {
    p.lo = (uint64_t)own16[0] | ((uint64_t)own16[1] << 16) | ((uint64_t)own16[2] << 32) |
           ((uint64_t)own16[3] << 48);
    p.hi = own16[4] | (own16[5] << 16);
    p.own = ownb[0] | (ownb[1] << 4) | (ownb[2] << 8) | (ownb[3] << 12) | (ownb[4] << 16) | (ownb[5] << 20);
    p.opp = oppb[0] | (oppb[1] << 4) | (oppb[2] << 8) | (oppb[3] << 12) | (oppb[4] << 16) | (oppb[5] << 20);
  } else {
    p.lo = (uint64_t)own16[3] | ((uint64_t)own16[4] << 16) | ((uint64_t)own16[5] << 32) |
           ((uint64_t)own16[0] << 48);
    p.hi = own16[1] | (own16[2] << 16);
    p.own = ownb[3] | (ownb[4] << 4) | (ownb[5] << 8) | (ownb[0] << 12) | (ownb[1] << 16) | (ownb[2] << 20);
    p.opp = oppb[3] | (oppb[4] << 4) | (oppb[5] << 8) | (oppb[0] << 12) | (oppb[1] << 16) | (oppb[2] << 20);
  }
  return p;
}

// ------------------------------------------------------------------------------------------
// Half-move legality
// ------------------------------------------------------------------------------------------
// narde.py:139-184 on an own-occupancy mask: a run of >= 6 consecutive own points with no
// opponent checker at any index below the run's first point.  The lowest long run has the
// fewest opponents below it, so only that one needs testing.
NHD bool violates_block(uint32_t a, uint32_t opp) {
  uint32_t t2 = a & (a >> 1);
  uint32_t t4 = t2 & (t2 >> 2);
  uint32_t w = t4 & (t2 >> 4);  // bit i: points i..i+5 all own
  if (!w) return false;
  uint32_t below = (w & (0u - w)) - 1u;
  return (opp & below) == 0u;
}

// narde.py:64-77: sources that may move `d` pips (bit mask), before the block filter.
NHD uint32_t cand_mask(uint32_t own, uint32_t opp, int d, bool head_ok) {
  uint32_t low = (1u << d) - 1u;
  uint32_t m = own & ~(opp << d) & ~low;  // lands on own/empty point (narde.py:69-72)
  if ((own >> 6) == 0u) m |= own & low;   // bear off: all home and die >= pos+1 (narde.py:73-77)
  if (!head_ok) m &= ~(1u << 23);
  return m;
}

NHD uint32_t after_mask(const Pos& P, int s, int t) {
  uint32_t a = P.cnt(s) == 1 ? P.own & ~(1u << s) : P.own;
  if (t >= 0) a |= 1u << t;
  return a;
}

// narde.py:78-89: drop candidates whose after-board violates the block rule
NHD uint32_t block_filter_each(const Pos& P, uint32_t m, int d) {
  uint32_t out = 0;
  for (uint32_t mm = m; mm; mm &= mm - 1) {
    int s = ctz32(mm);
    if (!violates_block(after_mask(P, s, s - d), P.opp)) out |= 1u << s;
  }
  return out;
}

// Empty points t for which own | {t} contains a violating 6-run (bit-parallel run arithmetic).
// A run violates iff it lies entirely below the opponent's lowest checker, so only that part of
// the board is looked at.  Only meaningful when `own` itself does not violate.
NHD uint32_t completing_points(uint32_t own, uint32_t opp) {
  uint32_t below = opp ? ((opp & (0u - opp)) - 1u) : 0xFFFFFFu;
  uint32_t a = own & below;
  uint32_t s1 = a, s2 = s1 & (a >> 1), s3 = s2 & (a >> 2), s4 = s3 & (a >> 3), s5 = s4 & (a >> 4);
  // e_j: bit i set when points i-j+1..i are all own  (runs of length j ENDING at i)
  uint32_t e1 = s1, e2 = s2 << 1, e3 = s3 << 2, e4 = s4 << 3, e5 = s5 << 4;
  // t completes a run of >= 6 when (run ending at t-1) + 1 + (run starting at t+1) >= 6
  uint32_t t = (s5 >> 1) | ((e1 << 1) & (s4 >> 1)) | ((e2 << 1) & (s3 >> 1)) | ((e3 << 1) & (s2 >> 1)) |
               ((e4 << 1) & (s1 >> 1)) | (e5 << 1);
  return t & ~own & below;
}

// narde.py:78-89 with the per-candidate board test only where it can fail: when the board is legal
// now, a move can only create a violation by landing on a completing point.
NHD uint32_t block_filter(const Pos& P, uint32_t m, int d) {
  if (violates_block(P.own, P.opp)) return block_filter_each(P, m, d);
  uint32_t risky = m & (completing_points(P.own, P.opp) << d);
  return risky ? ((m & ~risky) | block_filter_each(P, risky, d)) : m;
}

// True when no board reachable from P within this turn can contain a violating 6-run: the run
// would have to lie entirely below the opponent's lowest checker, inside the union of points the
// mover could occupy.  (Conservative pre-check; when it holds the block filter is skipped.)
NHD bool block_rule_irrelevant(const Pos& P, int d1, int d2) {
  uint32_t u = P.own;
  if (d1 == d2) {
    u |= u >> d1;
    u |= u >> (2 * d1);
    u |= P.own >> (4 * d1);
  } else {
    u |= (P.own >> d1) | (P.own >> d2) | (P.own >> (d1 + d2));
  }
  uint32_t below_opp = P.opp ? ((P.opp & (0u - P.opp)) - 1u) : 0xFFFFFFu;
  u &= below_opp;
  uint32_t t2 = u & (u >> 1);
  uint32_t t4 = t2 & (t2 >> 2);
  uint32_t w6 = t4 & (t2 >> 4);  // bit i: the 6-window starting at i could become all-own
  if (w6 == 0u) return true;
  // refinement: a turn adds at most `moves` newly occupied points (2 dice, or 4 for doubles), so a
  // window needing more new points than that can never fill up
  int moves = d1 == d2 ? 4 : 2;
  for (; w6; w6 &= w6 - 1) {
    int i = ctz32(w6);
    if (popc32((0x3Fu << i) & ~P.own) <= moves) return false;
  }
  return true;
}

// ------------------------------------------------------------------------------------------
// Tier R1: the reference's ordered half-move list (narde.py:58-92 + head filter :94-137)
// emit(from, to) is called in list order; to == 255 means 'off'.  Returns the list length.
// ------------------------------------------------------------------------------------------
struct HalfList {        // compact form of the list for a <= 2-dice roll
  uint32_t mask[2];      // per sorted die (descending): sources kept after all filters
  int die[2];
  int n;                 // list length including duplicates
};

template <class Emit>
NHD int half_moves_list(const Pos& P, const uint8_t* roll, int nroll, bool first_turn, Emit&& emit) {
  int r[4] = {0, 0, 0, 0};
  for (int i = 0; i < nroll; i++) r[i] = roll[i];
  // sorted(roll, reverse=True)  narde.py:59
  for (int i = 0; i < nroll; i++)
    for (int j = i + 1; j < nroll; j++)
      if (r[j] > r[i]) {
        int t = r[i];
        r[i] = r[j];
        r[j] = t;
      }
  int max_head = 1;  // narde.py:100-103: only a 2-element roll can equal [3,3]/[4,4]/[6,6]
  if (first_turn && nroll == 2 && r[0] == r[1] && (r[0] == 3 || r[0] == 4 || r[0] == 6)) max_head = 2;
  int n = 0, head = 0;
  for (int i = 0; i < nroll; i++) {
    int d = r[i];
    if (d < 1 || d > 6) continue;
    uint32_t m = block_filter(P, cand_mask(P.own, P.opp, d, true), d);
    for (; m; m &= m - 1) {  // pos ascending (narde.py:65)
      int s = ctz32(m);
      if (s == 23) {  // narde.py:131-134
        if (head >= max_head) continue;
        head++;
      }
      emit(s, s - d >= 0 ? s - d : 255);
      n++;
    }
  }
  return n;
}

// Compact two-dice list used by the step kernel (needs only length, first entry and membership).
NHD HalfList half_list2(const Pos& P, int d1, int d2, bool first_turn) {
  HalfList L;
  int hi = d1 > d2 ? d1 : d2, lo = d1 > d2 ? d2 : d1;
  L.die[0] = hi;
  L.die[1] = lo;
  int max_head = (first_turn && hi == lo && (hi == 3 || hi == 4 || hi == 6)) ? 2 : 1;
  L.mask[0] = block_filter(P, cand_mask(P.own, P.opp, hi, true), hi);
  L.mask[1] = hi == lo ? L.mask[0] : block_filter(P, cand_mask(P.own, P.opp, lo, true), lo);
  int head = (int)(L.mask[0] >> 23) & 1;
  if (head >= max_head) L.mask[1] &= ~(1u << 23);
  L.n = popc32(L.mask[0]) + popc32(L.mask[1]);
  return L;
}
NHD HalfList half_list1(const Pos& P, int d) {
  HalfList L;
  L.die[0] = d;
  L.die[1] = 0;
  L.mask[0] = block_filter(P, cand_mask(P.own, P.opp, d, true), d);
  L.mask[1] = 0;
  L.n = popc32(L.mask[0]);
  return L;
}
// is (from, to) in the list?  to == -1 means 'off'
NHD bool half_list_has(const HalfList& L, int from, int to) {
  if (from < 0 || from > 23) return false;
#pragma unroll
  for (int k = 0; k < 2; k++) {
    if ((L.mask[k] >> from) & 1u) {
      int t = from - L.die[k];
      if (t < 0 ? to == -1 : to == t) return true;
    }
  }
  return false;
}

// Apply one mover-frame half-move to the byte board (narde.py:36-56,108-125).
NHD void apply_half_move(State& s, int player, int from, int to /* -1 = off */) {
  int rot = player == 1 ? 0 : 12;
  int af = from + rot;
  if (af >= 24) af -= 24;
  state_add(s, af, -player);
  int ow = s.off_w(), ob = s.off_b();
  uint32_t fl = s.flags();
  if (to < 0) {
    if (player == 1)
      ow++;
    else
      ob++;
  } else {
    int at = to + rot;
    if (at >= 24) at -= 24;
    state_add(s, at, player);
  }
  fl &= ~(player == 1 ? FLAG_FIRST_W : FLAG_FIRST_B);  // narde.py:52-56
  s.set_meta(ow, ob, s.turn(), fl);
}

// narde_env.py:134-141
NHD bool game_ended(const State& s, int player, int* reward12) {
  int mine = player == 1 ? s.off_w() : s.off_b();
  int theirs = player == 1 ? s.off_b() : s.off_w();
  if (mine == 15) {
    *reward12 = theirs > 0 ? 1 : 2;
    return true;
  }
  *reward12 = 0;
  return false;
}

// narde_env.py:24-25 / narde.py:31-34 as 24 int32
NHD void obs24(const State& s, int player, int32_t* out) {
  for (int i = 0; i < 24; i++) {
    if (player == 1)
      out[i] = s.point(i);
    else
      out[i] = -s.point(i < 12 ? i + 12 : i - 12);
  }
}

// Tier R2: NardeEnv.step (narde_env.py:27-103) on one environment.  Codes outside [0,576) are
// treated as "not a legal move" (the reference's Discrete(576) never produces them).
NHD void step_reference(State& s, int d1, int d2, int code1, int code2, int* reward, int* done) {
  int player = s.turn();
  bool first_turn = (s.flags() & (player == 1 ? FLAG_FIRST_W : FLAG_FIRST_B)) != 0;
  Pos P = decode_pos(s, player);
  HalfList L = half_list2(P, d1, d2, first_turn);  // narde_env.py:31
  if (L.n == 1) {                                  // narde_env.py:41-43
    int k = L.mask[0] ? 0 : 1;
    int from = ctz32(L.mask[k]);
    int to = from - L.die[k];
    apply_half_move(s, player, from, to < 0 ? -1 : to);
  } else if (L.n >= 2) {  // narde_env.py:44-93
    bool ok1 = code1 >= 0 && code1 < 576, ok2 = code2 >= 0 && code2 < 576;
    int from1 = ok1 ? code1 / 24 : -1, to1 = ok1 ? code1 % 24 : 0;
    if (to1 == 0 && from1 >= 0 && from1 <= 5) to1 = -1;  // narde_env.py:50
    int from2 = ok2 ? code2 / 24 : -1, to2 = ok2 ? code2 % 24 : 0;
    if (to2 == 0 && from2 >= 0 && from2 <= 5) to2 = -1;  // narde_env.py:59
    if (ok1 && half_list_has(L, from1, to1)) {           // narde_env.py:63
      apply_half_move(s, player, from1, to1);
      int dist = to1 < 0 ? from1 + 1 : (from1 > to1 ? from1 - to1 : to1 - from1);  // :69-74
      // temp_dice.remove(dist) if present else pop(0)   narde_env.py:77-83 (dice UNSORTED)
      int rem = (d1 == dist) ? d2 : ((d2 == dist) ? d1 : d2);
      Pos P2 = decode_pos(s, player);
      HalfList L2 = half_list1(P2, rem);                 // narde_env.py:87
      if (ok2 && half_list_has(L2, from2, to2)) apply_half_move(s, player, from2, to2);
    }
  }
  int rew = 0;
  bool dn = game_ended(s, player, &rew);  // narde_env.py:96
  uint32_t fl = s.flags();
  if (dn) fl |= FLAG_DONE;
  s.set_meta(s.off_w(), s.off_b(), dn ? player : -player, fl);  // narde_env.py:99-100
  s.set_steps(s.steps() + 1);
  *reward = rew;
  *done = dn ? 1 : 0;
}

// ------------------------------------------------------------------------------------------
// Tier N1: full-turn enumeration.  A turn action is 4 half-moves packed in 64 bits:
//   slot k (bits 16k..16k+15) = from | to << 8, to == 255: bear off, slot == 0xFFFF: unused.
// Canonical order and representative sequence are specified in DESIGN.md ("canonical action
// order"); the oracle computes the same thing by brute force (oracle/narde_oracle.c).
// ------------------------------------------------------------------------------------------
NHD uint64_t pack_half(int from, int to) { return (uint64_t)((from & 0xFF) | ((to < 0 ? 255 : to) << 8)); }
static const uint64_t ACT_EMPTY = 0xFFFFFFFFFFFFFFFFull;
NHD uint64_t act_set(uint64_t act, int slot, int from, int to) {
  uint64_t m = 0xFFFFull << (16 * slot);
  return (act & ~m) | (pack_half(from, to) << (16 * slot));
}

// ---- non-doubles (a > b) ----------------------------------------------------------------
// A 2-move turn is a pair (p, q): p = source moved with the higher die a, q = source moved with
// the lower die b.  Distinct pairs give distinct afterstates except
//   (x-b, x) == (x, x-a)      the same checker (or an equivalent one) travelling a+b pips,
//   (p, q)   == (q, p)        when p, q < b: both checkers borne off by either die.
// Pairs are visited by ascending key (23-p)*32 + (23-q); a pair is emitted unless its
// smaller-key twin was present.
template <class Sink>
NHD int enum_nondouble(const Pos& P, int a, int b, bool blockchk, Sink& sink) {
  uint32_t Ca = cand_mask(P.own, P.opp, a, true);
  uint32_t S = cand_mask(P.own, P.opp, b, true);
  if (blockchk) {
    Ca = block_filter(P, Ca, a);
    S = block_filter(P, S, b);
  }
  // q in S after which every mover checker is home (enables a bear-off with the higher die)
  uint32_t q_home = 0;
  uint32_t outside = P.own & ~0x3Fu;
  if (outside == 0u) {
    q_home = S;
  } else if ((outside & (outside - 1u)) == 0u) {
    int qo = ctz32(outside);
    if (P.cnt(qo) == 1 && qo - b < 6) q_home = S & outside;
  }
  int n = 0;
  uint32_t chain_present = 0;  // bit x: pair (x, x-a) was present
  uint64_t bo_present = 0;     // bit 6p+q: pair (p, q) with p, q < 6 was present
  uint32_t rows = (P.own | (S >> b)) & 0xFFFFFFu;
  NPROF(nd_env++);
  if (blockchk) NPROF(nd_block_env++);
  while (rows) {
    NPROF(nd_rows++);
    int p = fls32(rows);
    rows &= ~(1u << p);
    int ta = p - a;
    // a-first: p moves a, then q moves b on the resulting board
    uint32_t m1 = 0;
    Pos P1 = P;
    if ((Ca >> p) & 1u) {
      P1.move(p, ta);
      m1 = cand_mask(P1.own, P1.opp, b, p != 23);
      if (blockchk) m1 = block_filter(P1, m1, b);
    }
    // b-first: q in S such that p can then move a
    uint32_t m2;
    if ((P.own >> p) & 1u) {
      m2 = S;
      if (P.cnt(p) == 1) m2 &= ~(1u << p);
    } else {
      m2 = p + b < 24 ? (S & (1u << (p + b))) : 0u;
    }
    if (ta >= 0) {
      if ((P.opp >> ta) & 1u) m2 = 0;
    } else {
      m2 &= q_home;
    }
    if (p == 23) m2 &= ~(1u << 23);
    if (blockchk) {
      uint32_t keep = 0;
      for (uint32_t mm = m2 & ~m1; mm; mm &= mm - 1) {
        int q = ctz32(mm);
        Pos Q = P;
        Q.move(q, q - b);
        if (!violates_block(after_mask(Q, p, ta), Q.opp)) keep |= 1u << q;
      }
      m2 = keep | (m2 & m1);
    }
    uint32_t pres = m1 | m2;
    while (pres) {
      NPROF(nd_pairs++);
      int q = fls32(pres);
      pres &= ~(1u << q);
      bool dup = false;
      if (q == p + b && ((chain_present >> q) & 1u)) dup = true;
      if (p < b && q < b && p < q && ((bo_present >> (6 * q + p)) & 1ull)) dup = true;
      if (q == ta) chain_present |= 1u << p;
      if (p < 6 && q < 6) bo_present |= 1ull << (6 * p + q);
      if (dup) continue;
      uint64_t act = ACT_EMPTY;
      if ((m1 >> q) & 1u) {
        act = act_set(act, 0, p, ta);
        act = act_set(act, 1, q, q - b);
      } else {
        act = act_set(act, 0, q, q - b);
        act = act_set(act, 1, p, ta);
      }
      sink(act);
      n++;
    }
  }
  if (n) return n;
  // maximal length 1: the higher die if it can be played (narde.py:6 rule 4), else the lower
  uint32_t m = Ca ? Ca : S;
  int d = Ca ? a : b;
  while (m) {
    int s = fls32(m);
    m &= ~(1u << s);
    sink(act_set(ACT_EMPTY, 0, s, s - d));
    n++;
  }
  return n;
}

// ---- doubles ----------------------------------------------------------------------------
// With one die value a turn is a multiset of sources; the afterstate depends only on the
// multiset.  Multisets are visited in descending-source DFS order (= ascending canonical key).
// Playing a multiset highest source first is legal whenever any order is, EXCEPT for the block
// rule (an intermediate 6-run can depend on the order); when the block rule can matter
// (blockchk) every multiset whose descending order fails is re-tested over all its orderings.

// Exhaustive ordering search (rare path).  src[0..k) sorted descending.  Finds the
// lexicographically first legal ordering (trying higher sources first); writes it to order[].
NHD bool dbl_order_search(const Pos& base, const int* src, int k, int d, int H, int* order) {
  NPROF(dbl_order_search++);
  // iterative DFS over permutations, depth <= 4
  Pos st[5];
  int head[5];
  int choice[4];   // index into src chosen at each depth
  uint32_t used = 0;
  st[0] = base;
  head[0] = 0;
  int depth = 0;
  choice[0] = -1;
  for (;;) {
    // advance choice at this depth
    int c = choice[depth] + 1;
    bool placed = false;
    for (; c < k; c++) {
      if ((used >> c) & 1u) continue;
      // skip equal sources already tried at this depth (same move)
      bool same = false;
      for (int e = 0; e < c; e++)
        if (!((used >> e) & 1u) && src[e] == src[c]) same = true;
      if (same) continue;
      int s = src[c];
      const Pos& cur = st[depth];
      uint32_t m = cand_mask(cur.own, cur.opp, d, head[depth] < H);
      if (!((m >> s) & 1u)) continue;
      Pos nx = cur;
      nx.move(s, s - d);
      if (violates_block(nx.own, nx.opp)) continue;
      st[depth + 1] = nx;
      head[depth + 1] = head[depth] + (s == 23);
      placed = true;
      break;
    }
    if (placed) {
      choice[depth] = c;
      used |= 1u << c;
      order[depth] = src[c];
      depth++;
      if (depth == k) return true;
      choice[depth] = -1;
    } else {
      if (depth == 0) return false;
      depth--;
      used &= ~(1u << choice[depth]);
    }
  }
}

// Ordering search, bounded-work variant used by the CTA-per-env exact kernel.  src[0..k) sorted descending, k <= 4.  A multiset is playable iff
// there is a chain of sub-multisets 0 c S1 c ... c M whose boards are all legal and whose steps
// are legal half-moves; boards depend only on the sub-multiset, so this is a reachability problem
// on the 2^k subsets (bounded work, no permutation blow-up).  Returns whether M is playable and
// writes the lexicographically first legal ordering (higher sources tried first) to order[].
NHD bool dbl_order_search_dp(const Pos& base, const int* src, int k, int d, int H, int* order) {
  const uint32_t full = (1u << k) - 1u;
  uint32_t own_s[16];
  uint32_t ok = 1u;  // bit S: board of subset S is consistent and legal (the start board counts as legal)
  own_s[0] = base.own;
  uint32_t headbits = 0;
  for (int i = 0; i < k; i++)
    if (src[i] == 23) headbits |= 1u << i;
  for (uint32_t S = 1; S <= full; S++) {
    Pos P = base;
    bool valid = true;
    for (int i = 0; i < k; i++) {  // highest sources first: arrivals precede departures
      if (!((S >> i) & 1u)) continue;
      if (!((P.own >> src[i]) & 1u)) {
        valid = false;
        break;
      }
      P.move(src[i], src[i] - d);
    }
    own_s[S] = P.own;
    if (valid && !violates_block(P.own, base.opp)) ok |= 1u << S;
  }
  if (!((ok >> full) & 1u)) return false;
  // good[S]: from subset S the remaining moves can be completed legally
  uint32_t good = 1u << full;
  for (int S = (int)full - 1; S >= 0; S--) {
    if (!((ok >> S) & 1u)) continue;
    for (int i = 0; i < k; i++) {
      if ((S >> i) & 1) continue;
      uint32_t T = (uint32_t)S | (1u << i);
      if (!((good >> T) & 1u)) continue;
      int s = src[i];
      if (!((own_s[S] >> s) & 1u)) continue;                                  // a checker to move
      if (s - d >= 0 ? ((base.opp >> (s - d)) & 1u) != 0 : (own_s[S] >> 6) != 0u) continue;  // narde.py:69-77
      if (s == 23 && popc32((uint32_t)S & headbits) >= H) continue;           // per-turn head budget
      good |= 1u << S;
      break;
    }
  }
  if (!(good & 1u)) return false;
  uint32_t S = 0;
  for (int step = 0; step < k; step++) {
    for (int i = 0; i < k; i++) {
      if ((S >> i) & 1u) continue;
      uint32_t T = S | (1u << i);
      if (!((good >> T) & 1u)) continue;
      int s = src[i];
      if (!((own_s[S] >> s) & 1u)) continue;
      if (s - d >= 0 ? ((base.opp >> (s - d)) & 1u) != 0 : (own_s[S] >> 6) != 0u) continue;
      if (s == 23 && popc32(S & headbits) >= H) continue;
      order[step] = s;
      S = T;
      break;
    }
  }
  return true;
}

struct DblCtx {
  int d, H, target;
  bool blockchk;
  int maxdepth;
  int n;
  uint32_t first_mask;   // restricts the highest source (level 0) -- lets callers split the tree
  uint32_t second_mask;  // restricts the second source (level 1)
};

template <int K, class Sink>
struct DblLevel {
  static NHD void run(const Pos& base, const Pos& P, DblCtx& cx, int head_used, int last, bool reach,
                      bool desc_ok, uint64_t act, int* src, Sink& sink) {
    uint32_t m = cand_mask(P.own, P.opp, cx.d, head_used < cx.H) & ((2u << last) - 1u);
    if (K == 0) m &= cx.first_mask;
    if (K == 1) m &= cx.second_mask;
    while (m) {
      int s = fls32(m);
      m &= ~(1u << s);
      Pos C = P;
      C.move(s, s - cx.d);
      src[K] = s;
      NPROF(dbl_nodes[K]++);
      bool r = true, dk = true;
      uint64_t a2 = act_set(act, K, s, s - cx.d);
      if (cx.blockchk) {
        bool v = violates_block(C.own, C.opp);
        dk = desc_ok && !v;
        r = false;
        if (!v) {
          if (reach) {
            r = true;
          } else {
            int order[4];
            r = dbl_order_search(base, src, K + 1, cx.d, cx.H, order);
          }
        }
      }
      if (r) {
        if (K + 1 > cx.maxdepth) cx.maxdepth = K + 1;
        if (K + 1 == cx.target) {
          uint64_t out = a2;
          if (!dk) {  // representative = first legal ordering, higher sources tried first
            int order[4];
            dbl_order_search(base, src, K + 1, cx.d, cx.H, order);
            out = ACT_EMPTY;
            for (int i = 0; i <= K; i++) out = act_set(out, i, order[i], order[i] - cx.d);
          }
          sink(out);
          cx.n++;
        }
      }
      if (K + 1 < cx.target) DblLevel<K + 1, Sink>::run(base, C, cx, head_used + (s == 23), s, r, dk, a2, src, sink);
    }
  }
};
template <class Sink>
struct DblLevel<4, Sink> {
  static NHD void run(const Pos&, const Pos&, DblCtx&, int, int, bool, bool, uint64_t, int*, Sink&) {}
};

// Returns the number of legal turn actions; *depth_out = half-moves per action (0 = pass).
template <class Sink>
NHD int enum_double(const Pos& P, int d, bool first_turn, bool blockchk, Sink& sink, int* depth_out) {
  DblCtx cx;
  cx.d = d;
  cx.H = (first_turn && (d == 3 || d == 4 || d == 6)) ? 2 : 1;  // narde.py:100-103 per turn
  cx.blockchk = blockchk;
  cx.target = 4;
  cx.maxdepth = 0;
  cx.n = 0;
  cx.first_mask = 0xFFFFFFu;
  cx.second_mask = 0xFFFFFFu;
  int src[4];
  DblLevel<0, Sink>::run(P, P, cx, 0, 23, true, true, ACT_EMPTY, src, sink);
  NPROF(dbl_env++);
  if (blockchk) NPROF(dbl_block_env++);
  if (cx.n == 0 && cx.maxdepth > 0) {  // max-dice: fewer than 4 playable; re-emit at that depth
    NPROF(dbl_second_pass++);
    cx.target = cx.maxdepth;
    DblLevel<0, Sink>::run(P, P, cx, 0, 23, true, true, ACT_EMPTY, src, sink);
  }
  *depth_out = cx.n ? cx.target : 0;
  return cx.n;
}

// Same walk when the number of playable dice (`target`, 1..4) is already known and the block rule
// cannot matter: one pass, emitting the depth-`target` multisets.
template <class Sink>
NHD int enum_double_at(const Pos& P, int d, int H, int target, Sink& sink) {
  DblCtx cx;
  cx.d = d;
  cx.H = H;
  cx.blockchk = false;
  cx.target = target;
  cx.maxdepth = 0;
  cx.n = 0;
  cx.first_mask = 0xFFFFFFu;
  cx.second_mask = 0xFFFFFFu;
  int src[4];
  DblLevel<0, Sink>::run(P, P, cx, 0, 23, true, true, ACT_EMPTY, src, sink);
  return cx.n;
}

// Sinks ------------------------------------------------------------------------------------
struct CountSink {
  NHD void operator()(uint64_t) {}
};
struct StoreSink {  // stores the first `cap` actions with stride `stride` (in elements)
  uint64_t* out;
  int cap;
  int64_t stride;
  int n;
  NHD void operator()(uint64_t a) {
    if (n < cap) out[(int64_t)n * stride] = a;
    n++;
  }
};
struct PickSink {  // remembers the action at ordinal `want`
  int want;
  int n;
  uint64_t picked;
  NHD void operator()(uint64_t a) {
    if (n == want) picked = a;
    n++;
  }
};
struct StorePickSink {
  uint64_t* out;
  int cap;
  int64_t stride;
  int n;
  NHD void operator()(uint64_t a) {
    if (n < cap) out[(int64_t)n * stride] = a;
    n++;
  }
};

// Enumerate the legal turn actions of `player` in state s for dice (d1, d2).
template <class Sink>
NHD int enumerate_turn(const Pos& P, int d1, int d2, bool first_turn, Sink& sink) {
  bool blockchk = !block_rule_irrelevant(P, d1, d2);
  if (d1 == d2) {
    int depth;
    return enum_double(P, d1, first_turn, blockchk, sink, &depth);
  }
  int a = d1 > d2 ? d1 : d2, b = d1 > d2 ? d2 : d1;
  return enum_nondouble(P, a, b, blockchk, sink);
}

// Apply a packed turn action (mover frame) to the byte board.
NHD void apply_action(State& s, int player, uint64_t act) {
#pragma unroll
  for (int k = 0; k < 4; k++) {
    uint32_t h = (uint32_t)(act >> (16 * k)) & 0xFFFFu;
    if (h == 0xFFFFu) break;
    int from = (int)(h & 0xFF), to = (int)(h >> 8);
    apply_half_move(s, player, from, to == 255 ? -1 : to);
  }
}

// End-of-turn bookkeeping for the full-rules step: termination (narde_env.py:134-141), reward
// (mode 0: README.md:107-108 "+1 iff WHITE wins"; mode 1: reference mover 1/2), player switch.
NHD void finish_turn(State& s, int player, int reward_mode, float* reward, int* done) {
  int r12 = 0;
  bool dn = game_ended(s, player, &r12);
  *reward = reward_mode == 1 ? (float)r12 : ((dn && player == 1) ? 1.0f : 0.0f);
  *done = dn ? 1 : 0;
  uint32_t fl = s.flags();
  if (dn) fl |= FLAG_DONE;
  s.set_meta(s.off_w(), s.off_b(), dn ? player : -player, fl);
  s.set_steps(s.steps() + 1);
}

// off / 15 as float32, bit-identical to numpy's np.float32(off / 15.0): the 16 possible values are
// rounded once from double by the host compiler (no fp64 arithmetic on the device).
#define NARDE_OFF15_TABLE                                                                                   \
  {(float)(0.0 / 15.0),  (float)(1.0 / 15.0),  (float)(2.0 / 15.0),  (float)(3.0 / 15.0),  (float)(4.0 / 15.0),  \
   (float)(5.0 / 15.0),  (float)(6.0 / 15.0),  (float)(7.0 / 15.0),  (float)(8.0 / 15.0),  (float)(9.0 / 15.0),  \
   (float)(10.0 / 15.0), (float)(11.0 / 15.0), (float)(12.0 / 15.0), (float)(13.0 / 15.0), (float)(14.0 / 15.0), \
   (float)(15.0 / 15.0)}
#if defined(__CUDACC__)
__device__ __constant__ float c_off15[16] = NARDE_OFF15_TABLE;
#endif
NHD float off15(int n) {
#if defined(__CUDA_ARCH__)
  return c_off15[n & 15];
#else
  const float t[16] = NARDE_OFF15_TABLE;
  return t[n & 15];
#endif
}

// README.md:44-102: one float2 of the 99 that make an env's Box(198) row.
//   k in [0,48): WHITE point k/2, half k%2;  k == 48: (bar, off)   ; k in [49,97): BLACK
//   k == 97: BLACK (bar, off) ; k == 98: turn one-hot
NHD void obs198_pair(const State& s, int k, float* x, float* y) {
  if (k == 98) {
    *x = s.turn() == 1 ? 1.0f : 0.0f;
    *y = s.turn() == 1 ? 0.0f : 1.0f;
    return;
  }
  int colour = k >= 49 ? 1 : 0;
  int kk = colour ? k - 49 : k;
  if (kk == 48) {
    int off = colour ? s.off_b() : s.off_w();
    *x = 0.0f;                              // bar / 2: no hitting in Narde (narde.py:71)
    *y = off15(off);                        // exactly np.float32(off / 15.0)
    return;
  }
  int v = s.point(kk >> 1);
  int n = colour ? -v : v;
  if (n < 0) n = 0;
  if (kk & 1) {
    *x = n >= 3 ? 1.0f : 0.0f;
    *y = n > 3 ? (float)(n - 3) * 0.5f : 0.0f;
  } else {
    *x = n >= 1 ? 1.0f : 0.0f;
    *y = n >= 2 ? 1.0f : 0.0f;
  }
}

// ------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. SC'11), counter = (env, step_lo, step_hi, stream), key = seed.
// ------------------------------------------------------------------------------------------
struct U4 {
  uint32_t x, y, z, w;
};
NHD U4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; r++) {
    uint32_t h0 = mulhi32(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
    uint32_t h1 = mulhi32(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
    uint32_t n0 = h1 ^ c1 ^ k0, n2 = h0 ^ c3 ^ k1;
    c0 = n0;
    c1 = l1;
    c2 = n2;
    c3 = l0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  U4 o = {c0, c1, c2, c3};
  return o;
}
NHD int die_from_word(uint32_t w) { return 1 + (int)mulhi32(w, 6u); }
NHD U4 turn_random(uint64_t seed, uint32_t env, uint64_t step) {
  return philox4x32_10(env, (uint32_t)step, (uint32_t)(step >> 32), 0u, (uint32_t)seed, (uint32_t)(seed >> 32));
}
// Another stream of the same counter space (stream layout: include/narde_b200.h, narde_segment_sample)
NHD U4 stream_random(uint64_t seed, uint32_t env, uint64_t step, uint32_t stream) {
  return philox4x32_10(env, (uint32_t)step, (uint32_t)(step >> 32), stream, (uint32_t)seed, (uint32_t)(seed >> 32));
}
// narde_env.py:111-117: roll one die each until they differ; the higher roll makes White start
NHD int opening_player(uint64_t seed, uint32_t env, uint64_t step) {
  for (uint32_t attempt = 0; attempt < 32; attempt++) {
    U4 r = philox4x32_10(env, (uint32_t)step, (uint32_t)(step >> 32), 1u + (attempt << 8), (uint32_t)seed,
                         (uint32_t)(seed >> 32));
    int w0 = die_from_word(r.x), b0 = die_from_word(r.y);
    if (w0 != b0) return w0 > b0 ? 1 : -1;
    int w1 = die_from_word(r.z), b1 = die_from_word(r.w);
    if (w1 != b1) return w1 > b1 ? 1 : -1;
  }
  return 1;
}

}  // namespace narde
