/*
 * narde_oracle.c -- TEST INFRASTRUCTURE ONLY (CPU oracle); see narde_oracle.h.
 *
 * Every Tier-R function is a line-by-line restatement of the Python reference; the
 * reference file:line each one follows is cited above it (paths relative to
 * /root/reference).  Written for obviousness, not speed: int arrays and loops, no
 * bit tricks, so that it shares no code or idiom with the CUDA path it checks.
 */
#include "narde_oracle.h"

#include <stdlib.h>
#include <string.h>

/* ------------------------------------------------------------------------------------------
 * Tier R
 * ---------------------------------------------------------------------------------------- */

/* gym_narde/envs/narde.py:21-29 */
void o_game_init(o_game *g) {
  memset(g, 0, sizeof(*g));
  g->board[23] = 15;
  g->board[11] = -15;
  g->borne_off_white = 0;
  g->borne_off_black = 0;
  g->first_turn_white = 1;
  g->first_turn_black = 1;
}

/* gym_narde/envs/narde.py:16-17: concatenate((-board[12:], -board[:12])) */
void o_rotate_board(const int32_t *board, int32_t *out) {
  int32_t tmp[24];
  for (int i = 0; i < 12; i++) tmp[i] = -board[12 + i];
  for (int i = 0; i < 12; i++) tmp[12 + i] = -board[i];
  memcpy(out, tmp, sizeof(tmp));
}

/* gym_narde/envs/narde.py:31-34 */
void o_get_perspective_board(const o_game *g, int player, int32_t *out) {
  if (player == 1)
    memcpy(out, g->board, sizeof(g->board));
  else
    o_rotate_board(g->board, out);
}

/* gym_narde/envs/narde.py:139-184 */
int o_violates_block_rule(const int32_t *board) {
  int i = 0;
  while (i < 24) {
    if (board[i] > 0) {
      int block_start = i;
      int block_length = 1;
      int j = i + 1;
      while (j < 24 && board[j] > 0) {
        block_length += 1;
        j += 1;
      }
      if (block_length >= 6) {
        int has_opponent_ahead = 0;
        for (int k = 0; k < block_start; k++) {
          if (board[k] < 0) {
            has_opponent_ahead = 1;
            break;
          }
        }
        if (!has_opponent_ahead) return 1;
      }
      i = j;
    } else {
      i += 1;
    }
  }
  return 0;
}

static int cmp_desc(const void *a, const void *b) {
  return *(const int32_t *)b - *(const int32_t *)a;
}

/* gym_narde/envs/narde.py:58-92 (candidate loops, block filter) + :94-106 (_validate_head_moves)
 * + :127-137 (_filter_head_moves) */
int o_get_valid_moves(const o_game *g, const int32_t *roll_in, int nroll, int player,
                      int32_t *out_moves) {
  int32_t roll[8];
  int32_t board[24];
  int32_t cand[O_MAX_MOVES * 2];
  int ncand = 0;
  if (nroll > 4) nroll = 4;
  for (int i = 0; i < nroll; i++) roll[i] = roll_in[i];
  qsort(roll, (size_t)nroll, sizeof(int32_t), cmp_desc); /* :59 sorted(roll, reverse=True) */
  if (player == 1)                                        /* :60 */
    memcpy(board, g->board, sizeof(board));
  else
    o_rotate_board(g->board, board);

  for (int r = 0; r < nroll; r++) { /* :64 */
    int die = roll[r];
    for (int pos = 0; pos < 24; pos++) { /* :65 */
      if (board[pos] <= 0) continue;     /* :66 */
      int new_pos = pos - die;           /* :69 */
      if (0 <= new_pos && new_pos < 24) {
        if (board[new_pos] >= 0) { /* :71 */
          cand[2 * ncand] = pos;
          cand[2 * ncand + 1] = new_pos;
          ncand++;
        }
      } else if (new_pos < 0) {
        int outside = 0; /* :75 np.sum(np.maximum(board[6:], 0)) == 0 */
        for (int k = 6; k < 24; k++) outside += board[k] > 0 ? board[k] : 0;
        if (outside == 0) {
          if (die >= pos + 1) { /* :76 */
            cand[2 * ncand] = pos;
            cand[2 * ncand + 1] = O_OFF;
            ncand++;
          }
        }
      }
    }
  }
  /* :78-89 block-rule filter on a copy of the board */
  int32_t filt[O_MAX_MOVES * 2];
  int nfilt = 0;
  for (int m = 0; m < ncand; m++) {
    int32_t copy[24];
    memcpy(copy, board, sizeof(copy));
    int from = cand[2 * m], to = cand[2 * m + 1];
    if (to == O_OFF) {
      copy[from] -= 1;
    } else {
      copy[from] -= 1;
      copy[to] += 1;
    }
    if (!o_violates_block_rule(copy)) {
      filt[2 * nfilt] = from;
      filt[2 * nfilt + 1] = to;
      nfilt++;
    }
  }
  /* :90-106 head rule */
  int first_turn = player == 1 ? g->first_turn_white : g->first_turn_black;
  int max_head_moves = 1;
  if (first_turn && nroll == 2) {
    /* sorted(roll) in [[3,3],[4,4],[6,6]] -- only a 2-element roll can match */
    if (roll[0] == roll[1] && (roll[0] == 3 || roll[0] == 4 || roll[0] == 6)) max_head_moves = 2;
  }
  /* :127-137 */
  int n = 0, head_moves_count = 0;
  for (int m = 0; m < nfilt; m++) {
    if (filt[2 * m] == 23) {
      if (head_moves_count < max_head_moves) {
        out_moves[2 * n] = filt[2 * m];
        out_moves[2 * n + 1] = filt[2 * m + 1];
        n++;
        head_moves_count++;
      }
    } else {
      out_moves[2 * n] = filt[2 * m];
      out_moves[2 * n + 1] = filt[2 * m + 1];
      n++;
    }
  }
  return n;
}

/* gym_narde/envs/narde.py:108-125 */
static void o_execute_move(o_game *g, int from_pos, int to_pos) {
  if (to_pos == O_OFF) {
    if (g->board[from_pos] > 0) {
      g->board[from_pos] -= 1;
      g->borne_off_white += 1;
    } else {
      g->board[from_pos] += 1;
      g->borne_off_black += 1;
    }
  } else {
    if (g->board[from_pos] > 0) {
      g->board[from_pos] -= 1;
      g->board[to_pos] += 1;
    } else {
      g->board[from_pos] += 1;
      g->board[to_pos] -= 1;
    }
  }
}

/* gym_narde/envs/narde.py:36-56 */
void o_execute_rotated_move(o_game *g, int from_pos, int to_pos, int player) {
  if (player != 1) {
    if (to_pos == O_OFF)
      o_execute_move(g, (from_pos + 12) % 24, O_OFF);
    else
      o_execute_move(g, (from_pos + 12) % 24, (to_pos + 12) % 24);
  } else {
    o_execute_move(g, from_pos, to_pos);
  }
  if (player == 1)
    g->first_turn_white = 0;
  else
    g->first_turn_black = 0;
}

/* gym_narde/envs/narde_env.py:134-141 */
int o_check_game_ended(const o_env *e, int32_t *reward) {
  if (e->current_player == 1 && e->game.borne_off_white == 15) {
    *reward = e->game.borne_off_black > 0 ? 1 : 2;
    return 1;
  } else if (e->current_player == -1 && e->game.borne_off_black == 15) {
    *reward = e->game.borne_off_white > 0 ? 1 : 2;
    return 1;
  }
  *reward = 0;
  return 0;
}

/* gym_narde/envs/narde_env.py:105-120 (np.random.seed is the caller's business: the dice
 * arrive as an explicit stream, white_roll then black_roll, repeated until they differ) */
int o_env_reset(o_env *e, const int32_t *rolls, int nrolls) {
  o_game_init(&e->game);
  int used = 0;
  for (;;) {
    if (used + 2 > nrolls) return -1;
    int white_roll = rolls[used], black_roll = rolls[used + 1];
    used += 2;
    if (white_roll != black_roll) {
      e->current_player = white_roll > black_roll ? 1 : -1;
      break;
    }
  }
  return used;
}

static int move_in_list(const int32_t *moves, int n, int from, int to) {
  for (int i = 0; i < n; i++)
    if (moves[2 * i] == from && moves[2 * i + 1] == to) return 1;
  return 0;
}

/* gym_narde/envs/narde_env.py:27-103.  Codes must be in [0,576) (Discrete(576)). */
void o_env_step(o_env *e, int d1, int d2, int code1, int code2, int32_t *obs24, int32_t *reward,
                int32_t *done) {
  int32_t dice[2] = {d1, d2}; /* :29, unsorted */
  int32_t valid[O_MAX_MOVES * 2];
  int n = o_get_valid_moves(&e->game, dice, 2, e->current_player, valid); /* :31 */
  int32_t rew = 0;
  int dn = 0;
  if (n == 0) { /* :33-39 */
    dn = o_check_game_ended(e, &rew);
    if (!dn) e->current_player *= -1;
    o_get_perspective_board(&e->game, e->current_player, obs24);
    *reward = rew;
    *done = dn;
    return;
  } else if (n == 1) { /* :41-43 */
    o_execute_rotated_move(&e->game, valid[0], valid[1], e->current_player);
  } else { /* :44-93 */
    int from1 = code1 / 24, to1 = code1 % 24;
    if (to1 == 0 && 0 <= from1 && from1 <= 5) to1 = O_OFF; /* :50-53 */
    int from2 = code2 / 24, to2 = code2 % 24;
    if (to2 == 0 && 0 <= from2 && from2 <= 5) to2 = O_OFF; /* :59-62 */
    if (move_in_list(valid, n, from1, to1)) {              /* :63 */
      o_execute_rotated_move(&e->game, from1, to1, e->current_player);
      int move_distance; /* :69-74 */
      if (to1 == O_OFF)
        move_distance = from1 + 1;
      else
        move_distance = abs(from1 - to1);
      int32_t temp[2] = {dice[0], dice[1]}; /* :77-83 */
      int ntemp = 2;
      if (temp[0] == move_distance) { /* list.remove: first occurrence */
        temp[0] = temp[1];
        ntemp = 1;
      } else if (temp[1] == move_distance) {
        ntemp = 1;
      } else { /* pop(0) */
        temp[0] = temp[1];
        ntemp = 1;
      }
      if (ntemp) { /* :86-90 */
        int32_t nv[O_MAX_MOVES * 2];
        int nn = o_get_valid_moves(&e->game, temp, ntemp, e->current_player, nv);
        if (move_in_list(nv, nn, from2, to2))
          o_execute_rotated_move(&e->game, from2, to2, e->current_player);
      }
    }
  }
  dn = o_check_game_ended(e, &rew);     /* :96 */
  if (!dn) e->current_player *= -1;     /* :99-100 */
  o_get_perspective_board(&e->game, e->current_player, obs24); /* :103 */
  *reward = rew;
  *done = dn;
}

/* ------------------------------------------------------------------------------------------
 * Tier N (README contract; SURVEY.md section 8c "N1/N2/N3").  No reference code exists for
 * these; the per-ply legality is the reference's own get_valid_moves([die]) on a scratch game.
 * ---------------------------------------------------------------------------------------- */

typedef struct {
  int depth;
  int ord;              /* 0: dice list as given (hi first / doubles); 1: lo first */
  int32_t board[24];
  int32_t off;
  int32_t seq[8];
} o_node;

typedef struct {
  o_node *v;
  size_t n, cap;
  int64_t visited;
} o_nodes;

static void nodes_push(o_nodes *ns, const o_node *nd) {
  if (ns->n == ns->cap) {
    ns->cap = ns->cap ? ns->cap * 2 : 256;
    ns->v = (o_node *)realloc(ns->v, ns->cap * sizeof(o_node));
  }
  ns->v[ns->n++] = *nd;
}

static void turn_dfs(const o_game *cur, const int32_t *dice, int ndice, int depth, int head_used,
                     int max_head, int ord, const int32_t *seq, o_nodes *ns) {
  if (depth == ndice) return;
  int32_t one[1] = {dice[depth]};
  int32_t mv[O_MAX_MOVES * 2];
  /* per-ply candidates = the reference's single-die list on a scratch game (narde.py:58-92) */
  int n = o_get_valid_moves(cur, one, 1, 1, mv);
  for (int i = 0; i < n; i++) {
    int from = mv[2 * i], to = mv[2 * i + 1];
    /* per-TURN head budget (narde.py:5 rule text; tests/test_narde_game_manager.py:77-129) */
    if (from == 23 && head_used >= max_head) continue;
    o_game child = *cur;
    o_execute_rotated_move(&child, from, to, 1);
    o_node nd;
    nd.depth = depth + 1;
    nd.ord = ord;
    memcpy(nd.board, child.board, sizeof(nd.board));
    nd.off = child.borne_off_white;
    for (int k = 0; k < 8; k++) nd.seq[k] = seq[k];
    nd.seq[2 * depth] = from;
    nd.seq[2 * depth + 1] = to;
    ns->visited++;
    nodes_push(ns, &nd);
    turn_dfs(&child, dice, ndice, depth + 1, head_used + (from == 23), max_head, ord, nd.seq, ns);
  }
}

typedef struct {
  o_turn_action act;
  int32_t rank; /* tie-break rank of the representative sequence within its afterstate */
} o_cand;

static int cmp_cand_board(const void *a, const void *b) {
  const o_cand *x = (const o_cand *)a, *y = (const o_cand *)b;
  int c = memcmp(x->act.after, y->act.after, sizeof(x->act.after));
  if (c) return c;
  if (x->act.key != y->act.key) return x->act.key < y->act.key ? -1 : 1;
  return x->rank < y->rank ? -1 : (x->rank > y->rank ? 1 : 0);
}

static int cmp_cand_key(const void *a, const void *b) {
  const o_cand *x = (const o_cand *)a, *y = (const o_cand *)b;
  return x->act.key < y->act.key ? -1 : (x->act.key > y->act.key ? 1 : 0);
}

static int cmp_int_asc(const void *a, const void *b) {
  return *(const int32_t *)a - *(const int32_t *)b;
}

int o_turn_enumerate(const int32_t *board_mover, int mover_off, int d1, int d2, int first_turn,
                     int cap, o_turn_action *out, int64_t *n_nodes) {
  o_game base;
  memset(&base, 0, sizeof(base));
  memcpy(base.board, board_mover, sizeof(base.board));
  base.borne_off_white = mover_off;
  int hi = d1 > d2 ? d1 : d2, lo = d1 > d2 ? d2 : d1;
  int doubles = d1 == d2;
  /* narde.py:100-103: two head checkers only on the first turn with 3-3, 4-4 or 6-6 */
  int max_head = (first_turn && doubles && (hi == 3 || hi == 4 || hi == 6)) ? 2 : 1;
  int32_t seq0[8] = {O_NONE, O_NONE, O_NONE, O_NONE, O_NONE, O_NONE, O_NONE, O_NONE};
  o_nodes ns = {0, 0, 0, 0};
  if (doubles) {
    int32_t dice[4] = {hi, hi, hi, hi};
    turn_dfs(&base, dice, 4, 0, 0, max_head, 0, seq0, &ns);
  } else {
    int32_t da[2] = {hi, lo}, db[2] = {lo, hi};
    turn_dfs(&base, da, 2, 0, 0, max_head, 0, seq0, &ns);
    turn_dfs(&base, db, 2, 0, 0, max_head, 1, seq0, &ns);
  }
  if (n_nodes) *n_nodes = ns.visited;
  int maxlen = 0;
  for (size_t i = 0; i < ns.n; i++)
    if (ns.v[i].depth > maxlen) maxlen = ns.v[i].depth;
  if (maxlen == 0) {
    free(ns.v);
    return 0;
  }
  /* "if only one is possible, use the higher die" (narde.py:6 rule 4) */
  int hi_only = 0;
  if (!doubles && maxlen == 1)
    for (size_t i = 0; i < ns.n; i++)
      if (ns.v[i].depth == 1 && ns.v[i].ord == 0) hi_only = 1;

  o_cand *cs = (o_cand *)malloc((ns.n ? ns.n : 1) * sizeof(o_cand));
  size_t nc = 0;
  for (size_t i = 0; i < ns.n; i++) {
    const o_node *nd = &ns.v[i];
    if (nd->depth != maxlen) continue;
    if (!doubles && maxlen == 1 && hi_only && nd->ord != 0) continue;
    o_cand c;
    memset(&c, 0, sizeof(c));
    c.act.n_moves = maxlen;
    memcpy(c.act.moves, nd->seq, sizeof(c.act.moves));
    memcpy(c.act.after, nd->board, sizeof(c.act.after));
    c.act.after_off = nd->off;
    /* canonical key, digit(s) = 23 - s so that higher sources sort first */
    if (doubles || maxlen == 1) {
      int32_t dg[4];
      int32_t code = 0;
      for (int k = 0; k < maxlen; k++) {
        dg[k] = 23 - nd->seq[2 * k];
        code = code * 32 + dg[k];
      }
      qsort(dg, (size_t)maxlen, sizeof(int32_t), cmp_int_asc);
      int32_t key = 0;
      for (int k = 0; k < maxlen; k++) key = key * 32 + dg[k];
      c.act.key = key; /* sources sorted descending */
      c.rank = code;   /* play-order code; smallest legal ordering is the representative */
    } else {
      int p = nd->ord == 0 ? nd->seq[0] : nd->seq[2]; /* source moved with the higher die */
      int q = nd->ord == 0 ? nd->seq[2] : nd->seq[0]; /* source moved with the lower die */
      c.act.key = (23 - p) * 32 + (23 - q);
      c.rank = nd->ord; /* prefer playing the higher die first */
    }
    cs[nc++] = c;
  }
  free(ns.v);
  /* group by afterstate; the first entry of each group (smallest key, then rank) represents it */
  qsort(cs, nc, sizeof(o_cand), cmp_cand_board);
  size_t ng = 0;
  for (size_t i = 0; i < nc; i++) {
    if (i == 0 || memcmp(cs[i].act.after, cs[i - 1].act.after, sizeof(cs[i].act.after)) != 0)
      cs[ng++] = cs[i];
  }
  qsort(cs, ng, sizeof(o_cand), cmp_cand_key);
  for (size_t i = 0; i < ng && (int)i < cap; i++) out[i] = cs[i].act;
  free(cs);
  return (int)ng;
}

/* README.md:44-102 (layout) and tests/test_observation_space.py:5-202 (bounds) */
void o_obs198(const int32_t *board_abs, int off_w, int off_b, int player, float *out) {
  int k = 0;
  for (int colour = 0; colour < 2; colour++) {
    for (int i = 0; i < 24; i++) {
      int n = colour == 0 ? board_abs[i] : -board_abs[i];
      if (n < 0) n = 0;
      out[k++] = n >= 1 ? 1.0f : 0.0f;
      out[k++] = n >= 2 ? 1.0f : 0.0f;
      out[k++] = n >= 3 ? 1.0f : 0.0f;
      out[k++] = n > 3 ? (float)((double)(n - 3) / 2.0) : 0.0f;
    }
    out[k++] = 0.0f; /* bar / 2: Narde has no hitting (narde.py:71), the bar is always empty */
    out[k++] = (float)((double)(colour == 0 ? off_w : off_b) / 15.0);
  }
  out[k++] = player == 1 ? 1.0f : 0.0f;
  out[k++] = player == 1 ? 0.0f : 1.0f;
}

/* Plays turn action a (NULL: no legal action) for the side to move and finishes the turn: the end-of-game check
 * (narde_env.py:96) and, unless the game ended, the player switch (:99-100).  Returns the done flag; *rew12 receives
 * the mover reward of o_check_game_ended. */
static int o_play_turn(o_env *e, const o_turn_action *a, int32_t *rew12) {
  const int player = e->current_player;
  if (a)
    for (int k = 0; k < a->n_moves; k++)
      o_execute_rotated_move(&e->game, a->moves[2 * k], a->moves[2 * k + 1], player);
  *rew12 = 0;
  const int dn = o_check_game_ended(e, rew12);
  if (!dn) e->current_player *= -1;
  return dn;
}

/* The mover's canonical turn list of e with dice (d1, d2): up to cap entries, returns the full count */
static int o_enumerate_env(const o_env *e, int d1, int d2, int cap, o_turn_action *out) {
  int32_t mover[24];
  const int player = e->current_player;
  o_get_perspective_board(&e->game, player, mover);
  return o_turn_enumerate(mover, player == 1 ? e->game.borne_off_white : e->game.borne_off_black, d1, d2,
                          player == 1 ? e->game.first_turn_white : e->game.first_turn_black, cap, out, 0);
}

int o_full_step(o_env *e, int d1, int d2, int action_idx, int reward_mode, float *reward,
                int32_t *done, float *obs198) {
  int player = e->current_player;
  int cap = 4096;
  static __thread o_turn_action *acts = 0; /* per-thread scratch, allocated once */
  if (!acts) acts = (o_turn_action *)malloc((size_t)cap * sizeof(o_turn_action));
  int n = o_enumerate_env(e, d1, d2, cap, acts);
  const o_turn_action *a = 0;
  if (n > 0) {
    if (action_idx < 0) action_idx = 0;
    if (action_idx >= n) action_idx = n - 1;
    a = &acts[action_idx];
  }
  int32_t rew12;
  int dn = o_play_turn(e, a, &rew12);
  if (reward_mode == 1)
    *reward = (float)rew12;
  else
    *reward = (dn && player == 1) ? 1.0f : 0.0f; /* README.md:107-108 */
  *done = dn;
  if (obs198)
    o_obs198(e->game.board, e->game.borne_off_white, e->game.borne_off_black, e->current_player,
             obs198);
  return n;
}

/* ------------------------------------------------------------------------------------------
 * Philox4x32-10 (Salmon et al., "Parallel random numbers: as easy as 1, 2, 3", SC'11; the same
 * generator as curand's curand_philox4x32_x.h).  Restated from the published algorithm.
 * ---------------------------------------------------------------------------------------- */
void o_philox4x32_10(const uint32_t ctr_in[4], const uint32_t key_in[2], uint32_t out[4]) {
  uint32_t c0 = ctr_in[0], c1 = ctr_in[1], c2 = ctr_in[2], c3 = ctr_in[3];
  uint32_t k0 = key_in[0], k1 = key_in[1];
  for (int r = 0; r < 10; r++) {
    uint64_t p0 = (uint64_t)0xD2511F53u * c0;
    uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
    uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
    uint32_t n1 = (uint32_t)p1;
    uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    uint32_t n3 = (uint32_t)p0;
    c0 = n0;
    c1 = n1;
    c2 = n2;
    c3 = n3;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  out[0] = c0;
  out[1] = c1;
  out[2] = c2;
  out[3] = c3;
}

static int die_from_word(uint32_t w) { return 1 + (int)(((uint64_t)w * 6u) >> 32); }

void o_turn_dice(uint64_t seed, uint32_t env, uint64_t step, int32_t *d1, int32_t *d2,
                 uint32_t *action_word) {
  uint32_t ctr[4] = {env, (uint32_t)step, (uint32_t)(step >> 32), 0u};
  uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
  uint32_t w[4];
  o_philox4x32_10(ctr, key, w);
  *d1 = die_from_word(w[0]);
  *d2 = die_from_word(w[1]);
  if (action_word) *action_word = w[2];
}

int o_opening_player(uint64_t seed, uint32_t env, uint64_t step) {
  uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
  for (uint32_t attempt = 0; attempt < 32; attempt++) {
    uint32_t ctr[4] = {env, (uint32_t)step, (uint32_t)(step >> 32), 1u + (attempt << 8)};
    uint32_t w[4];
    o_philox4x32_10(ctr, key, w);
    for (int h = 0; h < 2; h++) {
      int white_roll = die_from_word(w[2 * h]), black_roll = die_from_word(w[2 * h + 1]);
      if (white_roll != black_roll) return white_roll > black_roll ? 1 : -1; /* narde_env.py:117 */
    }
  }
  return 1;
}

/* ------------------------------------------------------------------------------------------
 * CPU baseline driver (bench.py cpu_baseline / --impl reference): full-rules random self-play of
 * n_envs environments for n_steps lock-step turns, same Philox dice/action stream and auto-reset
 * as the CUDA path, one Box(198) observation per env step.  Returns env steps executed.
 * ---------------------------------------------------------------------------------------- */
int64_t o_selfplay(uint64_t seed, uint32_t env_base, int n_envs, int n_steps, uint64_t step0,
                   int64_t *sum_actions, int64_t *episodes, double *obs_checksum) {
  o_env *envs = (o_env *)malloc((size_t)n_envs * sizeof(o_env));
  float obs[198];
  int64_t steps = 0, acts = 0, eps = 0;
  double chk = 0.0;
  for (int i = 0; i < n_envs; i++) {
    o_game_init(&envs[i].game);
    envs[i].current_player = o_opening_player(seed, env_base + (uint32_t)i, step0);
  }
  for (int t = 1; t <= n_steps; t++) {
    for (int i = 0; i < n_envs; i++) {
      int32_t d1, d2;
      uint32_t w;
      o_turn_dice(seed, env_base + (uint32_t)i, step0 + (uint64_t)t, &d1, &d2, &w);
      /* count first (to map the action word to an index), then step */
      int32_t mover[24];
      o_env *e = &envs[i];
      int pl = e->current_player;
      o_get_perspective_board(&e->game, pl, mover);
      float rew;
      int32_t done;
      /* o_full_step clamps the index; compute it from the count exactly like the CUDA path */
      static __thread o_turn_action *scratch = 0;
      if (!scratch) scratch = (o_turn_action *)malloc(4096 * sizeof(o_turn_action));
      int n = o_turn_enumerate(mover, pl == 1 ? e->game.borne_off_white : e->game.borne_off_black, d1, d2,
                               pl == 1 ? e->game.first_turn_white : e->game.first_turn_black, 4096, scratch, 0);
      int idx = n ? (int)(((uint64_t)w * (uint64_t)n) >> 32) : 0;
      if (n > 0) {
        const o_turn_action *a = &scratch[idx];
        for (int k = 0; k < a->n_moves; k++)
          o_execute_rotated_move(&e->game, a->moves[2 * k], a->moves[2 * k + 1], pl);
      }
      int32_t r12;
      done = o_check_game_ended(e, &r12);
      rew = (done && pl == 1) ? 1.0f : 0.0f;
      if (!done) e->current_player *= -1;
      if (done) {
        eps++;
        o_game_init(&e->game);
        e->current_player = o_opening_player(seed, env_base + (uint32_t)i, step0 + (uint64_t)t);
      }
      o_obs198(e->game.board, e->game.borne_off_white, e->game.borne_off_black, e->current_player, obs);
      chk += obs[97] + obs[195] + rew;
      acts += n;
      steps++;
    }
  }
  free(envs);
  if (sum_actions) *sum_actions = acts;
  if (episodes) *episodes = eps;
  if (obs_checksum) *obs_checksum = chk;
  return steps;
}

/* ------------------------------------------------------------------------------------------
 * Bulk trace of full-rules self-play (tests + bench.py's cpu_baseline leg): what o_selfplay plays,
 * written out turn by turn so that a run of the CUDA path at its benchmarked size (131 072 envs,
 * hundreds of graph-replayed steps) can be compared record by record.  The state records use the
 * boundary's own data format (include/narde_b200.h "State record": two 16-byte lanes per env).
 * ---------------------------------------------------------------------------------------- */

/* include/narde_b200.h:19-24 */
void o_pack_state(const o_env *e, int terminated, int episode_steps, uint8_t *lo16, uint8_t *hi16) {
  for (int k = 0; k < 16; k++) lo16[k] = (uint8_t)(int8_t)e->game.board[k];
  for (int k = 0; k < 8; k++) hi16[k] = (uint8_t)(int8_t)e->game.board[16 + k];
  hi16[8] = (uint8_t)e->game.borne_off_white;
  hi16[9] = (uint8_t)e->game.borne_off_black;
  hi16[10] = (uint8_t)(int8_t)e->current_player;
  hi16[11] = (uint8_t)((e->game.first_turn_white ? 1 : 0) | (e->game.first_turn_black ? 2 : 0) |
                       (terminated ? 4 : 0));
  hi16[12] = (uint8_t)(episode_steps & 0xFF);
  hi16[13] = (uint8_t)((episode_steps >> 8) & 0xFF);
  hi16[14] = hi16[15] = 0;
}

void o_unpack_state(const uint8_t *lo16, const uint8_t *hi16, o_env *e, int *terminated,
                    int *episode_steps) {
  for (int k = 0; k < 16; k++) e->game.board[k] = (int8_t)lo16[k];
  for (int k = 0; k < 8; k++) e->game.board[16 + k] = (int8_t)hi16[k];
  e->game.borne_off_white = hi16[8];
  e->game.borne_off_black = hi16[9];
  e->current_player = (int8_t)hi16[10];
  e->game.first_turn_white = (hi16[11] & 1) ? 1 : 0;
  e->game.first_turn_black = (hi16[11] & 2) ? 1 : 0;
  *terminated = (hi16[11] & 4) ? 1 : 0;
  *episode_steps = hi16[12] | (hi16[13] << 8);
}

/* include/narde_b200.h:28-29: u64 = 4 x u16 half-moves (from | to << 8), 255 = bear off,
 * 0xFFFF = unused slot */
uint64_t o_pack_action(const o_turn_action *a) {
  uint64_t v = 0;
  for (int k = 0; k < 4; k++) {
    uint64_t h = 0xFFFFu;
    if (k < a->n_moves) {
      int from = a->moves[2 * k], to = a->moves[2 * k + 1];
      h = (uint64_t)(from & 0xFF) | ((uint64_t)(to == O_OFF ? 255 : to) << 8);
    }
    v |= h << (16 * k);
  }
  return v;
}

/* position-sensitive checksum of a stored action list: sum_k act[k] * m(k) mod 2^64, m(k) odd
 * (splitmix64 of k) -- the test computes the same sum over the CUDA path's [N, cap] buffer */
uint64_t o_list_weight(int k) {
  uint64_t z = (uint64_t)(k + 1) * 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z ^= z >> 31;
  return z | 1ull;
}

int64_t o_selfplay_trace(uint64_t seed, uint32_t env_base, int n_envs, int n_steps, uint64_t step0,
                         const uint8_t *init_lo, const uint8_t *init_hi, const uint32_t *words,
                         int64_t words_stride, int word_mode, int cap, int reward_mode, int autoreset,
                         int max_episode_steps, int64_t row_stride, uint8_t *out_lo, uint8_t *out_hi,
                         int64_t *out_chosen, int32_t *out_count, uint8_t *out_dice, uint8_t *out_done,
                         float *out_reward, uint64_t *out_hash, int64_t *stats8, double *obs_checksum) {
  o_env *envs = (o_env *)malloc((size_t)n_envs * sizeof(o_env));
  float obs[198];
  double chk = 0.0;
  int *term = (int *)calloc((size_t)n_envs, sizeof(int));
  int *esteps = (int *)calloc((size_t)n_envs, sizeof(int));
  o_turn_action *scratch = (o_turn_action *)malloc(4096 * sizeof(o_turn_action));
  uint64_t wt[4096];
  for (int k = 0; k < 4096; k++) wt[k] = o_list_weight(k);
  int64_t st[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  int64_t turns = 0;
  for (int i = 0; i < n_envs; i++) {
    if (init_lo && init_hi) {
      o_unpack_state(init_lo + 16 * (size_t)i, init_hi + 16 * (size_t)i, &envs[i], &term[i], &esteps[i]);
    } else { /* narde_env.py:105-120 with the roll-off taken from the Philox stream */
      o_game_init(&envs[i].game);
      envs[i].current_player = o_opening_player(seed, env_base + (uint32_t)i, step0);
    }
  }
  for (int t = 1; t <= n_steps; t++) {
    const uint64_t step = step0 + (uint64_t)t;
    for (int i = 0; i < n_envs; i++) {
      o_env *e = &envs[i];
      const size_t r = (size_t)(t - 1) * (size_t)row_stride + (size_t)i;
      int32_t d1 = 0, d2 = 0, n = 0;
      uint64_t chosen = ~0ull, hash = 0;
      float rew = 0.0f;
      int bits = 0;
      if (term[i]) { /* without auto-reset a finished env idles: nothing changes, done stays set */
        bits = 1;
      } else {
        uint32_t w;
        o_turn_dice(seed, env_base + (uint32_t)i, step, &d1, &d2, &w);
        int pl = e->current_player;
        int32_t mover[24];
        o_get_perspective_board(&e->game, pl, mover);
        n = o_turn_enumerate(mover, pl == 1 ? e->game.borne_off_white : e->game.borne_off_black, d1, d2,
                             pl == 1 ? e->game.first_turn_white : e->game.first_turn_black, 4096, scratch, 0);
        int idx = 0;
        if (n > 0) {
          if (words && word_mode == 0) { /* caller's index, clamped */
            int32_t v = (int32_t)words[(size_t)(t - 1) * (size_t)words_stride + (size_t)i];
            idx = v < 0 ? 0 : (v >= n ? n - 1 : v);
          } else { /* u32 fraction of the list: the caller's, or the turn's Philox word */
            uint32_t f = words ? words[(size_t)(t - 1) * (size_t)words_stride + (size_t)i] : w;
            idx = (int)(((uint64_t)f * (uint64_t)n) >> 32);
          }
          const o_turn_action *a = &scratch[idx];
          chosen = o_pack_action(a);
          for (int k = 0; k < a->n_moves; k++)
            o_execute_rotated_move(&e->game, a->moves[2 * k], a->moves[2 * k + 1], pl);
          int stored = n < cap ? n : cap;
          if (stored > 4096) stored = 4096;
          for (int k = 0; k < stored; k++) hash += o_pack_action(&scratch[k]) * wt[k];
        }
        int32_t r12;
        int dn = o_check_game_ended(e, &r12); /* narde_env.py:96 */
        rew = reward_mode == 1 ? (float)r12 : ((dn && pl == 1) ? 1.0f : 0.0f); /* README.md:107-108 */
        if (!dn) e->current_player *= -1; /* narde_env.py:99-100 */
        esteps[i] += 1;
        bits = dn ? 1 : 0;
        /* gymnasium TimeLimit (gym_narde/__init__.py:6 max_episode_steps) */
        if (!dn && max_episode_steps > 0 && esteps[i] >= max_episode_steps) bits |= 2;
        st[5] += n;
        if (n > st[6]) st[6] = n;
        if (n > cap) st[7] += 1;
        if (bits) {
          st[0] += 1;
          st[4] += esteps[i];
          if (dn) {
            st[pl == 1 ? 1 : 2] += 1;
            int loser_off = pl == 1 ? e->game.borne_off_black : e->game.borne_off_white;
            if (loser_off == 0) st[3] += 1;
          }
          if (autoreset) {
            o_game_init(&e->game);
            e->current_player = o_opening_player(seed, env_base + (uint32_t)i, step);
            esteps[i] = 0;
          } else if (dn) {
            term[i] = 1;
          }
        }
        turns++;
      }
      if (obs_checksum) { /* the CUDA step writes one Box(198) row per env turn: do that work here too */
        o_obs198(e->game.board, e->game.borne_off_white, e->game.borne_off_black, e->current_player, obs);
        for (int k = 0; k < 198; k++) chk += obs[k];
      }
      if (out_lo && out_hi) o_pack_state(e, term[i], esteps[i], out_lo + 16 * r, out_hi + 16 * r);
      if (out_chosen) out_chosen[r] = (int64_t)chosen;
      if (out_count) out_count[r] = n;
      if (out_dice) {
        out_dice[2 * r] = (uint8_t)d1;
        out_dice[2 * r + 1] = (uint8_t)d2;
      }
      if (out_done) out_done[r] = (uint8_t)bits;
      if (out_reward) out_reward[r] = rew;
      if (out_hash) out_hash[r] = hash;
    }
  }
  if (stats8)
    for (int k = 0; k < 8; k++) stats8[k] = st[k];
  if (obs_checksum) *obs_checksum = chk;
  free(envs);
  free(term);
  free(esteps);
  free(scratch);
  return turns;
}

/* get_valid_actions (README.md:156-165) for n packed positions with given dice: legal-action count and the
 * checksum of the first min(count, cap) canonical list entries (as o_selfplay_trace computes it). */
void o_enumerate_batch(const uint8_t *lo, const uint8_t *hi, const uint8_t *dice, int64_t n, int cap,
                       int32_t *out_count, uint64_t *out_hash) {
  o_turn_action *scratch = (o_turn_action *)malloc(4096 * sizeof(o_turn_action));
  for (int64_t i = 0; i < n; i++) {
    o_env e;
    int term, esteps;
    o_unpack_state(lo + 16 * i, hi + 16 * i, &e, &term, &esteps);
    int cnt = 0;
    uint64_t hash = 0;
    if (!term) {
      int pl = e.current_player;
      int32_t mover[24];
      o_get_perspective_board(&e.game, pl, mover);
      cnt = o_turn_enumerate(mover, pl == 1 ? e.game.borne_off_white : e.game.borne_off_black, dice[2 * i],
                             dice[2 * i + 1], pl == 1 ? e.game.first_turn_white : e.game.first_turn_black, 4096,
                             scratch, 0);
      int stored = cnt < cap ? cnt : cap;
      if (stored > 4096) stored = 4096;
      for (int k = 0; k < stored; k++) hash += o_pack_action(&scratch[k]) * o_list_weight(k);
    }
    out_count[i] = cnt;
    out_hash[i] = hash;
  }
  free(scratch);
}

/* The afterstate rows of narde_afterstates_scan for n packed positions with given dice: counts_out[i] = the number of
 * legal turn actions (0 for a finished game), and for each of the first min(count, cap) canonical actions k the packed
 * action word (actions_out[i*cap + k]) and the state after playing it and finishing the turn as o_full_step does
 * (as_lo_out / as_hi_out row i*cap + k): terminated bit set when the game ended, episode steps + 1.  Entries at
 * k >= min(count, cap) are not written. */
void o_afterstates_batch(const uint8_t *lo, const uint8_t *hi, const uint8_t *dice, int64_t n, int cap,
                         int32_t *counts_out, uint64_t *actions_out, uint8_t *as_lo_out, uint8_t *as_hi_out) {
  o_turn_action *scratch = (o_turn_action *)malloc(4096 * sizeof(o_turn_action));
  for (int64_t i = 0; i < n; i++) {
    o_env e;
    int term, esteps;
    o_unpack_state(lo + 16 * i, hi + 16 * i, &e, &term, &esteps);
    const int cnt = term ? 0 : o_enumerate_env(&e, dice[2 * i], dice[2 * i + 1], 4096, scratch);
    counts_out[i] = cnt;
    const int stored = cnt < cap ? cnt : cap;
    for (int k = 0; k < stored; k++) {
      const size_t r = (size_t)i * (size_t)cap + (size_t)k;
      o_env t = e;
      int32_t rew12;
      const int dn = o_play_turn(&t, &scratch[k], &rew12);
      actions_out[r] = o_pack_action(&scratch[k]);
      o_pack_state(&t, dn, esteps + 1, as_lo_out + 16 * r, as_hi_out + 16 * r);
    }
  }
  free(scratch);
}
