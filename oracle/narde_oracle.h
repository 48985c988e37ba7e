/*
 * narde_oracle.h -- TEST INFRASTRUCTURE ONLY (CPU oracle).
 *
 * Plain-C restatement of the reference's rules engine and env step
 * (/root/reference/gym_narde/envs/narde.py, narde_env.py), plus the Tier-N
 * (README contract) turn enumeration composed from those primitives.
 *
 * Nothing under gym_narde_b200/ (the product) may include, link or call this.
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
 * --impl reference legs use it, and only as the checker / the CPU arm.
 *
 * Parity status: Tier R functions are PINNED against the real reference
 * (tests/test_oracle_vs_reference.py runs the Python reference in the build
 * container; tests/golden/ holds vectors generated from it).  Tier N functions
 * have no reference code: they are pinned only through the reference's own
 * per-ply primitive (get_valid_moves on a scratch game) and the KATs in
 * tests/golden/tier_n_kat.json.
 */
#ifndef NARDE_ORACLE_H
#define NARDE_ORACLE_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define O_OFF (-1)        /* the reference's 'off' destination */
#define O_NONE (-2)       /* empty half-move slot */
#define O_MAX_MOVES 96    /* 4 dice x 24 points */

typedef struct {
  int32_t board[24];            /* narde.py:23-25, White frame */
  int32_t borne_off_white;      /* narde.py:26 */
  int32_t borne_off_black;      /* narde.py:27 */
  int32_t first_turn_white;     /* narde.py:28 */
  int32_t first_turn_black;     /* narde.py:29 */
} o_game;

typedef struct {
  o_game game;                  /* narde_env.py:13 */
  int32_t current_player;       /* narde_env.py:14 (+1 White, -1 Black) */
} o_env;

/* ---- Tier R: literal restatement of the reference ---- */
void o_game_init(o_game *g);
void o_rotate_board(const int32_t *board, int32_t *out);
void o_get_perspective_board(const o_game *g, int player, int32_t *out);
int o_violates_block_rule(const int32_t *board);
/* moves: [n][2] = (from, to) with to == O_OFF for 'off'; returns n */
int o_get_valid_moves(const o_game *g, const int32_t *roll, int nroll, int player, int32_t *moves);
void o_execute_rotated_move(o_game *g, int from_pos, int to_pos, int player);
int o_check_game_ended(const o_env *e, int32_t *reward);
/* consumes dice rolls pairwise from `rolls` until white != black; returns #values consumed
 * (or -1 if the stream ran out) */
int o_env_reset(o_env *e, const int32_t *rolls, int nrolls);
void o_env_step(o_env *e, int d1, int d2, int code1, int code2, int32_t *obs24, int32_t *reward,
                int32_t *done);

/* ---- Tier N: README contract, composed from the primitives above ---- */
typedef struct {
  int32_t n_moves;              /* half-moves in this turn action (0..4) */
  int32_t moves[8];             /* (from,to) x4 in play order, mover frame; O_NONE padding */
  int32_t key;                  /* canonical sort key (see DESIGN.md "canonical action order") */
  int32_t after[24];            /* afterstate board, mover frame */
  int32_t after_off;            /* mover's borne-off count after the turn */
} o_turn_action;

/* Enumerate all legal full-turn actions.  board_mover: 24 ints in the mover's frame.
 * Returns the total number of distinct afterstates; writes min(total, cap) sorted entries.
 * n_nodes (optional) receives the number of DFS nodes visited. */
int o_turn_enumerate(const int32_t *board_mover, int mover_off, int d1, int d2, int first_turn,
                     int cap, o_turn_action *out, int64_t *n_nodes);

void o_obs198(const int32_t *board_abs, int off_w, int off_b, int player, float *out198);

/* Full-rules env step on an o_env (absolute frame). action_idx indexes o_turn_enumerate's list.
 * reward_mode: 0 = README "+1 iff WHITE wins", 1 = reference mover 1/2 (narde_env.py:134-141).
 * Returns the legal action count for this turn. */
int o_full_step(o_env *e, int d1, int d2, int action_idx, int reward_mode, float *reward,
                int32_t *done, float *obs198);

/* ---- Philox4x32-10 (counter-based dice stream shared with the CUDA path) ---- */
void o_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);
/* dice + action word for (seed, env, step): die = 1 + ((w*6)>>32) on w0,w1; out[2] = w2 */
void o_turn_dice(uint64_t seed, uint32_t env, uint64_t step, int32_t *d1, int32_t *d2,
                 uint32_t *action_word);
/* opening roll-off: returns +1 (White starts) or -1 */
int o_opening_player(uint64_t seed, uint32_t env, uint64_t step);

/* CPU baseline driver: full-rules random self-play, same dice/action stream as the CUDA path. */
int64_t o_selfplay(uint64_t seed, uint32_t env_base, int n_envs, int n_steps, uint64_t step0,
                   int64_t *sum_actions, int64_t *episodes, double *obs_checksum);

/* ---- bulk trace of full-rules self-play (parity at the benchmarked size; bench.py cpu_baseline) ----
 * State records use the boundary's data format (include/narde_b200.h:19-24), actions its u64
 * turn-action encoding (:28-29). */
void o_pack_state(const o_env *e, int terminated, int episode_steps, uint8_t *lo16, uint8_t *hi16);
void o_unpack_state(const uint8_t *lo16, const uint8_t *hi16, o_env *e, int *terminated,
                    int *episode_steps);
uint64_t o_pack_action(const o_turn_action *a);
uint64_t o_list_weight(int k);
/* Plays envs [env_base, env_base + n_envs) for turns step0+1 .. step0+n_steps the way the fused CUDA
 * step does: Philox dice, full enumeration, action choice (words == NULL: the turn's Philox word as
 * a fraction of the list; word_mode 0: words[t][i] is a clamped index, 1: a u32 fraction), apply,
 * termination / reward (reward_mode as o_full_step), TimeLimit truncation, optional auto-reset.
 * init_lo/init_hi: packed start states, NULL = fresh games whose roll-off is taken at step0.
 * Every out_* array (each may be NULL) is [n_steps][row_stride]; row (t-1, i) describes env i after
 * turn step0+t: packed state, chosen action, legal-action count, dice, done bits (1 terminated,
 * 2 truncated), reward, checksum of the first min(count, cap) list entries.  stats8 = the counters
 * of include/narde_b200.h:62-71 over this call; obs_checksum (may be NULL): the Box(198) row of every env turn is
 * computed (o_obs198) and summed into it.  Returns the number of env turns played. */
int64_t o_selfplay_trace(uint64_t seed, uint32_t env_base, int n_envs, int n_steps, uint64_t step0,
                         const uint8_t *init_lo, const uint8_t *init_hi, const uint32_t *words,
                         int64_t words_stride, int word_mode, int cap, int reward_mode, int autoreset,
                         int max_episode_steps, int64_t row_stride, uint8_t *out_lo, uint8_t *out_hi,
                         int64_t *out_chosen, int32_t *out_count, uint8_t *out_dice, uint8_t *out_done,
                         float *out_reward, uint64_t *out_hash, int64_t *stats8, double *obs_checksum);
/* get_valid_actions for n packed positions: count + checksum of the first min(count, cap) list entries */
void o_enumerate_batch(const uint8_t *lo, const uint8_t *hi, const uint8_t *dice, int64_t n, int cap,
                       int32_t *out_count, uint64_t *out_hash);
/* narde_afterstates_scan's rows for n packed positions: legal-action count, and for each of the first min(count, cap)
 * canonical actions its u64 word ([n][cap]) and the packed state after it and the end of the turn ([n][cap] x 16 bytes
 * per plane; the state o_full_step leaves, terminated bit and episode steps as narde_afterstates_scan writes them). */
void o_afterstates_batch(const uint8_t *lo, const uint8_t *hi, const uint8_t *dice, int64_t n, int cap,
                         int32_t *counts_out, uint64_t *actions_out, uint8_t *as_lo_out, uint8_t *as_hi_out);

#ifdef __cplusplus
}
#endif
#endif
