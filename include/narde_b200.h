/*
 * narde_b200.h -- C ABI of the B200-native batched Narde environment path.
 *
 * Drop-in boundary for the reference's rules engine + env step
 * (/root/reference/gym_narde/envs/narde.py, narde_env.py; SURVEY.md section 8b).  The reference
 * is pure Python with no FFI; the binding a maintainer would add is the ctypes stub shown in
 * INTEGRATION.md (the product's own host side, gym_narde_b200/_cabi.py, is exactly that stub).
 *
 * Conventions
 *   - every function returns 0 on success or a cudaError_t value (> 0) / -1 for bad arguments;
 *     nothing is thrown across the ABI;
 *   - every pointer is a DEVICE pointer owned by the caller (PyTorch allocates); the library
 *     allocates nothing and keeps no state;
 *   - work is enqueued asynchronously on `stream` (a cudaStream_t passed as void*; NULL = the
 *     legacy default stream);
 *   - n = number of environments in this shard; env_base = global id of the shard's first
 *     environment (multi-GPU sharding: rank r owns [env_base, env_base + n)).
 *
 * State record (two SoA planes of 16-byte lanes, one lane per environment per plane):
 *   lo[i] : int8 point counts 0..15            absolute (White) frame, +white / -black
 *   hi[i] : int8 point counts 16..23 | u8 off_white | u8 off_black | i8 turn (+1 White, -1 Black)
 *           | u8 flags (1 first_turn_white, 2 first_turn_black, 4 terminated)
 *           | u16 episode_steps | u16 reserved
 *   (replaces Narde.board/borne_off_* / first_turn_* , narde.py:21-29, + NardeEnv.current_player)
 *
 * Half-move encoding  : u8 from, u8 to (255 = bear off) in the MOVER's frame, as
 *                       Narde.get_valid_moves returns them (narde.py:58-92).
 * Turn-action encoding: u64 = 4 x u16 half-moves (from | to << 8), slot 0 played first,
 *                       0xFFFF = unused slot.
 */
#ifndef NARDE_B200_H
#define NARDE_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NARDE_ABI_VERSION 4
#define NARDE_MAX_HALF_MOVES 96 /* 4 dice x 24 points */
/* int32 words of the optional `workspace` of narde_step_full / narde_enumerate_fast for n environments (the caller
 * zero-fills it once): header [0] number of deferred envs of the call (cleared again by a NARDE_DEVICE_ADVANCE call),
 * [1] arrival counter of the exact kernel's CTAs, [2] arrival counter of the main kernel's CTAs (release/acquire
 * publication of the list to the programmatic dependent), [3] number of deferred envs of the last completed
 * NARDE_DEVICE_ADVANCE call, [4..7] reserved; [8..n+7] the list of deferred env indices */
#define NARDE_WORKSPACE_HEADER 8
#define NARDE_WORKSPACE_INTS(n) ((n) + NARDE_WORKSPACE_HEADER)

/* narde_step_full flags */
#define NARDE_REWARD_MOVER12 1   /* reward 1/2 to the mover (narde_env.py:134-141); default: README +1 iff WHITE wins */
#define NARDE_AUTORESET 2        /* reset a finished environment in the same step (obs = first obs of the new game) */
#define NARDE_PER_THREAD_KERNEL 8 /* narde_step_full: use the thread-per-env kernel (A/B testing; same results) */
#define NARDE_ACTION_FRACTION 32  /* narde_step_full: action_idx[i] is a u32 fraction f; plays action floor(f * count / 2^32) */
#define NARDE_ENUMERATE_ONLY 64   /* narde_step_full: write actions / counts (/ chosen) only, leave every state untouched;
                                    done[i] then receives the overflow flag (count > cap) */
#define NARDE_PACK_RESULT 128     /* narde_step_full (CTA-cooperative kernels): done[i] receives one packed byte per env -- bit 0
                                    terminated, bit 1 truncated, bits 2-3 the reward (0, 1 or 2); reward[] and truncated[] are
                                    not written.  One byte instead of six per env for a host-resident consumer. */
#define NARDE_DEVICE_ADVANCE 256   /* narde_step_full with workspace and step_dev: the step index is *step_dev + 1, and the kernels
                                    themselves store it back and clear the workspace when the step is complete -- no memset and no
                                    counter kernel in front of every step (two nodes of a replayed CUDA graph, ~2 us each).  The
                                    workspace's three counters are zero before the first call and are left zero by every call;
                                    it must not be shared with calls that do not set this flag. */
#define NARDE_HALF_MOVES_ONLY 4  /* narde_apply_actions: Narde.execute_rotated_move semantics (no end-of-turn bookkeeping) */

/* done[i] = 1 when the episode terminated (a player bore off 15 checkers); truncated[i] = 1 when
 * max_episode_steps was reached without termination (gymnasium TimeLimit semantics). */

/* stats[] slots (int64, accumulated with atomics; caller zeroes) */
#define NARDE_STAT_EPISODES 0
#define NARDE_STAT_WHITE_WINS 1
#define NARDE_STAT_BLACK_WINS 2
#define NARDE_STAT_MARS 3
#define NARDE_STAT_EPISODE_STEPS 4 /* sum of lengths of finished episodes */
#define NARDE_STAT_LEGAL_ACTIONS 5 /* sum of legal turn actions over all stepped envs */
#define NARDE_STAT_MAX_ACTIONS 6
#define NARDE_STAT_OVERFLOWS 7
#define NARDE_STAT_CLAMPED_ACTIONS 8 /* env turns whose caller-given action index was out of range and got clamped */
#define NARDE_NUM_STATS 9

int narde_abi_version(void);

/* Which device the library was built for ("sm_100a") and a launch-free self check. */
const char *narde_build_arch(void);

/* NardeEnv.reset (narde_env.py:105-120) for n environments: fresh Narde() (narde.py:21-29) and
 * the opening roll-off, dice from Philox4x32-10(key = seed, ctr = (env, step, 1 + attempt<<8)). */
int narde_reset(void *lo, void *hi, int64_t n, int64_t env_base, uint64_t seed, uint64_t step,
                void *stream);

/* Same, but only environments with mask[i] != 0 are reset (mask may be NULL = all). */
int narde_reset_masked(void *lo, void *hi, const uint8_t *mask, int64_t n, int64_t env_base,
                       uint64_t seed, uint64_t step, void *stream);

/* Narde.get_valid_moves(roll, current_player) (narde.py:58-92) for the player to move of each
 * environment.  dice: [n,4] u8, 0-padded (1, 2 or 4 dice).  moves: [n,96,2] u8 in the
 * reference's list order (die descending, point ascending, duplicates kept, head filter applied);
 * counts: [n] i32.  player_override: 0 = use each state's turn, +1/-1 = force that perspective. */
int narde_half_moves(const void *lo, const void *hi, const uint8_t *dice, int64_t n,
                     int player_override, uint8_t *moves, int32_t *counts, void *stream);

/* NardeEnv.step(action) (narde_env.py:27-103) with the dice supplied by the caller.
 * dice: [n,2] u8 in roll order (the order matters: narde_env.py:77-83).  codes: [n,2] i32 action
 * codes from*24+to.  Outputs: obs24 [n,24] i32 (narde_env.py:24-25), reward [n] i32 (0/1/2),
 * done [n] u8 (terminated), truncated [n] u8 (may be NULL).  max_episode_steps: 0 = no TimeLimit
 * (gym_narde/__init__.py:6 registers 1000).  Terminated environments are left untouched. */
int narde_step_ref(void *lo, void *hi, const uint8_t *dice, const int32_t *codes, int64_t n,
                   int32_t max_episode_steps, int32_t *obs24, int32_t *reward, uint8_t *done,
                   uint8_t *truncated, void *stream);

/* README get_valid_actions(roll) (README.md:156-165) for every environment: all legal full-turn
 * actions (max-dice rule, higher-die rule, per-turn head rule, doubles = up to 4 half-moves),
 * de-duplicated by afterstate, in canonical order.  dice: [n,2] u8.  actions: [n,cap] u64;
 * counts[i] = true number of legal actions (may exceed cap; then overflow[i] = 1 and only the
 * first cap are stored).  overflow may be NULL. */
int narde_enumerate(const void *lo, const void *hi, const uint8_t *dice, int64_t n, int32_t cap,
                    uint64_t *actions, int32_t *counts, uint8_t *overflow, void *stream);

/* Same results as narde_enumerate through the CTA-cooperative kernels of the fused step (work items dealt
 * evenly over a 128-environment CTA, order-dependent doubles turns handed to the exact kernel when a
 * workspace of NARDE_WORKSPACE_INTS(n) int32 is given): the fast path VecNardeEnv.get_valid_actions uses. */
int narde_enumerate_fast(const void *lo, const void *hi, const uint8_t *dice, int64_t n, int32_t cap,
                         uint64_t *actions, int32_t *counts, uint8_t *overflow, int32_t *workspace,
                         void *stream);

/* One fused full-rules env step for n environments:
 *   dice (dice_in [n,2] u8, or Philox(seed, env_base+i, step) when NULL) -> legal-turn
 *   enumeration (written to actions/counts like narde_enumerate; actions may be NULL) -> action
 *   choice (action_idx[i], clamped; NULL = Philox-uniform) -> apply -> termination / reward
 *   -> player switch -> optional auto-reset -> Box(198) observation (README.md:44-102).
 * Any of actions, counts, dice_out, obs198, reward, done, truncated, chosen, stats may be NULL.
 * workspace: optional scratch of NARDE_WORKSPACE_INTS(n) int32 owned by the caller.  With it, the rare doubles
 * turns in which the 6-prime block rule makes the move ORDER matter are handed to a second,
 * CTA-per-environment kernel (a programmatic dependent launch that overlaps the tail of the main
 * kernel; same results, shorter tail); without it they are resolved inline.
 * step_dev: optional device-resident step counter that overrides `step`, so that a captured CUDA
 * graph of the step can be replayed (advance it with narde_advance_counter inside the graph). */
int narde_step_full(void *lo, void *hi, int64_t n, int64_t env_base, uint64_t seed, uint64_t step,
                    const uint8_t *dice_in, const int32_t *action_idx, int32_t cap,
                    uint64_t *actions, int32_t *counts, uint8_t *dice_out, uint64_t *chosen,
                    float *obs198, float *reward, uint8_t *done, uint8_t *truncated, int64_t *stats,
                    int32_t flags, int32_t max_episode_steps, int32_t *workspace, const uint64_t *step_dev,
                    void *stream);

/* narde_step_full with a second destination for the state planes: mirror_lo / mirror_hi ([n] 16-byte lanes, e.g.
 * pinned HOST memory) receive every environment's state after the turn as well.  For a host-side consumer the
 * 32-byte record is a lossless encoding of the Box(198) observation (README.md:44-102 is a function of board, off
 * counts and side to move): 32 B per env cross PCIe instead of 792 (gym_narde_b200.expand_obs198 decodes it). */
/* mirror_hi == NULL with mirror_lo != NULL selects the COMPACT host record instead: mirror_lo is [n] records of
 * NARDE_COMPACT_RECORD_BYTES = 20 bytes (five little-endian u32 words): bits 0..119 the 24 points, 5 bits each, two's
 * complement (+white / -black, absolute frame, point 0 first); bits 120..123 off_white, 124..127 off_black; word 4:
 * bit 0 side to move (1 = WHITE), bits 1..3 the state flags (first_w, first_b, done), bits 4..7 the turn's result
 * (terminated, truncated, reward 0..2 in two bits -- the NARDE_PACK_RESULT byte), bits 8..23 episode steps.  13 B less
 * per env across PCIe than planes + result byte: the posted writes end before the kernel does
 * (gym_narde_b200.state.unpack_compact decodes it; VecNardeEnv.step_host(obs="compact")). */
#define NARDE_COMPACT_RECORD_BYTES 20
int narde_step_full_mirror(void *lo, void *hi, int64_t n, int64_t env_base, uint64_t seed, uint64_t step,
                           const uint8_t *dice_in, const int32_t *action_idx, int32_t cap, uint64_t *actions,
                           int32_t *counts, uint8_t *dice_out, uint64_t *chosen, float *obs198, float *reward,
                           uint8_t *done, uint8_t *truncated, int64_t *stats, int32_t flags, int32_t max_episode_steps,
                           int32_t *workspace, const uint64_t *step_dev, void *mirror_lo, void *mirror_hi,
                           void *stream);

/* Observations of the current states: Box(198) float32 (README.md:44-102) / the reference's
 * mover-perspective int32[24] (narde_env.py:24-25). */
int narde_obs198(const void *lo, const void *hi, int64_t n, float *obs198, void *stream);
int narde_obs24(const void *lo, const void *hi, int64_t n, int32_t *obs24, void *stream);

/* Apply caller-chosen turn actions (from narde_enumerate) without re-enumerating: afterstate
 * transition + termination/reward/switch as in narde_step_full.  acts: [n] u64. */
int narde_apply_actions(void *lo, void *hi, const uint64_t *acts, int64_t n, int32_t flags,
                        float *reward, uint8_t *done, void *stream);

/* DecomposedDQN.forward(x) with state_size 198 (train_deepq_pytorch.py:184-236: Linear(198,256)-ReLU-
 * Linear(256,256)-ReLU-Linear(256,576)) for `rows` afterstate observations, bf16 operands and fp32
 * accumulation on the tcgen05 tensor cores.  wpack / bias: weights re-packed by
 * gym_narde_b200/mlp.py:pack_weights (K-major interleave operand stages) and the three bias vectors
 * back to back (1088 floats).
 *   narde_mlp_forward         x [rows,198] f32 (README.md:44-102 rows) -> q [rows,576] f32
 *   narde_mlp_score           x [rows,198] f32 -> score [rows] f32 = max_a q[row, a]
 *   narde_mlp_forward_states  packed states (lo/hi planes as above) -> q; the Box(198) encoding is
 *                             computed inside the kernel (32 B per row read instead of 792 B)
 *   narde_mlp_score_states    packed states -> score: the afterstate-scoring call of the actor */
int narde_mlp_forward(const float *x, int64_t rows, const void *wpack, const float *bias, float *q,
                      void *stream);
int narde_mlp_score(const float *x, int64_t rows, const void *wpack, const float *bias, float *score,
                    void *stream);
int narde_mlp_forward_states(const void *lo, const void *hi, int64_t rows, const void *wpack,
                             const float *bias, float *q, void *stream);
int narde_mlp_score_states(const void *lo, const void *hi, int64_t rows, const int64_t *rows_dev,
                           const void *wpack, const float *bias, float *score, void *stream);
/* rows_dev (may be NULL): device-resident row count, min(*rows_dev, rows) rows are scored -- lets the
 * afterstate generator and the scorer run back to back without a host synchronisation. */

/* Variants with identical results (A/B; DESIGN.md 4b): the scorer as a cta_group::2 kernel (wpack2 = weights packed for
 * it by gym_narde_b200/mlp.py:pack_weights(two_sm=True)), and a process-wide switch that runs the narde_mlp_* entries
 * above as clusters of two CTAs sharing every weight stage by multicast (also NARDE_MLP_PAIR=1 in the environment). */
int narde_mlp_score_states_2sm(const void *lo, const void *hi, int64_t rows, const int64_t *rows_dev,
                               const void *wpack2, const float *bias, float *score, void *stream);
int narde_mlp_use_cluster_pair(int on);

/* DecomposedDQN.forward(x, selected_move1) (train_deepq_pytorch.py:203-233): the Q-values of the SECOND move,
 * move2_head(cat(features, onehot(move1))).  The one-hot half of that layer is a column gather, so the kernel is
 * the same three-layer GEMM chain with wpack / bias built from the feature network and the first 256 input columns
 * of move2_head (same packing), plus w2b_t [576,576] f32 with row m = move2_head.weight[:, 256 + m], added to the
 * output row of every sample with move1 == m.  move1: [rows] i32 codes in [0,576) (clamped to that range). */
int narde_mlp_forward_move2(const float *x, int64_t rows, const int32_t *move1, const void *wpack,
                            const float *bias, const float *w2b_t, float *q2, void *stream);
int narde_mlp_forward_move2_states(const void *lo, const void *hi, int64_t rows, const int32_t *move1,
                                   const void *wpack, const float *bias, const float *w2b_t, float *q2,
                                   void *stream);

/* The afterstate of every stored legal turn action (the batched form of the enumeration loop of
 * DQNAgent.act, train_deepq_pytorch.py:430-507): row offsets[i] + k of (as_lo, as_hi) = state of
 * environment i after actions[i*cap + k] and the end-of-turn bookkeeping of narde_apply_actions, for
 * k < min(counts[i], cap).  offsets: [n] i64 exclusive prefix sums of min(counts, cap) (caller computes).
 * row_env (may be NULL): [rows] i32, the environment of each row. */
int narde_afterstates(const void *lo, const void *hi, const uint64_t *actions, const int32_t *counts,
                      const int64_t *offsets, int64_t n, int32_t cap, void *as_lo, void *as_hi,
                      int32_t *row_env, void *stream);

/* The same rows with the offsets computed on the device in the same launch (no host-side prefix sum): offsets
 * (may be NULL) receives the exclusive prefix sums of min(counts, cap), *rows_out (may be NULL) the total number of
 * rows.  scratch: NARDE_AFTERSTATE_SCRATCH_WORDS(n) u64 words, zero before the first call; every call leaves them
 * ready for the next one (calls sharing a scratch buffer must be stream-ordered).
 * rows_cap > 0 bounds the row buffers: rows at or beyond rows_cap are not written, *rows_out is clipped to it, and
 * counts_eff (may be NULL; [n] i32) receives min(counts, cap) for environments whose rows all fit and 0 otherwise. */
#define NARDE_AFTERSTATE_SCRATCH_WORDS(n) (((n) + 127) / 128 + 4)
int narde_afterstates_scan(const void *lo, const void *hi, const uint64_t *actions, const int32_t *counts,
                           int64_t n, int32_t cap, int64_t *offsets, int64_t *rows_out, void *as_lo, void *as_hi,
                           int32_t *row_env, uint64_t *scratch, int64_t rows_cap, int32_t *counts_eff, void *stream);

/* Environments whose legal list exceeds the stored capacity (overflow[i] != 0, as narde_enumerate_fast reports it) are
 * copied -- state planes, dice, env index -- into a side batch of m slots (m a multiple of 32; consecutive entries are
 * dealt to different 32-slot tiles so that the long lists spread over the CTAs), to be enumerated again with a large capacity
 * (DQNAgent.act, train_deepq_pytorch.py:430-507, looks at every legal move, not at the first `cap`).  Unused slots become
 * finished games (no legal action).  ctrl: 4 i32 words, zero before the first call: [0] overflowing envs of this call
 * (cleared by narde_scatter_choice), [2] running total of envs that did not fit into m slots.
 * narde_scatter_choice writes choice[sub_idx[s]] = sub_choice[s] (and value, if given) for the gathered slots; a slot
 * with sub_counts_eff[s] == 0 (no afterstate rows: row pool exhausted) is skipped, and it as well as a slot with
 * sub_counts[s] > cap (list longer than the side capacity) adds one to ctrl[2].  sub_actions ([m, cap] u64) and
 * act_out ([n] u64), both optional: act_out[sub_idx[s]] = the chosen action itself. */
int narde_gather_overflow(const void *lo, const void *hi, const uint8_t *dice, const uint8_t *overflow, int64_t n,
                          int32_t m, void *sub_lo, void *sub_hi, uint8_t *sub_dice, int32_t *sub_idx, int32_t *ctrl,
                          void *stream);
/* narde_gather_overflow that also zeroes act_override[i] ([n] u64, may be NULL) for every environment, so that a turn
 * starts with no override that an earlier choice left unconsumed (a narde_scatter_choice whose choice was then played by
 * narde_step_full instead of narde_step_chosen); this turn's narde_scatter_choice writes its overrides after it. */
int narde_gather_overflow_clear(const void *lo, const void *hi, const uint8_t *dice, const uint8_t *overflow, int64_t n,
                                int32_t m, void *sub_lo, void *sub_hi, uint8_t *sub_dice, int32_t *sub_idx, int32_t *ctrl,
                                uint64_t *act_override, void *stream);
int narde_scatter_choice(const int32_t *sub_choice, const float *sub_value, const int32_t *sub_idx,
                         const int32_t *sub_counts_eff, const int32_t *sub_counts, int32_t m, int32_t cap,
                         int32_t *choice, float *value, int32_t *ctrl, const uint64_t *sub_actions,
                         uint64_t *act_out, void *stream);

/* The turn of narde_step_full(action_idx = choice) when the legal lists of this very turn are already in
 * actions / counts (narde_enumerate_fast or narde_step_full(NARDE_ENUMERATE_ONLY) with the same dice): no second
 * enumeration -- env i plays actions[i*cap + clamp(choice[i])], or act_override[i] when that word is not 0 (the
 * action of an index beyond the stored capacity, as narde_scatter_choice's act_out delivers it; the word is
 * cleared again) -- then termination / reward / player switch / truncation / auto-reset / statistics / Box(198)
 * exactly as narde_step_full.  dice: [n,2] u8, the turn's dice (episode bookkeeping only).  flags:
 * NARDE_REWARD_MOVER12 | NARDE_AUTORESET.  counts, dice and the lists are not written. */
int narde_step_chosen(void *lo, void *hi, int64_t n, int64_t env_base, uint64_t seed, uint64_t step,
                      const uint8_t *dice, const int32_t *choice, const uint64_t *actions, int32_t cap,
                      const int32_t *counts, uint64_t *act_override, uint64_t *chosen, float *obs198, float *reward,
                      uint8_t *done, uint8_t *truncated, int64_t *stats, int32_t flags, int32_t max_episode_steps,
                      const uint64_t *step_dev, void *stream);

/* Greedy policy over each environment's segment of afterstate scores: idx_out[i] = argmax_k
 * score[offsets[i] + k] (mode 0), or argmin when BLACK is to move (mode 1: the net scores positions for
 * WHITE).  best_out (may be NULL): the chosen score.  Ties: lowest index; empty segment: 0. */
int narde_segment_argmax(const float *score, const int64_t *offsets, const int32_t *counts, const void *hi,
                         int64_t n, int32_t cap, int32_t mode, int32_t *idx_out, float *best_out,
                         void *stream);

/* Exploring policy over the same segments (epsilon-greedy and softmax, exact and reproducible on the host).
 * Every random word is a Philox4x32-10 word with key = seed and counter = (g, step_lo, step_hi, stream), where g is the
 * environment's global id and step the turn number its dice were rolled with (narde_roll_dice).  The low byte of
 * `stream` tells the uses apart:
 *   0             the dice (words x, y) and the environment's own uniform action (word z, narde_step_full)
 *   1 + (a << 8)  the opening roll-off, attempt a (narde_reset)
 *   2             the exploration coin (word x)
 *   3 + (k << 8)  the Gumbel noise of action k of the canonical list (word x)
 * With params = {epsilon, inv_temperature} (device float32[2], read by the kernel: a captured graph picks up new values):
 *   - environment g explores iff (coin >> 8) < floor(epsilon * 2^24) (epsilon 1: always, 0: never); it then plays
 *     k = (z * c) >> 32 over its c = min(counts[i], cap) actions, where z is word z of stream 0: exactly the uniform
 *     choice of narde_step_full when c is the whole list;
 *   - otherwise, with inv_temperature > 0, k = argmax_k (sign * score_k * inv_temperature + G_k), G_k = -log(-log(u_k)),
 *     u_k = ((w_k >> 9) + 0.5) * 2^-23 (strictly inside (0, 1) in float32): Gumbel-max, an exact sample of
 *     softmax(sign * score / temperature); sign = -1 for BLACK to move in mode 1, else +1; ties: lowest index;
 *   - otherwise the arg-max of narde_segment_argmax, bit for bit (zero parameters: the greedy choice).
 * value_out (may be NULL) receives score[offsets[i] + k] of the chosen k (0 for an empty segment).
 * env_idx (may be NULL): [n] i32, the environment of slot i (g = env_base + env_idx[i]; a side batch of
 * narde_gather_overflow); slots of -1 are skipped.  NULL: g = env_base + i.  step_dev (may be NULL) overrides `step`
 * with the device-resident turn number, as in narde_step_full.  A side batch sampled with the same rule over the whole
 * list uses the same coin and, per index k, the same noise as the main pass: narde_scatter_choice's override of the
 * main pass's choice is an exact sample over every legal action. */
int narde_segment_sample(const float *score, const int64_t *offsets, const int32_t *counts, const void *hi,
                         int64_t n, int32_t cap, int32_t mode, const int32_t *env_idx, int64_t env_base,
                         uint64_t seed, uint64_t step, const uint64_t *step_dev, const float *params,
                         int32_t *idx_out, float *value_out, void *stream);

/* Trainer-compatible action codes for every stored legal turn action: the reference's (move1_code,
 * move2_code) pairs (train_deepq_pytorch.py:432-437,495-507; action_to_idx :752-761): code = from*24 + to,
 * to = 0 for a bear-off, move2_code = 0 when the turn has a single half-move.  codes: [n,cap,3] i32 =
 * (move1_code, move2_code, number of half-moves of the turn: doubles turns may have 3 or 4, of which the
 * reference's pair space can only name the first two).  Slots k >= counts[i] are written as zeros. */
int narde_action_codes(const uint64_t *actions, const int32_t *counts, int64_t n, int32_t cap,
                       int32_t *codes, void *stream);

/* Append one 48-byte trajectory record per environment (state after the turn, action played, reward,
 * dice, done bits) to records [n] (16-byte aligned): the device-resident replay / trajectory ring
 * (the reference only checkpoints model weights, train_deepq_pytorch.py:1136-1145).  Layout:
 * lo lane | hi lane | u64 action | f32 reward | u8 die1 | u8 die2 | u8 done (1 terminated, 2 truncated) | u8 0.
 * dice, chosen, reward, done, truncated may be NULL. */
int narde_trajectory_append(const void *lo, const void *hi, const uint8_t *dice, const uint64_t *chosen,
                            const float *reward, const uint8_t *done, const uint8_t *truncated, int64_t n,
                            void *records, void *stream);

/* *counter += 1 on the device (one tiny launch); see step_dev above. */
int narde_advance_counter(uint64_t *counter, void *stream);

/* The turn's dice for every environment from the counter-based stream the fused step uses:
 * Philox4x32-10(key = seed, ctr = (env_base+i, step_lo, step_hi, 0)), die = 1 + ((w*6) >> 32) on
 * words 0 and 1 (replaces np.random.randint(1,7) x2, narde_env.py:29).  dice: [n,2] u8. */
int narde_roll_dice(int64_t n, int64_t env_base, uint64_t seed, uint64_t step, uint8_t *dice,
                    void *stream);

/* Narde._violates_block_rule(board) (narde.py:139-184) for n mover-frame boards: [n,24] int8 in,
 * [n] u8 out. */
int narde_violates_block_rule(const int8_t *boards, int64_t n, uint8_t *out, void *stream);

#ifdef __cplusplus
}
#endif
#endif
