/* colosseum_b200.h -- C ABI of libcolosseum_b200.so: batched, bit-packed, B200-native (sm_100a) game
 * dynamics for ColosseumRL's Tron, Blokus and 2/3/4-player Tic Tac Toe.
 *
 * The reference has no FFI for this path: its boundary is the Python ABC `BaseEnvironment`
 * (colosseumrl/BaseEnvironment.py:10-283) plus one Cython entry point
 * (`next_state_inplace`, colosseumrl/envs/tron/CyTronGrid.pyx:3-7).  Each entry point below names the
 * reference function(s) it replaces; INTEGRATION.md shows the ctypes binding a maintainer adds.
 *
 * Conventions
 *  - every `state`, `actions`, `result`, `stats`, ... pointer is a DEVICE pointer into caller-owned memory
 *    (e.g. torch.Tensor.data_ptr()); the library never allocates, frees or retains them;
 *  - kernels are enqueued on `stream` (a cudaStream_t passed as void*) and never synchronise;
 *  - return value 0 = OK, non-zero = error (crl_last_error() gives a thread-local message);
 *  - per-environment data errors (illegal action id) never fail the call: they set the error bit of that
 *    environment's result record and are applied as a pass / no-op (match_server.py:192-198 behaviour);
 *  - B = number of environments in the batch; all per-environment arrays are dense over [0, B).
 *  - there is NO CPU fallback: without a CUDA device every compute entry point returns CRL_ERR_CUDA.
 */
#ifndef COLOSSEUM_B200_H
#define COLOSSEUM_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CRL_OK 0
#define CRL_ERR_ARG 1
#define CRL_ERR_CUDA 2
#define CRL_ERR_UNSUPPORTED 3

#define CRL_PLAYER_ABSOLUTE (-1) /* observe: plain unpack, no perspective transform */
#define CRL_PLAYER_MOVER (-2)    /* observe (Blokus, Tic Tac Toe): each game from the perspective of its current mover */
#define CRL_PLAYER_ALL (-3)      /* observe (Tron): the views of all players at once */

#define CRL_FLAG_AUTO_RESET 1 /* an environment whose stored terminal flag is set is replaced by new_state() before the step */
#define CRL_FLAG_COMPACT_RESULT 2 /* crl_tron_step: write the 4-byte record (below) instead of the 8-byte one;
                                     crl_ttt_step: write the 1-byte record (below) instead of the 4-byte one */
#define CRL_FLAG_COMPACT2_RESULT 8 /* crl_tron_step only: write the 2-byte record (below) */
#define CRL_FLAG_PACKED_ACTIONS 4 /* crl_tron_step only: actions are uint8[B], 2 bits per player (action & 3) */

/* statistics buffer: int64[CRL_STAT_ROWS][CRL_NSTAT] on the device, accumulated (+=) by step / rollout kernels.
 * CTAs spread their partial sums over the rows so that same-address L2 atomics do not serialise; the value of
 * slot s is the sum over rows of stats[row][s]. */
#define CRL_NSTAT 32
#define CRL_STAT_ROWS 256
#define CRL_ST_STEPS 0     /* env-steps                                   */
#define CRL_ST_EPISODES 1  /* finished episodes (terminal transitions)    */
#define CRL_ST_EPLEN 2     /* sum of finished-episode lengths             */
#define CRL_ST_WINS 3      /* [3..6]  wins per seat                       */
#define CRL_ST_NOWIN 7     /* finished episodes without a winner          */
#define CRL_ST_SCORE 8     /* [8..11] sum of final scores per seat        */
#define CRL_ST_ERRORS 12   /* illegal actions                             */
#define CRL_ST_NVALID 13   /* sum of valid-action counts                  */
#define CRL_ST_RANK 14     /* [14..17] sum of final ranks per seat        */
#define CRL_ST_REWARD 18   /* sum over steps of sum_p (p+1) * reward_p    */

typedef void *crl_stream_t; /* cudaStream_t */

int crl_version(void);
const char *crl_last_error(void);
/* Select + validate the device (compute capability 10.x required). Idempotent. */
int crl_init(int device);

/* Philox4x32-10 words for environments [first_env, first_env+B) at `step`: out = uint32[B][4].
 * counter = (env_lo, env_hi, step, tag), key = (seed_lo, seed_hi). */
int crl_philox_words(uint32_t *out, uint64_t seed, uint64_t first_env, uint32_t step, uint32_t tag, int64_t B,
                     crl_stream_t stream);

/* Reader side of the statistics buffer: out[s] = sum over the CRL_STAT_ROWS rows of stats_rows[r][s]
 * (out = int64[CRL_NSTAT] on the device; accumulate != 0: out[s] += ...).  One tiny launch; the 32-slot vector is what a
 * multi-GPU job all-reduces (NCCL) once per measurement window -- the engine's only collective (SURVEY.md section 8e;
 * the reference has no counterpart: its statistics are Python-side counters in the callers' loops). */
int crl_stats_reduce(const int64_t *stats_rows, int64_t *out, int accumulate, crl_stream_t stream);

/* HOST helpers for actors whose policy runs on the host (match_server.py:201-218: actions arrive on the host, results
 * go back to it): launch a captured step graph (cudaGraphExec_t) on `stream` and record `done_event` (cudaEvent_t, may
 * be NULL) behind it in ONE foreign call; block until an event has completed.  CRL_ERR_ARG = the calling thread's
 * current device does not own the handles (nothing was launched; retry under a device guard). */
int crl_host_graph_launch(void *graph_exec, crl_stream_t stream, void *done_event_or_null);
/* the pipelined actor's whole step in one foreign call: launch this batch's step, then block until `wait_event` (the
 * completion event of the OLDEST batch in flight, may be NULL) has completed */
int crl_host_graph_launch_wait(void *graph_exec, crl_stream_t stream, void *done_event_or_null, void *wait_event_or_null);
int crl_host_event_wait(void *event);

/* ------------------------------------------------------------------------------------------- Tron
 * Any shape the reference's config string can name within 5 <= N <= 64, 2 <= P <= 8 (TronGridEnvironment.py:28-58;
 * CyTronGrid.pyx:8-9 takes N and P from the array shapes).  Two state layouts, chosen by the shape alone:
 *  - N <= 19 and P <= 4 (BASELINE.json's 19x19 4-player and everything near it): the tuned path.  Packed state 208 bytes
 *    per environment, SoA [13][B] of 16-byte vectors, of which a step moves 160 (three owner-code bit-planes and the
 *    header; vectors 9..11 are reserved and zero) (csrc/tron.cuh); actions int8[B][4]; result 8 bytes.  Everything
 *    below describes this path.
 *  - every other shape: the "wide" path (csrc/tron_wide.cuh), same entry points and semantics.  Packed state uint32
 *    [W][B], W = P * ceil(N*N/32) + 2P + 1 (crl_tron_state_bytes tells); actions int8[B][8]; result 16 bytes per
 *    environment = int8 reward[8] | u8 terminal | u8 alive mask | u8 winners mask | u8 0 | u32 ranking (3 bits per
 *    player); crl_tron_ranking writes uint32[B] (3 bits per player); the compact-record / packed-action flags are not
 *    available; the per-seat statistics slots cover seats 0..3.  crl_tron_action_stride / crl_tron_result_bytes return
 *    4 / 8 or 8 / 16 so that callers can size their buffers without knowing the rule.
 * actions: int8[B][4]  (0 forward, +1 right, -1 left; TronGridEnvironment.STRING_TO_ACTION :62-67),
 *          entries of dead / absent players are ignored.  With CRL_FLAG_PACKED_ACTIONS: uint8[B], player p's
 *          action in bits 2p..2p+1 as (action & 3), i.e. 0 forward, 1 right, 3 left -- a quarter of the PCIe bytes.
 * result:  8 bytes per environment: int8 reward[4] | u8 terminal | u8 alive mask | u8 winners mask |
 *          u8 ranking (2 bits per player, competition ranking of compute_ranking).
 *          With CRL_FLAG_COMPACT_RESULT: 4 bytes per environment = the second half of that record (terminal | alive |
 *          winners | ranking).  The rewards follow from it exactly as the reference computes them
 *          (TronGridEnvironment.py:313-320): reward[p] = alive[p] ? 1 : -1, plus 9 for the winners of a terminal step.
 *          It halves what a host-side actor has to read back over PCIe per step.
 *          With CRL_FLAG_COMPACT2_RESULT: 2 bytes per environment, byte 0 = alive mask | terminal << 4, byte 1 =
 *          ranking.  Nothing is lost: the winners of a terminal step ARE its alive players (:316-319) and the rewards
 *          follow as above; the device -> host read of a host-side actor (the slowest leg of its step) halves again. */
int64_t crl_tron_state_bytes(int N, int P, int64_t B);
/* HOST functions: int8 actions per environment (4 or 8) and bytes of a result record (8 or 16) for this shape; -1 if
 * the shape is unsupported.  (The reference's counterpart is the length P of its per-player lists.) */
int crl_tron_action_stride(int N, int P);
int crl_tron_result_bytes(int N, int P);
/* HOST function. generate_start_positions (TronGridEnvironment.py:183-226) with new_state's defaults:
 * heads[p] = y*N + x, directions[p] in {0 N, 1 E, 2 S, 3 W}. */
int crl_tron_start_positions(int N, int P, int32_t *heads, int32_t *directions);
/* new_state (TronGridEnvironment.py:228-263) for every environment, or where mask[e] != 0 */
int crl_tron_reset(void *state, const uint8_t *mask_or_null, int64_t B, int N, int P, crl_stream_t stream);
/* The same two with new_state's optional arguments (TronGridEnvironment.py:228: ring_offset = how far in from the wall
 * the spawn ring lies, spawn_offset = shift of every spawn along its arc; the defaults are 1 and 2).  An integer
 * spawn_offset is deterministic in the reference (:222-224: randint(o, o + 1) == o for every player).
 * CRL_ERR_ARG if the ring is degenerate for this N / P. */
int crl_tron_start_positions_at(int N, int P, int ring_offset, int spawn_offset, int32_t *heads, int32_t *directions);
int crl_tron_reset_at(void *state, const uint8_t *mask_or_null, int64_t B, int N, int P, int ring_offset, int spawn_offset,
                      crl_stream_t stream);
/* ... and with ONE OFFSET PER PLAYER, the reference's (lo, hi) tuple form: generate_start_positions draws
 * `offsets = [np.random.randint(lo, hi) for _ in range(num_players)]` (:222-224) and uses offsets[p] for player p's
 * head and direction.  spawn_offsets = int32[P] on the HOST (the draw is the caller's: numpy's global RNG seeded from
 * the wall clock, :255, is not reproducible by design).  crl_tron_step_spawns is crl_tron_step whose auto-reset
 * (CRL_FLAG_AUTO_RESET) restarts finished games from THESE spawns instead of the default new_state(). */
int crl_tron_start_positions_spawns(int N, int P, int ring_offset, const int32_t *spawn_offsets, int32_t *heads,
                                    int32_t *directions);
int crl_tron_reset_spawns(void *state, const uint8_t *mask_or_null, int64_t B, int N, int P, int ring_offset,
                          const int32_t *spawn_offsets, crl_stream_t stream);
int crl_tron_step_spawns(const void *state_in, void *state_out, const int8_t *actions, uint8_t *result, int64_t *stats,
                         int64_t B, int N, int P, int flags, int ring_offset, const int32_t *spawn_offsets,
                         crl_stream_t stream);
/* next_state (TronGridEnvironment.py:265-323 -> CyTronGrid.pyx:3-62) + compute_ranking (:483-508).
 * state_out may equal state_in (in place). stats may be NULL. */
int crl_tron_step(const void *state_in, void *state_out, const int8_t *actions, uint8_t *result,
                  int64_t *stats_or_null, int64_t B, int N, int P, int flags, crl_stream_t stream);
/* uniform random policy: action of player p = {0,+1,-1}[philox(env, step, tag 1)[p] % 3] */
int crl_tron_policy_random(int8_t *actions, uint64_t seed, uint64_t first_env, uint32_t step, int64_t B,
                           crl_stream_t stream);
/* the same policy for the wide layout: actions int8[B][8]; players 4..7 use {0,+1,-1}[(philox(...)[p - 4] / 3) % 3]
 * (one Philox call per environment and step) */
int crl_tron_policy_random_wide(int8_t *actions, uint64_t seed, uint64_t first_env, uint32_t step, int64_t B,
                                crl_stream_t stream);
/* K fused random-policy steps with auto-reset, state kept in registers (identical to K x policy+step) */
int crl_tron_rollout(void *state, uint8_t *result_or_null, int64_t *stats_or_null, uint64_t seed,
                     uint64_t first_env, uint32_t step0, int K, int64_t B, int N, int P, crl_stream_t stream);
/* state_to_observation (TronGridEnvironment.py:363-405, CyTronGrid.pyx:65-71). player = CRL_PLAYER_ABSOLUTE: plain
 * unpack; player = CRL_PLAYER_ALL: the views of all P players in one pass (nview = P, else nview = 1).
 * board int8[B][nview][N][N]; heads (y*N+x) / directions / deaths int32[B][nview][P] (may be NULL); terminal u8[B]
 * (may be NULL) */
int crl_tron_observe(const void *state, int player, int8_t *board, int32_t *heads, int32_t *directions,
                     int32_t *deaths, uint8_t *terminal_or_null, int64_t B, int N, int P, crl_stream_t stream);
/* compute_ranking (TronGridEnvironment.py:483-508) of any state, without stepping it: ranking u8[B], 2 bits per
 * player (the same value crl_tron_step writes into result byte 7) */
int crl_tron_ranking(const void *state, uint8_t *ranking, int64_t B, int N, int P, crl_stream_t stream);
/* import a reference-layout state */
int crl_tron_pack(void *state, const int8_t *board, const int32_t *heads, const int32_t *directions,
                  const int32_t *deaths, int64_t B, int N, int P, crl_stream_t stream);

/* ------------------------------------------------------------------------------------ Tic Tac Toe
 * n = 2 (3x3), 3 (3x5), 4 (3x3x3).  Packed state: 16 bytes per environment, uint4[B] (csrc/ttt.cuh).
 * actions: int8[B], C-order flat cell index, negative = '' (pass).
 * result:  4 bytes per environment: int8 reward (mover's) | u8 flags (1 terminal, 2 invalid action, 4 placed) |
 *          u8 winners mask | u8 ranking bits (bit p = rank of p: winners 0, others 1).
 *          crl_ttt_step with CRL_FLAG_COMPACT_RESULT: ONE byte per environment = flags (bits 0..2, as above) |
 *          (winner + 1) << 3 (0 = None) | the player who moved << 6.  Nothing is lost: the mover's reward is +1 if it is
 *          the winner, -1 if somebody else is, else 0 (tictactoe_2p_env.py:302-308); winners mask and ranking follow from
 *          the winner; a quarter of the bytes a host-side actor reads back per step.                          */
int crl_ttt_cells(int n);                                                     /* HOST: 9 / 15 / 27 */
/* HOST: the winning lines as cell masks (cross-check of WINNING_SHAPES, tictactoe_4p_env.py:19-38); returns count */
int crl_ttt_lines(int n, uint32_t *line_masks_or_null, int capacity);
/* new_state (tictactoe_2p_env.py:139-170) */
int crl_ttt_reset(void *state, const uint8_t *mask_or_null, int64_t B, int n, crl_stream_t stream);
/* next_state (2p :240-315, 3p :241-316, 4p :271-346). valid_after (uint32[B], may be NULL) receives the
 * empty-cell mask of the NEW state (= valid_actions of the next mover). */
int crl_ttt_step(const void *state_in, void *state_out, const int8_t *actions, uint8_t *result,
                 uint32_t *valid_after_or_null, int64_t *stats_or_null, int64_t B, int n, int flags,
                 crl_stream_t stream);
/* valid_actions (2p :317-348): bit c = cell c empty; 0 <=> [''] */
int crl_ttt_valid_actions(const void *state, uint32_t *mask, int64_t B, int n, crl_stream_t stream);
/* uniform random policy: the (philox(env, step, tag 3)[0] % n_empty)-th empty cell, -1 if none.  With
 * CRL_FLAG_AUTO_RESET a finished game is treated as the fresh board the step will reset it to. */
int crl_ttt_policy_random(const void *state, int8_t *actions, uint64_t seed, uint64_t first_env, uint32_t step,
                          int64_t B, int n, int flags, crl_stream_t stream);
int crl_ttt_rollout(void *state, uint8_t *result_or_null, int64_t *stats_or_null, uint64_t seed, uint64_t first_env,
                    uint32_t step0, int K, int64_t B, int n, crl_stream_t stream);
/* state_to_observation (2p :382-407; 4p relabels with % 3, tictactoe_4p_env.py:50). player < 0: absolute.
 * board int8[B][cells] (-1 empty); winner int8[B] (-1 None) and mover int8[B] may be NULL. */
int crl_ttt_observe(const void *state, int player, int8_t *board, int8_t *winner_or_null, int8_t *mover_or_null,
                    int64_t B, int n, crl_stream_t stream);
int crl_ttt_pack(void *state, const int8_t *board, const int8_t *winner, const int8_t *mover, int64_t B, int n,
                 crl_stream_t stream);

/* ------------------------------------------------------------------------------------------ Blokus
 * 4 players, 20x20.  Packed state: 352 bytes per game, AoS uint4[B][22] (csrc/blokus.cuh).
 * Action id = ((piece*400 + y*20 + x)*8 + orientation)*5 + shift  for the reference's action string
 * "{piece};({x}, {y});{orientation}{shift}" (BlokusEnvironment.py:55-106; piece in PIECE_TYPES order, board.py:24-44;
 * orientation in ORIENTATIONS order, board.py:47); -1 = '' (pass).
 * result: 8 bytes per game: int8 reward (mover's) | u8 flags (1 terminal, 2 illegal action, 4 placed) |
 *         u8 winners mask | u8 ranking bits (bit p = rank of p: winners 0, others 1) | u8 next mover |
 *         u8 next-players mask (1 << next mover) | u8 terminal (0 / 1) | 1 unused.  */
int64_t crl_blokus_state_bytes(int64_t B);
/* new_state (BlokusEnvironment.py:248-289) */
int crl_blokus_reset(void *state, const uint8_t *mask_or_null, int64_t B, crl_stream_t stream);
/* valid_actions (BlokusEnvironment.py:453-500 -> board.py:170-193 -> computation.py:145-180) for `player`
 * (player < 0: each game's current mover).  counts int32[B] receives the full list length; action_ids
 * int32[B][capacity] the ids in the reference's order (truncated at capacity; counts[g] > capacity signals it).
 * counts[g] == 0 <=> [''].  With CRL_FLAG_AUTO_RESET a finished game is treated as the fresh game the step will
 * reset it to.  stats (optional): CRL_ST_NVALID += counts. */
int crl_blokus_legal(const void *state, int player, int32_t *counts, int32_t *action_ids, int32_t capacity,
                     int64_t *stats_or_null, int64_t B, int flags, crl_stream_t stream);
/* is_valid_action (BlokusEnvironment.py:667-719) for `player` (< 0: each game's current mover): valid[g] = 1 iff
 * actions[g] is in that player's valid list (the pass id -1 is not), without enumerating the list. */
int crl_blokus_is_valid(const void *state, int player, const int32_t *actions, uint8_t *valid, int64_t B, int flags,
                        crl_stream_t stream);
/* next_state (BlokusEnvironment.py:357-451): apply (board.py:87-98, ai.py:44-54), the lagged terminal test
 * (:424: old board, old round, new inventories), winners / reward (:425-440), round / mover advance (:446-449).
 * Unlike the reference (which applies any string blindly) an id that is not in the mover's valid list sets the
 * illegal-action flag and is applied as a pass. */
int crl_blokus_step(const void *state_in, void *state_out, const int32_t *actions, uint8_t *result,
                    int64_t *stats_or_null, int64_t B, int flags, crl_stream_t stream);
/* uniform random policy over a generated list: ids[g][philox(env, step, tag 2)[0] % counts[g]], -1 if empty */
int crl_blokus_policy_random(const int32_t *counts, const int32_t *action_ids, int32_t capacity, int32_t *actions,
                             uint64_t seed, uint64_t first_env, uint32_t step, int64_t B, crl_stream_t stream);
/* K fused random-policy steps with auto-reset: identical to K x (crl_blokus_legal(player -1, CRL_FLAG_AUTO_RESET)
 * -> crl_blokus_policy_random(step0 + t) -> crl_blokus_step(CRL_FLAG_AUTO_RESET)) whenever every list fits the
 * capacity of that sequence.  No list is materialised: the pick is ids[philox(env, step0 + t, tag 2)[0] % n] over the
 * FULL list of length n, so the trajectories equal the oracle's (oracle_rollout.c) for any list length, and the
 * three-launch sequence's only while counts <= its capacity (it draws from the stored prefix otherwise).
 * result (may be NULL): the 8-byte record of the last step.  stats (may be NULL): the same slots the three launches add
 * (CRL_ST_NVALID included), counted per game in 64 bits, so any K is accepted.  B == 0 or K == 0: no-op. */
int crl_blokus_rollout(void *state, uint8_t *result_or_null, int64_t *stats_or_null, uint64_t seed,
                       uint64_t first_env, uint32_t step0, int K, int64_t B, crl_stream_t stream);
/* a host-side policy's choice (the agent of match_server.py:201-218 answers with one of the strings valid_actions gave
 * it): actions[g] = action_ids[g][choice[g]], -1 (pass) if choice[g] < 0 or >= counts[g].  The policy only needs the list
 * lengths on the host; the lists stay on the device. */
int crl_blokus_pick(const int32_t *counts, const int32_t *action_ids, int32_t capacity, const int32_t *choice,
                    int32_t *actions, int64_t B, crl_stream_t stream);
/* state_to_observation (BlokusEnvironment.py:721-768).  player >= 0: board int8[B][20][20] of relative ids (-1
 * empty) rotated by rot90(k=-player), pieces u8[B][4][21] by relative id, score int32[B][4] rolled by -player.
 * player < 0: absolute unpack (board 0 empty / 1..4 colour).  meta int32[B][4] (may be NULL) = round, mover,
 * terminal, episode steps. */
int crl_blokus_observe(const void *state, int player, int8_t *board, uint8_t *pieces, int32_t *score,
                       int32_t *meta_or_null, int64_t B, crl_stream_t stream);
int crl_blokus_pack(void *state, const int8_t *board, const uint8_t *pieces, const int32_t *score, const int32_t *meta,
                    int64_t B, crl_stream_t stream);

#ifdef __cplusplus
}
#endif

/* device-side Tron opponents (the avoid policy and its fused rollout) */
#include "colosseum_b200_tron_policy.h"
/* one learner seat against device-side random opponents (Tic Tac Toe, Blokus) */
#include "colosseum_b200_learner.h"
/* Blokus placements: a fixed action space with legality masks, and placement -> action id */
#include "colosseum_b200_placement.h"
#endif
