/* colosseum_b200_learner.h -- one learner seat against device-side random opponents, for the turn-based games of
 * libcolosseum_b200.so (included by colosseum_b200.h; the same conventions: device pointers, the caller's stream,
 * 0 = OK, crl_last_error() on failure).
 *
 * An *advance* is one launch per learner move: it applies the learner's move and plays the other seats, each on the
 * uniform random policy, until the learner is to move again.  The reference has no single-player wrapper for these
 * games, so the rule is THIS ENGINE'S DEFINITION, pinned by a C oracle (tests/oracle_learner.c).  P is the number of
 * players (Tic Tac Toe: n; Blokus: 4).  For game e, learner seat `seat` and step counter t:
 *   1. A stored game that is terminal is replaced by new_state().  It is not reported: it ended in an earlier call.
 *   2. If actions != NULL and the mover is `seat`, actions[e] is applied exactly as crl_ttt_step / crl_blokus_step
 *      apply it (an illegal action is flagged and applied as a pass; -1 is a pass).  Otherwise the learner does not
 *      move (flag 8).
 *   3. j = 0.  While the game is terminal or its mover is not `seat`:
 *        terminal: it is the finished game of this call; it is restarted (new_state()).
 *        else: opponent move j.  w = philox(seed, first_env + e, t, tag 6 + (j >> 2))[j & 3]; the move is the
 *        (w % m)-th valid action of the mover in the reference's order, m = the number of valid actions (Tic Tac Toe:
 *        the k-th empty cell in C order; Blokus: the k-th id of the mover's full list, drawn as crl_blokus_rollout
 *        draws it, without the list in memory; a mover known to have no move passes).  m == 0: a pass.  j++.
 * No game can end within its first P - 1 moves (a Tic Tac Toe line needs 5, 7 or 9 moves; every Blokus colour has a
 * move in round 0), so a call finishes at most one game and makes at most 2P - 2 opponent moves.  On return every game
 * is non-terminal and its mover is `seat`.  A Blokus learner without a move is still handed its turn: its list from
 * crl_blokus_legal(player = seat) is empty and it passes with -1, as the reference's agent answers ''.
 *
 * Learner reward (0 unless the call finished a game): Tic Tac Toe +1 if `seat` won, -1 if another seat won, 0 for a
 * full board (current_rewards); Blokus the learner's index in the stable ascending sort of the final scores,
 * #{q : sc[q] < sc[seat] or (sc[q] == sc[seat] and q < seat)} (the step's reward when the learner moves last).
 * Record per game: int8 reward | u8 flags (1 a game finished, 2 the learner's action was illegal, 4 the learner
 * placed, 8 the learner did not move) | u8 winners mask of the finished game (0 if none) | u8 opponent moves played.
 * Tic Tac Toe: 4 bytes; Blokus: 8 bytes, the same 4 and then the finished game's scores of seats 0..3 (u8 each), else 0.
 * Statistics (may be NULL): every env-step, the learner's and the opponents', adds the slots crl_ttt_step /
 * crl_blokus_step add; a Blokus opponent move also adds its m to CRL_ST_NVALID, as crl_blokus_rollout does.
 */
#ifndef COLOSSEUM_B200_LEARNER_H
#define COLOSSEUM_B200_LEARNER_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Tic Tac Toe advance, in place on state (16-byte aligned).  actions_or_null: int8[B] cells of the learner (NULL: the
 * learner does not move); result: uint32[B] records (4-byte aligned); valid_after_or_null: uint32[B] empty-cell masks
 * of the returned games, i.e. the learner's valid actions (4-byte aligned).
 * CRL_ERR_UNSUPPORTED: n not in {2, 3, 4}, B >= 2^31.  CRL_ERR_ARG: null state or result, B < 0, seat outside [0, n),
 * a misaligned state, result or valid_after buffer.  B == 0: no-op. */
int crl_ttt_advance(void *state, const int8_t *actions_or_null, int seat, uint8_t *result,
                    uint32_t *valid_after_or_null, int64_t *stats_or_null, uint64_t seed, uint64_t first_env,
                    uint32_t step, int64_t B, int n, crl_stream_t stream);

/* Blokus advance, in place on state (16-byte aligned).  actions_or_null: int32[B] action ids of the learner (4-byte
 * aligned; NULL: the learner does not move); result: uint8[B][8] records (8-byte aligned).
 * CRL_ERR_ARG: null state or result, B < 0, seat outside [0, 4), a misaligned state, result or actions buffer.
 * B == 0: no-op. */
int crl_blokus_advance(void *state, const int32_t *actions_or_null, int seat, uint8_t *result,
                       int64_t *stats_or_null, uint64_t seed, uint64_t first_env, uint32_t step, int64_t B,
                       crl_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif
