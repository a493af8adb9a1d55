/* colosseum_b200_tron_policy.h -- device-side Tron opponents of libcolosseum_b200.so (included by colosseum_b200.h;
 * the same conventions: device pointers, the caller's stream, 0 = OK, crl_last_error() on failure).
 *
 * The avoid policy is a heuristic opponent in the shape of the reference's SimpleAvoidAgent (envs/tron/rllib.py:69-96,
 * which asks env.next_cell at :85 and :91): go forward if that cell is free, else try one side, else take the other.
 * The reference's source is not available to this project, so the exact rule is THIS ENGINE'S DEFINITION, pinned by a
 * C oracle (tests/oracle_tron_avoid.c) the way the random policy is.  For environment e, step t and seat p, decided
 * on the state BEFORE the step:
 *   w = philox(seed, first_env + e, t, tag 4 + (p >> 2))[p & 3]          (seats 0..3: tag 4, seats 4..7: tag 5)
 *   noise: if (w >> 16) < noise_q16 (0..65536), the action is {0, +1, -1}[(w & 0xFFFF) % 3]
 *   else:  forward (0) if the forward cell is free -- on the board and owned by nobody (heads are owned cells);
 *          else side s = (w & 1) ? +1 (right) : -1 (left) if that cell is free; else -s.
 *   Dead seats (deaths != 0) get 0: the step ignores them.
 */
#ifndef COLOSSEUM_B200_TRON_POLICY_H
#define COLOSSEUM_B200_TRON_POLICY_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* The avoid policy for the seats of seat_mask (bit p = seat p, bits < P), written into actions -- int8[B][4] on the
 * tuned layout (4-byte aligned), int8[B][8] on the wide one (8-byte aligned); crl_tron_action_stride tells.  The bytes
 * of the other seats are left as they are (one read-modify-write of each environment's action word), so a learner can
 * write its own seat and let the policy fill the rest, or crl_tron_policy_random fill the rest first.
 * flags: CRL_FLAG_AUTO_RESET decides a game whose stored terminal flag is set on the new_state() the step will restart
 * it from, placed with ring_offset and spawn_offsets_or_null (int32[P] on the HOST, as crl_tron_step_spawns takes
 * them; NULL = new_state's defaults, every offset 2).  Other flags are ignored.
 * CRL_ERR_ARG: null state or actions, B < 0, mask bits at or above P, noise_q16 outside 0..65536, a degenerate spawn
 * ring, a state that is not 16-byte aligned (tuned layout) or a misaligned action buffer.  B == 0: no-op. */
int crl_tron_policy_avoid(const void *state, int8_t *actions, int seat_mask, int noise_q16, uint64_t seed,
                          uint64_t first_env, uint32_t step, int64_t B, int N, int P, int flags, int ring_offset,
                          const int32_t *spawn_offsets_or_null, crl_stream_t stream);

/* K fused steps in one launch, seats of avoid_mask on the avoid policy and the others on the random policy: identical
 * to K x (crl_tron_policy_random[_wide](step0 + k) -> crl_tron_policy_avoid(avoid_mask, CRL_FLAG_AUTO_RESET) ->
 * crl_tron_step_spawns(CRL_FLAG_AUTO_RESET)), the statistics slots included, with finished games restarted from
 * ring_offset / spawn_offsets_or_null (NULL = the defaults).  With avoid_mask == 0 and the default spawns this is
 * crl_tron_rollout bit for bit.  result (may be NULL): the record of the last step; stats may be NULL.
 * CRL_ERR_ARG: null state, B < 0, K < 0, mask bits at or above P, noise_q16 outside 0..65536, a degenerate spawn ring,
 * a state that is not 16-byte aligned (tuned layout).  B == 0 or K == 0: no-op. */
int crl_tron_rollout_avoid(void *state, uint8_t *result_or_null, int64_t *stats_or_null, uint64_t seed,
                           uint64_t first_env, uint32_t step0, int K, int64_t B, int N, int P, int avoid_mask,
                           int noise_q16, int ring_offset, const int32_t *spawn_offsets_or_null, crl_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif
