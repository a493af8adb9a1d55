/* TEST INFRASTRUCTURE ONLY -- CPU oracle of the Tron avoid policy and of its mixed-policy rollout.
 *
 * Restates, independently of the CUDA source, the rule declared in include/colosseum_b200_tron_policy.h (this
 * engine's definition of an opponent in the shape of the reference's SimpleAvoidAgent, envs/tron/rllib.py:69-96),
 * on the reference's unpacked layout (oracle/oracle_tron.c), and drives oracle_tron.c's dynamics with it.  Compiled
 * together with oracle/oracle_tron.c by tests/cases_tron_avoid.py; nothing in the product path uses it.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <pthread.h>
#include <unistd.h>

#define NSTAT 32

int orc_tron_start_positions(int N, int P, int ring_offset, int spawn_offset, int64_t *heads, int64_t *directions);
int orc_tron_next_state(int N, int P, int64_t *board, int64_t *heads, int64_t *directions, int64_t *deaths,
                        const int64_t *actions, int64_t *rewards, int *alive_mask, int *winners_mask);
void orc_tron_compute_ranking(int N, int P, const int64_t *board, const int64_t *deaths, int64_t *rank);

/* Philox4x32-10 (Random123), counter = (env_lo, env_hi, t, tag), key = (seed_lo, seed_hi) */
static void philox(uint64_t seed, uint64_t env, uint32_t t, uint32_t tag, uint32_t r[4]) {
    uint32_t c0 = (uint32_t)env, c1 = (uint32_t)(env >> 32), c2 = t, c3 = tag;
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    for (int i = 0; i < 10; i++) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    r[0] = c0; r[1] = c1; r[2] = c2; r[3] = c3;
}

static const int64_t MOVE[3] = {0, 1, -1};

/* new_state with one spawn offset per player: player p's head and direction depend on its own offset only
 * (TronGridEnvironment.py:216-224), so they are the p-th entries of generate_start_positions at that offset */
int orc_tron_new_state_spawns(int N, int P, int ring_offset, const int32_t *spawn_offsets, int64_t *board,
                              int64_t *heads, int64_t *directions, int64_t *deaths) {
    int64_t h[8], d[8];
    memset(board, 0, sizeof(int64_t) * N * N);
    for (int p = 0; p < P; p++) {
        if (orc_tron_start_positions(N, P, ring_offset, spawn_offsets ? spawn_offsets[p] : 2, h, d)) return -1;
        heads[p] = h[p]; directions[p] = d[p];
    }
    for (int p = 0; p < P; p++) { deaths[p] = 0; board[heads[p]] = p + 1; }
    return 0;
}

/* a cell is free if it is on the board and nobody owns it (heads are owned cells) */
static int cell_free(int N, const int64_t *board, int64_t x, int64_t y) {
    return x >= 0 && x < N && y >= 0 && y < N && board[y * N + x] == 0;
}

/* the cell one step ahead after turning by `a` (CyTronGrid.pyx:31-41) */
static int free_after(int N, const int64_t *board, int64_t head, int64_t dir, int a) {
    int64_t x = head % N, y = head / N, d = (dir + a + 4) % 4;
    if (d == 0) y -= 1; else if (d == 1) x += 1; else if (d == 2) y += 1; else x -= 1;
    return cell_free(N, board, x, y);
}

/* The avoid actions of the seats in `mask` for one environment, written into actions[P]; other seats untouched. */
void orc_tron_avoid_actions(int N, int P, const int64_t *board, const int64_t *heads, const int64_t *directions,
                            const int64_t *deaths, int mask, int noise_q16, uint64_t seed, uint64_t env, uint32_t t,
                            int64_t *actions) {
    uint32_t r[8];
    philox(seed, env, t, 4, r);                                  /* seats 0..3: tag 4 */
    philox(seed, env, t, 5, r + 4);                              /* seats 4..7: tag 5 */
    for (int p = 0; p < P; p++) {
        if (!(mask >> p & 1)) continue;                          /* seats outside the mask keep their action */
        uint32_t w = r[p];
        if (deaths[p] != 0) { actions[p] = 0; continue; }        /* dead seats get 0 */
        if ((int64_t)(w >> 16) < noise_q16) { actions[p] = MOVE[(w & 0xFFFF) % 3]; continue; }   /* noise */
        if (free_after(N, board, heads[p], directions[p], 0)) { actions[p] = 0; continue; }     /* forward */
        int side = (w & 1) ? 1 : -1;                             /* the coin: right if w & 1, else left */
        actions[p] = free_after(N, board, heads[p], directions[p], side) ? side : -side;        /* else the other */
    }
}

typedef struct {
    int N, P; uint64_t seed; int64_t env0, B; uint32_t t0; int K, fresh, mask, noise_q16, ring_offset;
    const int32_t *spawns;
    int64_t *board, *heads, *directions, *deaths; uint8_t *terminal; int32_t *ep_len;
    int tid, T; int64_t loc[NSTAT];
} job_t;

/* the oracle_rollout.c loop (auto-reset, statistics slots) with the avoid policy on the seats of `mask` */
static void env_rollout(job_t *a, int64_t e) {
    int N = a->N, P = a->P;
    int64_t *bd = a->board + e * N * N, *hd = a->heads + e * P, *dr = a->directions + e * P, *de = a->deaths + e * P;
    int64_t *loc = a->loc;
    if (a->fresh) { orc_tron_new_state_spawns(N, P, a->ring_offset, a->spawns, bd, hd, dr, de); a->terminal[e] = 0; a->ep_len[e] = 0; }
    for (int s = 0; s < a->K; s++) {
        /* auto-reset first: the policy decides on the game the step moves on */
        if (a->terminal[e]) { orc_tron_new_state_spawns(N, P, a->ring_offset, a->spawns, bd, hd, dr, de); a->terminal[e] = 0; a->ep_len[e] = 0; }
        uint32_t r[4];
        philox(a->seed, (uint64_t)(a->env0 + e), a->t0 + s, 1, r);
        int64_t act[8] = {0}, rew[8];
        for (int p = 0; p < P && p < 8; p++) act[p] = MOVE[(p < 4 ? r[p] : r[p - 4] / 3) % 3];   /* random policy, tag 1 */
        orc_tron_avoid_actions(N, P, bd, hd, dr, de, a->mask, a->noise_q16, a->seed, (uint64_t)(a->env0 + e),
                               a->t0 + s, act);
        int alive, winners;
        int term = orc_tron_next_state(N, P, bd, hd, dr, de, act, rew, &alive, &winners);
        a->ep_len[e]++; loc[0]++;
        for (int p = 0; p < P; p++) loc[18] += (p + 1) * rew[p];
        if (term) {
            int64_t rank[8];
            orc_tron_compute_ranking(N, P, bd, de, rank);
            loc[1]++; loc[2] += a->ep_len[e];
            if (!winners) loc[7]++;
            for (int p = 0; p < P && p < 4; p++) {
                if (winners >> p & 1) loc[3 + p]++;
                int64_t cells = 0;
                for (int c = 0; c < N * N; c++) cells += bd[c] == p + 1;
                loc[8 + p] += cells;
                loc[14 + p] += rank[p];
            }
            a->terminal[e] = 1;
        }
    }
}

static void *job_main(void *p) {
    job_t *j = (job_t *)p;
    for (int64_t e = j->tid; e < j->B; e += j->T) env_rollout(j, e);
    return NULL;
}

/* K steps (t = t0 .. t0+K-1) of envs [env0, env0+B): seats of `mask` avoid, the others random; finished games restart
 * from (ring_offset, spawn_offsets[P] or NULL = the defaults).  Arrays as orc_tron_rollout's; stats[32] += the slots. */
void orc_tron_rollout_avoid(int N, int P, uint64_t seed, int64_t env0, int64_t B, uint32_t t0, int K, int fresh,
                            int mask, int noise_q16, int ring_offset, const int32_t *spawn_offsets, int64_t *board,
                            int64_t *heads, int64_t *directions, int64_t *deaths, uint8_t *terminal, int32_t *ep_len,
                            int64_t *stats, int nthreads) {
    if (nthreads <= 0) { long n = sysconf(_SC_NPROCESSORS_ONLN); nthreads = n > 0 ? (int)n : 1; }
    if (nthreads > B) nthreads = (int)(B > 0 ? B : 1);
    job_t *jobs = (job_t *)calloc(nthreads, sizeof(job_t));
    pthread_t *th = (pthread_t *)calloc(nthreads, sizeof(pthread_t));
    for (int i = 0; i < nthreads; i++) {
        job_t j = {N, P, seed, env0, B, t0, K, fresh, mask, noise_q16, ring_offset, spawn_offsets,
                   board, heads, directions, deaths, terminal, ep_len, i, nthreads, {0}};
        jobs[i] = j;
        if (i > 0) pthread_create(&th[i], NULL, job_main, &jobs[i]);
    }
    job_main(&jobs[0]);
    for (int i = 1; i < nthreads; i++) pthread_join(th[i], NULL);
    if (stats) for (int i = 0; i < nthreads; i++) for (int k = 0; k < NSTAT; k++) stats[k] += jobs[i].loc[k];
    free(jobs); free(th);
}
