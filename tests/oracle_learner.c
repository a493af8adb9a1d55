/* TEST INFRASTRUCTURE ONLY -- CPU oracle of the single-learner advance (crl_ttt_advance, crl_blokus_advance).
 *
 * Restates, independently of the CUDA source, the rule declared in include/colosseum_b200_learner.h on the
 * reference's unpacked layouts (oracle/oracle_ttt.c, oracle/oracle_blokus.c), with their next_state / valid_actions and
 * Philox.  Compiled together with the oracle/*.c files by tests/cases_learner.py; nothing in the product path uses it.
 *
 * Statistics: int64[32], the slots of include/colosseum_b200.h, added per env-step as the step kernels add them
 * (oracle/oracle_rollout.c lists them); a Blokus opponent move also adds its valid-move count to slot 13.  A Tic Tac
 * Toe episode can last more than 31 steps when the learner passes or plays illegal cells; its state then keeps 31, and
 * that is the length crl_ttt_step adds.
 * Record: rec[0] reward (int8), rec[1] flags, rec[2] winners mask, rec[3] opponent moves; Blokus rec[4..7] scores.
 */
#include <assert.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <pthread.h>
#include <unistd.h>

#define NSTAT 32
#define BLOKUS_CAP 16384

int orc_ttt_cells(int n);
int orc_ttt_next_state(int n, int8_t *board, int *winner, int player, int action, int *reward, int *terminal, int *winner_out);
int orc_ttt_valid_actions(int n, const int8_t *board, int32_t *out);
int orc_blokus_valid_moves(const int64_t *board, int round_count, int color, const uint8_t *inventory, int32_t *out_ids, int cap);
int orc_blokus_next_state(int64_t *board, int *round_count, uint8_t *inventory, int64_t *scores, int mover,
                          int action_id, int *reward, int *terminal, int *winners_mask);

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

/* opponent move j's word: philox(seed, env, t, tag 6 + (j >> 2))[j & 3] */
static uint32_t opponent_word(uint64_t seed, uint64_t env, uint32_t t, int j) {
    uint32_t r[4];
    philox(seed, env, t, 6u + (uint32_t)(j >> 2), r);
    return r[j & 3];
}

/* ------------------------------------------------------------------ Tic Tac Toe */
static int ttt_terminal(int n, const int8_t *board, int winner) {
    int32_t va[32];
    return winner >= 0 || orc_ttt_valid_actions(n, board, va) == 0;
}

static void ttt_new(int n, int8_t *board, int32_t *winner, int32_t *mover, int32_t *ep_len) {
    memset(board, -1, orc_ttt_cells(n)); *winner = -1; *mover = 0; *ep_len = 0;
}

/* one next_state with the statistics of crl_ttt_step; returns terminal */
static int ttt_env_step(int n, int8_t *board, int32_t *winner, int32_t *mover, int32_t *ep_len, int action, int64_t *st,
                        int *winner_out) {
    int32_t va[32];
    int nv = orc_ttt_valid_actions(n, board, va), cells = orc_ttt_cells(n);
    int illegal = action >= 0 && (action >= cells || board[action] != -1);
    int w = *winner, m = *mover, rew, term;
    *mover = orc_ttt_next_state(n, board, &w, m, action, &rew, &term, winner_out);
    *winner = w; *ep_len += 1;
    st[0]++; st[13] += nv; st[12] += illegal; st[18] += (int64_t)(m + 1) * rew;
    if (term) {
        st[1]++; st[2] += *ep_len < 31 ? *ep_len : 31;        /* the state keeps min(episode steps, 31) */
        if (*winner_out < 0) st[7]++; else st[3 + *winner_out]++;
        for (int p = 0; p < n; p++) st[14 + p] += (p == *winner_out) ? 0 : 1;
    }
    return term;
}

/* the rule for one game; has_action = 0 is the NULL mode */
void orc_ttt_advance(int n, int seat, int has_action, int action, uint64_t seed, uint64_t env, uint32_t t, int8_t *board,
                     int32_t *winner, int32_t *mover, int32_t *ep_len, uint8_t rec[4], int64_t *st) {
    int cells = orc_ttt_cells(n), flags = 0, reward = 0, winners = 0, finished = 0, j = 0, wout;
    if (ttt_terminal(n, board, *winner)) ttt_new(n, board, winner, mover, ep_len);           /* 1 */
    if (has_action && *mover == seat) {                                                      /* 2 */
        int placed = action >= 0 && action < cells && board[action] == -1;
        int illegal = action >= 0 && !placed;
        ttt_env_step(n, board, winner, mover, ep_len, action, st, &wout);
        flags |= illegal << 1 | placed << 2;
    } else {
        flags |= 8;
    }
    for (;;) {                                                                               /* 3 */
        if (ttt_terminal(n, board, *winner)) {
            assert(!finished);                                   /* at most one finished game per call */
            finished = 1;
            flags |= 1;
            winners = *winner >= 0 ? 1 << *winner : 0;
            reward = *winner < 0 ? 0 : (*winner == seat ? 1 : -1);
            ttt_new(n, board, winner, mover, ep_len);
            continue;
        }
        if (*mover == seat) break;
        int32_t va[32];
        int m = orc_ttt_valid_actions(n, board, va);
        int a = m ? va[opponent_word(seed, env, t, j) % (uint32_t)m] : -1;
        ttt_env_step(n, board, winner, mover, ep_len, a, st, &wout);
        j++;
        assert(j <= 2 * n - 2);
    }
    rec[0] = (uint8_t)(int8_t)reward; rec[1] = (uint8_t)flags; rec[2] = (uint8_t)winners; rec[3] = (uint8_t)j;
}

/* ------------------------------------------------------------------ Blokus */
/* one next_state with the statistics of crl_blokus_step (+ nvalid); returns terminal */
static int blk_env_step(int64_t *board, int32_t *round, uint8_t *inv, int64_t *sc, int32_t *mover, uint8_t *terminal,
                        int32_t *ep_len, int action, int illegal, int nvalid, int64_t *st, int *winners) {
    int rew, term, rc = *round, m = *mover;
    *mover = orc_blokus_next_state(board, &rc, inv, sc, m, action, &rew, &term, winners);
    *round = rc; *terminal = (uint8_t)term; *ep_len += 1;
    st[0]++; st[12] += illegal; st[13] += nvalid; st[18] += (int64_t)(m + 1) * rew;
    if (term) {
        st[1]++; st[2] += *ep_len;
        if (!*winners) st[7]++;
        for (int p = 0; p < 4; p++) {
            if (*winners >> p & 1) st[3 + p]++; else st[14 + p]++;
            st[8 + p] += sc[p];
        }
    }
    return term;
}

static void blk_new(int64_t *board, int32_t *round, uint8_t *inv, int64_t *sc, int32_t *mover, uint8_t *terminal,
                    int32_t *ep_len) {
    memset(board, 0, sizeof(int64_t) * 400); memset(inv, 1, 84); memset(sc, 0, sizeof(int64_t) * 4);
    *round = 0; *mover = 0; *terminal = 0; *ep_len = 0;
}

/* the rule for one game; ids: scratch of BLOKUS_CAP ids */
void orc_blokus_advance(int seat, int has_action, int action, uint64_t seed, uint64_t env, uint32_t t, int64_t *board,
                        int32_t *round, uint8_t *inv, int64_t *sc, int32_t *mover, uint8_t *terminal, int32_t *ep_len,
                        uint8_t rec[8], int64_t *st, int32_t *ids) {
    int flags = 0, reward = 0, winners = 0, finished = 0, j = 0, w;
    int64_t final[4] = {0, 0, 0, 0};
    if (*terminal) blk_new(board, round, inv, sc, mover, terminal, ep_len);                  /* 1 */
    if (has_action && *mover == seat) {                                                      /* 2 */
        int m = orc_blokus_valid_moves(board, *round, seat + 1, inv + seat * 21, ids, BLOKUS_CAP), legal = 0;
        assert(m <= BLOKUS_CAP);
        for (int i = 0; i < m && action >= 0; i++) legal |= ids[i] == action;
        blk_env_step(board, round, inv, sc, mover, terminal, ep_len, legal ? action : -1, action >= 0 && !legal, 0, st, &w);
        flags |= (action >= 0 && !legal) << 1 | legal << 2;
    } else {
        flags |= 8;
    }
    for (;;) {                                                                               /* 3 */
        if (*terminal) {
            assert(!finished);
            finished = 1;
            flags |= 1;
            winners = 0;
            int64_t mx = 0;
            for (int q = 0; q < 4; q++) mx = sc[q] > mx ? sc[q] : mx;
            for (int q = 0; q < 4; q++) {
                winners |= (sc[q] == mx) << q;
                reward += sc[q] < sc[seat] || (sc[q] == sc[seat] && q < seat);
                final[q] = sc[q];
            }
            blk_new(board, round, inv, sc, mover, terminal, ep_len);
            continue;
        }
        if (*mover == seat) break;
        int m = orc_blokus_valid_moves(board, *round, *mover + 1, inv + *mover * 21, ids, BLOKUS_CAP);
        assert(m <= BLOKUS_CAP);
        int a = m ? ids[opponent_word(seed, env, t, j) % (uint32_t)m] : -1;
        blk_env_step(board, round, inv, sc, mover, terminal, ep_len, a, 0, m, st, &w);
        j++;
        assert(j <= 6);
    }
    rec[0] = (uint8_t)(int8_t)reward; rec[1] = (uint8_t)flags; rec[2] = (uint8_t)winners; rec[3] = (uint8_t)j;
    for (int q = 0; q < 4; q++) rec[4 + q] = (uint8_t)final[q];
}

/* ------------------------------------------------------------------ batches (pthreads over interleaved games) */
typedef struct {
    int game, n, seat; const void *actions; uint64_t seed; int64_t env0, B; uint32_t t;
    int8_t *tboard; int64_t *bboard; int32_t *winner_or_round, *mover, *ep_len; uint8_t *inv, *terminal, *rec;
    int64_t *scores; int tid, T; int64_t loc[NSTAT];
} job_t;

static void *job_main(void *p) {
    job_t *a = (job_t *)p;
    int32_t *ids = a->game ? (int32_t *)malloc(sizeof(int32_t) * BLOKUS_CAP) : NULL;
    for (int64_t e = a->tid; e < a->B; e += a->T) {
        const uint64_t env = (uint64_t)(a->env0 + e);
        if (a->game == 0) {
            int cells = orc_ttt_cells(a->n);
            int act = a->actions ? ((const int8_t *)a->actions)[e] : -1;
            orc_ttt_advance(a->n, a->seat, a->actions != NULL, act, a->seed, env, a->t, a->tboard + e * cells,
                            a->winner_or_round + e, a->mover + e, a->ep_len + e, a->rec + 4 * e, a->loc);
        } else {
            int act = a->actions ? ((const int32_t *)a->actions)[e] : -1;
            orc_blokus_advance(a->seat, a->actions != NULL, act, a->seed, env, a->t, a->bboard + e * 400,
                               a->winner_or_round + e, a->inv + e * 84, a->scores + e * 4, a->mover + e, a->terminal + e,
                               a->ep_len + e, a->rec + 8 * e, a->loc, ids);
        }
    }
    free(ids);
    return NULL;
}

static void run(job_t proto, int64_t *stats, int nthreads) {
    if (nthreads <= 0) { long n = sysconf(_SC_NPROCESSORS_ONLN); nthreads = n > 0 ? (int)n : 1; }
    if (nthreads > proto.B) nthreads = (int)(proto.B > 0 ? proto.B : 1);
    job_t *jobs = (job_t *)calloc(nthreads, sizeof(job_t));
    pthread_t *th = (pthread_t *)calloc(nthreads, sizeof(pthread_t));
    for (int i = 0; i < nthreads; i++) {
        jobs[i] = proto; jobs[i].tid = i; jobs[i].T = nthreads;
        if (i > 0) pthread_create(&th[i], NULL, job_main, &jobs[i]);
    }
    job_main(&jobs[0]);
    for (int i = 1; i < nthreads; i++) pthread_join(th[i], NULL);
    if (stats) for (int i = 0; i < nthreads; i++) for (int k = 0; k < NSTAT; k++) stats[k] += jobs[i].loc[k];
    free(jobs); free(th);
}

/* games [env0, env0 + B), in place; board int8[B][cells], winner / mover / ep_len int32[B]; actions int8[B] or NULL;
 * rec uint8[B][4]; stats[32] += the slots */
void orc_ttt_advance_batch(int n, int seat, const int8_t *actions, uint64_t seed, int64_t env0, int64_t B, uint32_t t,
                           int8_t *board, int32_t *winner, int32_t *mover, int32_t *ep_len, uint8_t *rec, int64_t *stats,
                           int nthreads) {
    job_t j = {0};
    j.game = 0; j.n = n; j.seat = seat; j.actions = actions; j.seed = seed; j.env0 = env0; j.B = B; j.t = t;
    j.tboard = board; j.winner_or_round = winner; j.mover = mover; j.ep_len = ep_len; j.rec = rec;
    run(j, stats, nthreads);
}

/* board int64[B][400], round / mover / ep_len int32[B], inventory u8[B][4][21], scores int64[B][4], terminal u8[B];
 * actions int32[B] or NULL; rec uint8[B][8] */
void orc_blokus_advance_batch(int seat, const int32_t *actions, uint64_t seed, int64_t env0, int64_t B, uint32_t t,
                              int64_t *board, int32_t *round, uint8_t *inventory, int64_t *scores, int32_t *mover,
                              uint8_t *terminal, int32_t *ep_len, uint8_t *rec, int64_t *stats, int nthreads) {
    job_t j = {0};
    j.game = 1; j.seat = seat; j.actions = actions; j.seed = seed; j.env0 = env0; j.B = B; j.t = t;
    j.bboard = board; j.winner_or_round = round; j.inv = inventory; j.scores = scores; j.mover = mover;
    j.terminal = terminal; j.ep_len = ep_len; j.rec = rec;
    run(j, stats, nthreads);
}
