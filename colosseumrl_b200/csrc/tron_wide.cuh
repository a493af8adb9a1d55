// Tron beyond the default shape: any board 5 <= N <= 64 and 2 <= P <= 8 players (sm_100a).
//
// The reference takes any "N;P" (TronGridEnvironment.py:28-58; CyTronGrid.pyx:8-9 reads N and P from the array
// shapes).  The tuned kernels of tron.cuh cover N <= 19, P <= 4 (384-bit planes, four byte lanes -- BASELINE.json's
// configuration and everything near it); every other shape runs here: same semantics, same entry points, a plain
// one-thread-per-environment formulation of
//   next_state_inplace            envs/tron/CyTronGrid.pyx:3-62
//   TronGridEnvironment.next_state envs/tron/TronGridEnvironment.py:265-323
//   compute_ranking               :483-508   (incl. the deaths[-1] wrap-around, in place and ascending like the reference)
//   new_state                     :228-263
//   state_to_observation          :363-405 + relative_player_inplace CyTronGrid.pyx:65-71
//
// HBM layout ("wide"): SoA of 32-bit words, uint32 [W][B], word-major so that every access of a warp is coalesced:
//   word p * WPP + j          bits 32 j .. 32 j + 31 of player p's bitboard (bit y*N + x), WPP = ceil(N*N / 32)
//   word H + p                header of player p: head x | head y << 8 | direction << 16 | deaths << 20     (H = P * WPP)
//   word H + P + p            cells owned by player p (= compute_ranking's score)
//   word H + 2 P              terminal | episode steps << 1
// W = P * WPP + 2 P + 1 (N = 21, P = 4: 65 words = 260 B; N = 11, P = 6: 37 words).
// actions: int8 [B][8]; result record: 16 bytes = int8 reward[8] | u8 terminal | u8 alive mask | u8 winners mask | u8 0 |
// u32 ranking, 3 bits per player.
#pragma once
#include "crl_common.cuh"
#include "philox.cuh"
#include "tron.cuh"             // tron_avoid_decide

#define TRONW_MAXP 8

struct TronWideParams {
    int N, P, WPP, W;
    int start_head[TRONW_MAXP], start_dir[TRONW_MAXP];
};

// one environment's view of a word-major buffer
struct TronWideRef {
    uint32_t *base;      // &state[e]
    long long B;
    __device__ __forceinline__ uint32_t &operator[](int w) const { return base[(long long)w * B]; }
};

struct TronWideEnv {
    int hx[TRONW_MAXP], hy[TRONW_MAXP], dir[TRONW_MAXP], death[TRONW_MAXP], cells[TRONW_MAXP];
    uint32_t terminal, ep_len;
};

struct TronWideOut {
    int reward[TRONW_MAXP];
    uint32_t alive, winners, terminal, rank;      // rank: 3 bits per player
};

__device__ __forceinline__ void tronw_hdr_load(TronWideEnv &s, const TronWideRef &st, const TronWideParams &prm) {
    const int H = prm.P * prm.WPP;
#pragma unroll
    for (int p = 0; p < TRONW_MAXP; p++) {
        if (p < prm.P) {
            const uint32_t h = st[H + p];
            s.hx[p] = (int)(h & 255u); s.hy[p] = (int)(h >> 8 & 255u); s.dir[p] = (int)(h >> 16 & 3u); s.death[p] = (int)(h >> 20 & 15u);
            s.cells[p] = (int)st[H + prm.P + p];
        } else {
            s.hx[p] = s.hy[p] = s.dir[p] = s.death[p] = s.cells[p] = 0;
        }
    }
    const uint32_t m = st[H + 2 * prm.P];
    s.terminal = m & 1u; s.ep_len = m >> 1;
}

__device__ __forceinline__ void tronw_hdr_store(const TronWideEnv &s, const TronWideRef &st, const TronWideParams &prm) {
    const int H = prm.P * prm.WPP;
#pragma unroll
    for (int p = 0; p < TRONW_MAXP; p++)
        if (p < prm.P) {
            st[H + p] = (uint32_t)s.hx[p] | (uint32_t)s.hy[p] << 8 | (uint32_t)s.dir[p] << 16 | (uint32_t)s.death[p] << 20;
            st[H + prm.P + p] = (uint32_t)s.cells[p];
        }
    st[H + 2 * prm.P] = s.terminal | s.ep_len << 1;
}

// new_state (TronGridEnvironment.py:228-263): header only; the planes are written by the caller
__device__ __forceinline__ void tronw_new_hdr(TronWideEnv &s, const TronWideParams &prm) {
#pragma unroll
    for (int p = 0; p < TRONW_MAXP; p++) {
        const bool on = p < prm.P;
        s.hx[p] = on ? prm.start_head[p] % prm.N : 0; s.hy[p] = on ? prm.start_head[p] / prm.N : 0;
        s.dir[p] = on ? prm.start_dir[p] : 0; s.death[p] = 0; s.cells[p] = on ? 1 : 0;
    }
    s.terminal = 0; s.ep_len = 0;
}

// word w (< P * WPP) of a fresh board: the spawn bit of its plane's player if it lies in this word
__device__ __forceinline__ uint32_t tronw_spawn_word(int w, const TronWideParams &prm) {
    const int p = w / prm.WPP, j = w - p * prm.WPP;
    int head = 0;
#pragma unroll
    for (int q = 0; q < TRONW_MAXP; q++) head = (q == p) ? prm.start_head[q] : head;
    return (head >> 5) == j ? 1u << (head & 31) : 0u;
}

// CyTronGrid.pyx:15-62 -- players strictly in index order against the board as it is being updated -- on the planes
// in `st` (already the output buffer), then TronGridEnvironment.py:309-321
__device__ __forceinline__ void tronw_step_env(TronWideEnv &s, const TronWideRef &st, const int8_t *act,
                                               const TronWideParams &prm, TronWideOut &o) {
    const int N = prm.N, P = prm.P;
#pragma unroll 1
    for (int i = 0; i < P; i++) {
        int hx = 0, hy = 0, dr = 0, de = 0, a = 0;                        // (register arrays: constant indices only)
#pragma unroll
        for (int q = 0; q < TRONW_MAXP; q++)
            if (q == i) { hx = s.hx[q]; hy = s.hy[q]; dr = s.dir[q]; de = s.death[q]; a = (int)act[q]; }
        if (de > 0) continue;                                             // pyx:16
        const int d = (dr + a + 4) & 3;                                   // pyx:31
        int x = hx, y = hy;
        if (d == 0) y -= 1; else if (d == 1) x += 1; else if (d == 2) y += 1; else x -= 1;   // pyx:34-41
        int nde = 0, kill = -1;
        bool moved = false;
        if (x < 0 || x >= N || y < 0 || y >= N) {
            nde = i + 1;                                                  // pyx:47-48
        } else {
            const int cell = y * N + x, wj = cell >> 5;
            const uint32_t bit = 1u << (cell & 31);
            int owner = 0;
#pragma unroll 1
            for (int q = 0; q < P; q++)
                if (st[q * prm.WPP + wj] & bit) owner = q + 1;            // planes are disjoint: at most one owner
            if (owner) {
                nde = owner;                                              // pyx:51-53
                int ohx = 0, ohy = 0;
#pragma unroll
                for (int q = 0; q < TRONW_MAXP; q++)
                    if (q == owner - 1) { ohx = s.hx[q]; ohy = s.hy[q]; }
                if (ohx == x && ohy == y) kill = owner - 1;               // pyx:56-57 (no liveness check)
            } else {
                st[i * prm.WPP + wj] |= bit;                              // pyx:60-62
                moved = true;
            }
        }
#pragma unroll
        for (int q = 0; q < TRONW_MAXP; q++) {
            if (q == i) {
                s.dir[q] = d;                                             // pyx:44 (also when i dies)
                s.death[q] = nde;
                if (moved) { s.hx[q] = x; s.hy[q] = y; s.cells[q] += 1; }
            }
        }
#pragma unroll
        for (int q = 0; q < TRONW_MAXP; q++)
            if (q == kill) s.death[q] = i + 1;                            // (kill == i: a player running into its own head cell)
    }
    s.ep_len += 1;
    uint32_t alive = 0;
    int n_alive = 0;
#pragma unroll
    for (int p = 0; p < TRONW_MAXP; p++)
        if (p < P && s.death[p] == 0) { alive |= 1u << p; n_alive++; }    // py:310
    o.alive = alive;
    o.terminal = n_alive <= 1;                                            // py:316
    o.winners = o.terminal ? alive : 0u;                                  // py:319
#pragma unroll
    for (int p = 0; p < TRONW_MAXP; p++)
        o.reward[p] = p < P ? ((alive >> p & 1u) ? (o.terminal ? 10 : 1) : -1) : 0;   // py:313, 320-321
    s.terminal = o.terminal;
}

// compute_ranking (TronGridEnvironment.py:483-508): scores = cells owned; for every p of tie_locations (computed up
// front, :492, with numpy's negative-index wrap for the alive: deaths[-1] is the LAST player) ascending and in place
// score[p] = min(score[p], score[deaths[p] - 1]) where Counter[-1] reads 0 (:493-495); competition ranking by
// descending score (:497-506).  3 bits per player.
__device__ __forceinline__ uint32_t tronw_ranking(const TronWideEnv &s, const TronWideParams &prm) {
    const int P = prm.P;
    int score[TRONW_MAXP];
    uint32_t tie = 0;
#pragma unroll
    for (int p = 0; p < TRONW_MAXP; p++) score[p] = s.cells[p];
#pragma unroll
    for (int p = 0; p < TRONW_MAXP; p++) {
        if (p < P) {
            int k = s.death[p] - 1;
            if (k < 0) k += P;
            int dk = 0;
#pragma unroll
            for (int q = 0; q < TRONW_MAXP; q++) dk = (q == k) ? s.death[q] : dk;
            if (dk == p + 1) tie |= 1u << p;
        }
    }
#pragma unroll
    for (int p = 0; p < TRONW_MAXP; p++) {
        if (tie >> p & 1u) {
            const int killer = s.death[p] - 1;
            int ks = 0;
#pragma unroll
            for (int q = 0; q < TRONW_MAXP; q++) ks = (q == killer) ? score[q] : ks;
            score[p] = min(score[p], ks);
        }
    }
    uint32_t rk = 0;
#pragma unroll
    for (int p = 0; p < TRONW_MAXP; p++) {
        if (p < P) {
            int r = 0;
#pragma unroll
            for (int q = 0; q < TRONW_MAXP; q++) r += (q < P && q != p && score[q] > score[p]) ? 1 : 0;
            rk |= (uint32_t)r << (3 * p);
        }
    }
    return rk;
}

__device__ __forceinline__ void tronw_store_result(uint4 *result, long long e, const TronWideOut &o) {
    uint32_t r0 = 0, r1 = 0;
#pragma unroll
    for (int p = 0; p < 4; p++) {
        r0 |= ((uint32_t)o.reward[p] & 255u) << (8 * p);
        r1 |= ((uint32_t)o.reward[4 + p] & 255u) << (8 * p);
    }
    result[e] = make_uint4(r0, r1, o.terminal | o.alive << 8 | o.winners << 16, o.rank);
}

// episode statistics (seats 0..3 only: the statistics vector has four per-seat slots)
__device__ __forceinline__ void tronw_stats(const BlockStats &bs, bool valid, const TronWideEnv &s, const TronWideOut &o, int P) {
    const bool t = valid && o.terminal;
    int rw = 0;
#pragma unroll
    for (int p = 0; p < TRONW_MAXP; p++) rw += (p + 1) * o.reward[p];
    bs.add(ST_STEPS, valid ? 1 : 0);
    bs.add(ST_REWARD, valid ? rw : 0);
    bs.add(ST_EPISODES, t ? 1 : 0);
    bs.add(ST_EPLEN, t ? (int)s.ep_len : 0);
    bs.add(ST_NOWIN, (t && o.winners == 0u) ? 1 : 0);
#pragma unroll
    for (int p = 0; p < 4; p++) {
        bs.add(ST_WINS + p, (t && (o.winners >> p & 1u)) ? 1 : 0);
        bs.add(ST_SCORE + p, (t && p < P) ? s.cells[p] : 0);
        bs.add(ST_RANK + p, (t && p < P) ? (int)(o.rank >> (3 * p) & 7u) : 0);
    }
}

__device__ __forceinline__ void tronw_zero_out(TronWideOut &o) {
#pragma unroll
    for (int p = 0; p < TRONW_MAXP; p++) o.reward[p] = 0;
    o.alive = o.winners = o.terminal = o.rank = 0u;
}

// next_state for a batch; out may equal in
__global__ void __launch_bounds__(128)
tronw_step_kernel(const uint32_t *__restrict__ in, uint32_t *__restrict__ out, const int8_t *__restrict__ actions,
                  uint4 *__restrict__ result, crl_u64 *stats, long long B, TronWideParams prm, int flags) {
    __shared__ int sm_stat[CRL_NSTAT];
    BlockStats bs{sm_stat};
    if (stats) bs.init();
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = e < B;
    TronWideEnv s;
    TronWideOut o;
    tronw_zero_out(o);
    tronw_new_hdr(s, prm);
    if (valid) {
        const TronWideRef src{const_cast<uint32_t *>(in) + e, B}, dst{out + e, B};
        tronw_hdr_load(s, src, prm);
        const bool reset = (flags & CRL_FLAG_AUTO_RESET) && s.terminal;
        if (reset) tronw_new_hdr(s, prm);
        const int PW = prm.P * prm.WPP;
        if (reset) {
            for (int w = 0; w < PW; w++) dst[w] = tronw_spawn_word(w, prm);
        } else if (in != out) {
            for (int w = 0; w < PW; w++) dst[w] = src[w];
        }
        int8_t act[TRONW_MAXP];
        const uint2 a8 = *(const uint2 *)(actions + e * TRONW_MAXP);
#pragma unroll
        for (int p = 0; p < TRONW_MAXP; p++) act[p] = (int8_t)((p < 4 ? a8.x : a8.y) >> (8 * (p & 3)));
        tronw_step_env(s, dst, act, prm, o);
        o.rank = tronw_ranking(s, prm);
        tronw_hdr_store(s, dst, prm);
        tronw_store_result(result, e, o);
    }
    if (stats) {
        tronw_stats(bs, valid, s, o, prm.P);
        bs.flush(stats);
    }
}

// action of player p at (env, step): {0, +1, -1}[r[p] % 3] for p < 4, {0, +1, -1}[(r[p - 4] / 3) % 3] for p >= 4
// (one Philox call per environment and step; identical to oracle/oracle_rollout.c and oracle/make_golden.py)
__device__ __forceinline__ void tronw_random_actions(int8_t *act, crl_u64 seed, crl_u64 env, uint32_t step) {
    const uint4 r = env_words(seed, env, step, CRL_TAG_TRON);
    const uint32_t rr[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int p = 0; p < TRONW_MAXP; p++) {
        const uint32_t m = (p < 4 ? rr[p & 3] : rr[p & 3] / 3u) % 3u;
        act[p] = (int8_t)(m == 2u ? -1 : (int)m);
    }
}

__global__ void tronw_policy_random_kernel(int8_t *__restrict__ actions, long long B, crl_u64 seed, crl_u64 first_env,
                                           uint32_t step) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= B) return;
    int8_t act[TRONW_MAXP];
    tronw_random_actions(act, seed, first_env + (crl_u64)e, step);
    uint32_t lo = 0, hi = 0;
#pragma unroll
    for (int p = 0; p < 4; p++) { lo |= ((uint32_t)act[p] & 255u) << (8 * p); hi |= ((uint32_t)act[4 + p] & 255u) << (8 * p); }
    *(uint2 *)(actions + e * TRONW_MAXP) = make_uint2(lo, hi);
}

// The avoid policy (tron.cuh: tron_avoid_decide) for the seats in `mask`, written into act[]; the other seats keep
// theirs, dead seats get 0.  A cell is occupied if its bit is set in any of the P player planes of `st` or, when
// `fresh` (a game the step will restart), if it is one of new_state's spawns.  Seats 0..3 draw their word from tag
// CRL_TAG_TRON_AVOID, seats 4..7 from the next tag.
__device__ __forceinline__ void tronw_avoid_actions(int8_t *act, const TronWideEnv &s, const TronWideRef &st, bool fresh,
                                                    const TronWideParams &prm, uint32_t mask, uint32_t noise_q16,
                                                    crl_u64 seed, crl_u64 env, uint32_t step) {
    auto occupied = [&](int cell) {
        if (fresh) {
            bool spawn = false;
#pragma unroll
            for (int q = 0; q < TRONW_MAXP; q++) spawn |= q < prm.P && prm.start_head[q] == cell;
            return spawn;
        }
        uint32_t any = 0;
#pragma unroll 1
        for (int q = 0; q < prm.P; q++) any |= st[q * prm.WPP + (cell >> 5)];
        return ((any >> (cell & 31)) & 1u) != 0u;
    };
    uint4 lo = make_uint4(0u, 0u, 0u, 0u), hi = lo;
    if (mask & 0x0Fu) lo = env_words(seed, env, step, CRL_TAG_TRON_AVOID);
    if (mask & 0xF0u) hi = env_words(seed, env, step, CRL_TAG_TRON_AVOID + 1u);
    const uint32_t rr[TRONW_MAXP] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
#pragma unroll
    for (int p = 0; p < TRONW_MAXP; p++)
        if ((mask >> p) & 1u)
            act[p] = (int8_t)(s.death[p] ? 0 : tron_avoid_decide(s.hx[p], s.hy[p], s.dir[p], prm.N, rr[p], noise_q16, occupied));
}

// crl_tron_policy_avoid on the wide layout: one thread per environment, actions int8[B][8] read-modify-written as one
// 8-byte word.  Only the words of the <= 3 candidate cells are read, from each of the P planes: the wide layout is
// word-major, so a warp's loads of one word index are coalesced, and the board (up to 1 KB per environment) is far
// larger than what the lookups touch.
__global__ void __launch_bounds__(128)
tronw_policy_avoid_kernel(const uint32_t *__restrict__ st, int8_t *__restrict__ actions, long long B, TronWideParams prm,
                          uint32_t mask, uint32_t noise_q16, crl_u64 seed, crl_u64 first_env, uint32_t step, int flags) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= B) return;
    const TronWideRef src{const_cast<uint32_t *>(st) + e, B};
    TronWideEnv s;
    tronw_hdr_load(s, src, prm);
    const bool fresh = (flags & CRL_FLAG_AUTO_RESET) && s.terminal;       // decide on the game the step will restart
    if (fresh) tronw_new_hdr(s, prm);
    uint2 a8 = *(const uint2 *)(actions + e * TRONW_MAXP);
    int8_t act[TRONW_MAXP];
#pragma unroll
    for (int p = 0; p < TRONW_MAXP; p++) act[p] = (int8_t)((p < 4 ? a8.x : a8.y) >> (8 * (p & 3)));
    tronw_avoid_actions(act, s, src, fresh, prm, mask, noise_q16, seed, first_env + (crl_u64)e, step);
    a8 = make_uint2(0u, 0u);
#pragma unroll
    for (int p = 0; p < TRONW_MAXP; p++) (p < 4 ? a8.x : a8.y) |= ((uint32_t)act[p] & 255u) << (8 * (p & 3));
    *(uint2 *)(actions + e * TRONW_MAXP) = a8;
}

// K random-policy steps with auto-reset, in place.  AVOID: the seats of avoid_mask play the avoid policy instead
// (= K x policy_random_wide -> policy_avoid(avoid_mask, CRL_FLAG_AUTO_RESET) -> step(CRL_FLAG_AUTO_RESET)); a finished
// game is already restarted before the actions are drawn, so the policy sees the board the step moves on.
template <bool AVOID = false>
__global__ void __launch_bounds__(128)
tronw_rollout_kernel(uint32_t *__restrict__ state, uint4 *__restrict__ result, crl_u64 *stats, long long B,
                     TronWideParams prm, crl_u64 seed, crl_u64 first_env, uint32_t step0, int K, uint32_t avoid_mask,
                     uint32_t noise_q16) {
    __shared__ int sm_stat[CRL_NSTAT];
    BlockStats bs{sm_stat};
    if (stats) bs.init();
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = e < B;
    TronWideEnv s;
    TronWideOut o;
    tronw_zero_out(o);
    tronw_new_hdr(s, prm);
    const TronWideRef st{state + (valid ? e : 0), B};
    if (valid) tronw_hdr_load(s, st, prm);
    for (int k = 0; k < K; k++) {
        if (valid) {
            if (s.terminal) {
                tronw_new_hdr(s, prm);
                for (int w = 0; w < prm.P * prm.WPP; w++) st[w] = tronw_spawn_word(w, prm);
            }
            int8_t act[TRONW_MAXP];
            tronw_random_actions(act, seed, first_env + (crl_u64)e, step0 + (uint32_t)k);
            if constexpr (AVOID)
                tronw_avoid_actions(act, s, st, false, prm, avoid_mask, noise_q16, seed, first_env + (crl_u64)e,
                                    step0 + (uint32_t)k);
            tronw_step_env(s, st, act, prm, o);
            o.rank = tronw_ranking(s, prm);
        }
        if (stats) tronw_stats(bs, valid, s, o, prm.P);
    }
    if (valid) {
        tronw_hdr_store(s, st, prm);
        if (result) tronw_store_result(result, e, o);
    }
    if (stats) bs.flush(stats);
}

// new_state for all / masked environments: one thread per (word, environment)
__global__ void tronw_reset_kernel(uint32_t *__restrict__ state, const uint8_t *__restrict__ mask, long long B, TronWideParams prm) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= B * prm.W) return;
    const int w = (int)(idx / B);
    const long long e = idx - (long long)w * B;
    if (mask && !mask[e]) return;
    const int H = prm.P * prm.WPP;
    uint32_t v;
    if (w < H) {
        v = tronw_spawn_word(w, prm);
    } else if (w < H + prm.P) {
        int head = 0, dir = 0;
#pragma unroll
        for (int q = 0; q < TRONW_MAXP; q++)
            if (q == w - H) { head = prm.start_head[q]; dir = prm.start_dir[q]; }
        v = (uint32_t)(head % prm.N) | (uint32_t)(head / prm.N) << 8 | (uint32_t)dir << 16;
    } else {
        v = w < H + 2 * prm.P ? 1u : 0u;
    }
    state[idx] = v;
}

// state_to_observation (TronGridEnvironment.py:385-405): one thread per (environment, view, cell); the per-player
// vectors are written by the threads of cell 0.  player >= 0: that player's view; -1: absolute; -3: all P views.
__global__ void tronw_observe_kernel(const uint32_t *__restrict__ st, long long B, TronWideParams prm, int player,
                                     int8_t *__restrict__ board, int32_t *__restrict__ heads, int32_t *__restrict__ dirs,
                                     int32_t *__restrict__ deaths, uint8_t *__restrict__ terminal) {
    const int N = prm.N, P = prm.P, NN = N * N, nview = player == -3 ? P : 1;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= B * nview * NN) return;
    const int cell = (int)(idx % NN);
    const long long ev = idx / NN;
    const int view = (int)(ev % nview);
    const long long e = ev / nview;
    const int viewer = player == -3 ? view : player;
    const uint32_t *base = st + e;
    int owner = 0;
    for (int q = 0; q < P; q++)
        if (base[(long long)(q * prm.WPP + (cell >> 5)) * B] >> (cell & 31) & 1u) owner = q + 1;
    int v = owner;
    if (viewer >= 0 && owner > 0) v = ((owner - (viewer + 1) + P) % P) + 1;         // CyTronGrid.pyx:65-71
    board[idx] = (int8_t)v;
    if (cell == 0) {
        const int H = P * prm.WPP;
        for (int c = 0; c < P; c++) {
            const int src = viewer >= 0 ? (c + viewer) % P : c;                    // py:392
            const uint32_t h = base[(long long)(H + src) * B];
            const long long o = ev * P + c;
            if (heads) heads[o] = (int)(h >> 8 & 255u) * N + (int)(h & 255u);
            if (dirs) dirs[o] = (int)(h >> 16 & 3u);
            if (deaths) deaths[o] = (int)(h >> 20 & 15u);
        }
        if (terminal && view == 0) terminal[e] = (uint8_t)(base[(long long)(H + 2 * P) * B] & 1u);
    }
}

// compute_ranking of an arbitrary state: uint32 per environment, 3 bits per player
__global__ void tronw_ranking_kernel(const uint32_t *__restrict__ st, long long B, TronWideParams prm, uint32_t *__restrict__ ranking) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= B) return;
    TronWideEnv s;
    tronw_hdr_load(s, TronWideRef{const_cast<uint32_t *>(st) + e, B}, prm);
    ranking[e] = tronw_ranking(s, prm);
}

// import a reference-layout state; one thread per (word, environment)
__global__ void tronw_pack_kernel(uint32_t *__restrict__ st, long long B, TronWideParams prm, const int8_t *__restrict__ board,
                                  const int32_t *__restrict__ heads, const int32_t *__restrict__ dirs,
                                  const int32_t *__restrict__ deaths) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= B * prm.W) return;
    const int w = (int)(idx / B), N = prm.N, P = prm.P, NN = N * N, H = P * prm.WPP;
    const long long e = idx - (long long)w * B;
    const int8_t *bd = board + e * NN;
    uint32_t v = 0;
    if (w < H) {
        const int p = w / prm.WPP, j = w - p * prm.WPP;
        for (int b = 0; b < 32; b++) {
            const int c = 32 * j + b;
            if (c < NN && bd[c] == p + 1) v |= 1u << b;
        }
    } else if (w < H + P) {
        const int p = w - H, h = heads[e * P + p];
        v = (uint32_t)(h % N) | (uint32_t)(h / N) << 8 | ((uint32_t)dirs[e * P + p] & 3u) << 16 | ((uint32_t)deaths[e * P + p] & 15u) << 20;
    } else if (w < H + 2 * P) {
        const int p = w - H - P;
        for (int c = 0; c < NN; c++) v += bd[c] == p + 1;
    } else {
        int alive = 0;
        for (int p = 0; p < P; p++) alive += deaths[e * P + p] == 0;
        v = alive <= 1 ? 1u : 0u;
    }
    st[idx] = v;
}
