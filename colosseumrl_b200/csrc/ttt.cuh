// Generalised Tic Tac Toe (2p 3x3, 3p 3x5, 4p 3x3x3): batched next_state with the win test done as
// shifted-mask compares, fused with terminal / winners / ranking / valid-action mask (sm_100a).
//
// Replaces (reference file:line):
//   TicTacToe{2,3,4}PlayerEnv.next_state   envs/tictactoe/tictactoe_2p_env.py:240-315, _3p_env.py:241-316,
//                                          _4p_env.py:271-346 (13 scipy.signal.correlate calls per step for 4p)
//   valid_actions / is_valid_action        tictactoe_2p_env.py:317-380
//   new_state                              :139-170
//   state_to_observation                   :382-407 (+ the "% 3" relabel quirk of tictactoe_4p_env.py:50)
//
// HBM layout: ONE 16-byte vector per environment, uint4 state[B], MOVER-RELATIVE: word j holds the cells of the
// player who moves j turns from now,
//   .x = cells of the mover (bit = C-order flat cell index, <= 27 bits) | mover << 27 | (winner + 1) << 29
//   .y = cells of player (mover + 1) % n | min(episode steps, 31) << 27
//   .z = cells of player (mover + 2) % n,   .w = cells of player (mover + 3) % n       (words >= n are zero)
// so a move is `x |= bit` followed by a rotation of the four words (register renaming): no 4-way select on the mover
// to find its cells and none to write them back (the seat-indexed layout spent 13 ALU-pipe instructions per step on
// those).  A warp loads/stores 512 contiguous bytes per instruction; one thread owns one environment.
//
// Win test: for every line direction d (4 in 2-D, 13 in 3-D) with flat stride s_d, three in a row exists iff
//   m & (m >> s_d) & (m >> 2 s_d) & START_d != 0,  START_d = cells where a length-3 segment along d fits.
// This equals "3 in scipy.signal.correlate(mask, pattern, 'valid')" for the reference's WINNING_SHAPES
// (checked against the oracle's 8 / 20 / 49 line tables in tests/test_abi.py::test_ttt_line_tables).
#pragma once
#include "crl_common.cuh"
#include "philox.cuh"
#include "ttt_tables.h"

#define TTT_MAX_DIRS 13

struct TTTParams {
    int n;          // players: 2, 3, 4
    int cells;      // 9, 15, 27
    int ndirs;
    uint32_t cellmask;
    uint32_t stride[TTT_MAX_DIRS];
    uint32_t start[TTT_MAX_DIRS];
};

struct TTTEnv {
    uint32_t c[4];       // MOVER-RELATIVE: c[j] = cells of player (mover + j) % n
    int mover, winner1;  // winner1 = winner + 1, 0 = None
    uint32_t ep_len;
};

struct TTTOut {
    int reward, terminal, error, placed, winners, nvalid;
    uint32_t valid_after;
};

__device__ __forceinline__ void ttt_decode(TTTEnv &s, uint4 v) {
    s.c[0] = v.x & 0x07ffffffu; s.c[1] = v.y & 0x07ffffffu; s.c[2] = v.z & 0x07ffffffu; s.c[3] = v.w & 0x07ffffffu;
    s.mover = (v.x >> 27) & 3; s.winner1 = (v.x >> 29) & 7;
    s.ep_len = v.y >> 27;
}
__device__ __forceinline__ uint4 ttt_encode(const TTTEnv &s) {
    return make_uint4(s.c[0] | (uint32_t)s.mover << 27 | (uint32_t)s.winner1 << 29,
                      s.c[1] | min(s.ep_len, 31u) << 27, s.c[2], s.c[3]);
}
__device__ __forceinline__ void ttt_new_state(TTTEnv &s) {
    s.c[0] = s.c[1] = s.c[2] = s.c[3] = 0; s.mover = 0; s.winner1 = 0; s.ep_len = 0;
}
template <int NP>
__device__ __forceinline__ bool ttt_is_terminal(const TTTEnv &s) {
    return s.winner1 != 0 || ((s.c[0] | s.c[1] | s.c[2] | s.c[3]) == TTTGeo<NP>::CELLMASK);
}
// cells of absolute player p (observation / export side): the word (p - mover) mod NP
template <int NP>
__device__ __forceinline__ uint32_t ttt_cells_of(const TTTEnv &s, int p) {
    int j = p - s.mover;
    j += j < 0 ? NP : 0;
    uint32_t r = 0;
#pragma unroll
    for (int q = 0; q < NP; q++) r |= (q == j) ? s.c[q] : 0u;
    return r;
}

// next_state (tictactoe_2p_env.py:283-315).  action: C-order flat cell index, negative = '' (pass).
template <int NP>
__device__ __forceinline__ void ttt_step_env(TTTEnv &s, int action, TTTOut &o) {
    constexpr uint32_t CELLMASK = TTTGeo<NP>::CELLMASK;
    uint32_t occ = s.c[0] | s.c[1] | s.c[2] | s.c[3];
    o.nvalid = __popc(~occ & CELLMASK);
    const bool in_range = (unsigned)action < (unsigned)TTTGeo<NP>::CELLS;
    const uint32_t bit = in_range ? (1u << action) : 0u;
    const bool cell_free = in_range && !(occ & bit);                 // is_valid_action (:350-380)
    const bool placed = cell_free && s.winner1 == 0;                 // :293
    o.error = (action >= 0 && !cell_free) ? 1 : 0;                   // invalid action: silent no-op in the reference
    o.placed = placed;
    uint32_t mine = s.c[0];                                          // the mover's cells are word 0
    if (placed) {
        mine |= bit;                                                 // :295
        if (TTTGeo<NP>::win(mine)) s.winner1 = s.mover + 1;          // :297-300
        occ |= bit;
    }
    o.reward = 0; o.terminal = 0; o.winners = 0;
    if (s.winner1) {                                                 // :302-308 (winner persists in the state)
        o.reward = (s.winner1 - 1 == s.mover) ? 1 : -1;
        o.winners = 1 << (s.winner1 - 1);
        o.terminal = 1;
    }
    if (occ == CELLMASK) o.terminal = 1;                             // :310-311 draw / full board
    o.valid_after = ~occ & CELLMASK;
    // the turn passes (:313): every word moves one seat closer to the move, the old mover goes to the back
#pragma unroll
    for (int j = 0; j + 1 < NP; j++) s.c[j] = s.c[j + 1];
    s.c[NP - 1] = mine;
    s.mover = (s.mover + 1 == NP) ? 0 : s.mover + 1;
    s.ep_len += 1;
}

// result record, 4 bytes: int8 reward | u8 flags (1 terminal, 2 invalid action, 4 placed) | u8 winners mask |
// u8 ranking bits (bit p = rank of player p: winners 0, everybody else 1 -- BaseEnvironment.py:173-195)
template <int NP>
__device__ __forceinline__ uint32_t ttt_pack_result(const TTTOut &o) {
    uint32_t rank = ((1u << NP) - 1u) & ~(uint32_t)o.winners;
    return ((uint32_t)o.reward & 0xffu) | (uint32_t)(o.terminal | o.error << 1 | o.placed << 2) << 8 |
           (uint32_t)o.winners << 16 | rank << 24;
}

// Episode statistics: every thread ACCUMULATES the packed counters of up to TTT_ACC_MAX env-steps in four registers
// (a handful of instructions per env-step), then the warp reduces them once (4 redux.sync), lane l < 15 extracts
// counter l from the warp-uniform sums and adds it to the CTA's shared partial -- ONE atomic instruction per warp and
// flush -- and the CTA adds its partial to its row of the global buffer once.  (The first version reduced and
// flushed after every env-step with two barriers: 40 % of the step kernel's time.)
//   A: steps | episodes << 8 | episodes without winner << 16 | illegal actions << 24       (sums <= 32 * 4 = 128)
//   W: wins per seat, 8 bits each.    The "not a winner" counters follow: rank[q] = episodes - wins[q]
//   D: valid-action count (12 bits: <= 27 * 128) | episode length of finished episodes << 12 (<= 31 * 128)
//   R: (mover + 1) * reward, biased by +4 per env-step (<= 8 * 128)
//   lane constants: word (0..3) | shift << 4 | bits << 10 | slot << 16 | kind << 24 (1: episodes - x, 2: x - 4 * steps)
#define TTT_ACC_MAX 4
#ifndef TTT_DBG
#define TTT_DBG 0
#endif
// where a warp's statistics sums go: 1 = straight to the CTA's row of the global buffer (fire-and-forget RED.64, no
// shared partial, no barriers), 0 = a shared partial per CTA + two barriers + one flush per CTA (round 1).  Measured
// (us per 1,048,576-env step, 4 chains / 1 chain): next_state 6.92 / 9.65 against 7.85 / 11.59 -> global; fused rollout
// 8.88 / 13.79 against 8.97 / 12.65 -> shared (its flush sits before the state store of the last step)
#ifndef TTT_STATS_GLOBAL_STEP
#define TTT_STATS_GLOBAL_STEP 1
#endif
#ifndef TTT_STATS_GLOBAL_ROLLOUT
#define TTT_STATS_GLOBAL_ROLLOUT 0
#endif
#define TTT_ROLLOUT_MINB 8     // default register budget of the fused rollout kernel (see its template parameter)
#define TTT_SL(word, shift, bits, slot, kind) ((word) | (shift) << 4 | (bits) << 10 | (slot) << 16 | (kind) << 24)
__constant__ uint32_t TTT_STAT_LANE[32] = {
    TTT_SL(0, 0, 8, ST_STEPS, 0), TTT_SL(0, 8, 8, ST_EPISODES, 0), TTT_SL(0, 16, 8, ST_NOWIN, 0), TTT_SL(0, 24, 8, ST_ERRORS, 0),
    TTT_SL(1, 0, 8, ST_WINS + 0, 0), TTT_SL(1, 8, 8, ST_WINS + 1, 0), TTT_SL(1, 16, 8, ST_WINS + 2, 0), TTT_SL(1, 24, 8, ST_WINS + 3, 0),
    TTT_SL(1, 0, 8, ST_RANK + 0, 1), TTT_SL(1, 8, 8, ST_RANK + 1, 1), TTT_SL(1, 16, 8, ST_RANK + 2, 1), TTT_SL(1, 24, 8, ST_RANK + 3, 1),
    TTT_SL(2, 0, 12, ST_NVALID, 0), TTT_SL(2, 12, 12, ST_EPLEN, 0), TTT_SL(3, 0, 12, ST_REWARD, 2),
    0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
#define TTT_STAT_LANES 15

struct TTTStatAcc {
    uint32_t A, W, D, R;
    __device__ __forceinline__ void clear() { A = W = D = R = 0u; }
    // fused rollout: its rewards are accumulated without the +4 bias per env-step that flush() removes
    __device__ __forceinline__ void bias_from_steps() { R += 4u * (A & 255u); }
    // one env-step of a live thread
    template <int NP>
    __device__ __forceinline__ void add(const TTTOut &o, int mover, uint32_t ep_len) {
        const uint32_t t = o.terminal ? 1u : 0u;
        const uint32_t w = t ? (uint32_t)o.winners : 0u;
        A += 1u | t << 8 | (t & (uint32_t)(o.winners == 0)) << 16 | (uint32_t)o.error << 24;
        W += (w * 0x00204081u) & 0x01010101u;                               // bit q -> byte q
        D += (uint32_t)o.nvalid | (t ? min(ep_len, 31u) : 0u) << 12;
        R += (uint32_t)((mover + 1) * o.reward + 4);
    }
    // warp-collective: reduce, extract, add to the CTA's shared partial, clear
    template <int NP, bool GLOBAL>
    __device__ __forceinline__ void flush(int *sm_stat, uint32_t lane_const, crl_u64 *row) {
        const uint32_t a = __reduce_add_sync(0xffffffffu, A), w = __reduce_add_sync(0xffffffffu, W);
        const uint32_t d = __reduce_add_sync(0xffffffffu, D), r = __reduce_add_sync(0xffffffffu, R);
#ifndef TTT_FLUSH_BRANCHY
        // branch-free: the word by two selects on its two index bits, the field by shift + mask, the two derived kinds
        // by selects (the first version compiled to a chain of branches around moves)
        const uint32_t lo = (lane_const & 1u) ? w : a, hi = (lane_const & 1u) ? r : d;
        const uint32_t x = (lane_const & 2u) ? hi : lo;
        int val = (int)((x >> ((lane_const >> 4) & 31u)) & ((1u << ((lane_const >> 10) & 31u)) - 1u));
        const uint32_t kind = lane_const >> 24;
        const int notwin = ((lane_const >> 7) & 7u) < (uint32_t)NP ? (int)((a >> 8) & 255u) - val : 0;       // not-a-winner, seats < NP
        val = kind == 1u ? notwin : val;
        val -= kind == 2u ? 4 * (int)(a & 255u) : 0;                        // remove the reward bias
#else
        const uint32_t word = lane_const & 15u;
        const uint32_t x = word == 0u ? a : word == 1u ? w : word == 2u ? d : r;
        int val = (int)((x >> ((lane_const >> 4) & 31u)) & ((1u << ((lane_const >> 10) & 31u)) - 1u));
        const uint32_t kind = lane_const >> 24;
        if (kind == 1u) val = ((lane_const >> 7) & 7u) < (uint32_t)NP ? (int)((a >> 8) & 255u) - val : 0;
        if (kind == 2u) val -= 4 * (int)(a & 255u);
#endif
        const int slot = (int)((lane_const >> 16) & 255u);
        if ((int)(threadIdx.x & 31) < TTT_STAT_LANES && val != 0) {
            if (GLOBAL) atomicAdd(&row[slot], (crl_u64)(long long)val);
            else atomicAdd(&sm_stat[slot], val);
        }
        clear();
    }
};

__device__ __forceinline__ void ttt_zero_out(TTTOut &o) {
    o.reward = o.terminal = o.error = o.placed = o.winners = o.nvalid = 0; o.valid_after = 0;
}

// Grid-stride: the launcher sizes the grid so that a thread steps at most TTT_ACC_MAX environments.
template <int NP>
__global__ void __launch_bounds__(256, 8)
ttt_step_kernel(const uint4 *__restrict__ in, uint4 *__restrict__ out, const int8_t *__restrict__ actions,
                uint32_t *__restrict__ result, uint32_t *__restrict__ valid_after, crl_u64 *stats, long long B,
                int flags) {
    __shared__ int sm_stat[CRL_NSTAT];
    if (stats && !TTT_STATS_GLOBAL_STEP) { if (threadIdx.x < CRL_NSTAT) sm_stat[threadIdx.x] = 0; __syncthreads(); }
    crl_u64 *const row = stats ? stats + (blockIdx.x & (CRL_STAT_ROWS - 1)) * CRL_NSTAT : nullptr;
    TTTStatAcc acc;
    acc.clear();
    const long long stride = (long long)gridDim.x * blockDim.x;
    // (PDL launch: the grid may become resident while its predecessor drains; an L2 prefetch prologue like Tron's was
    // measured and dropped -- this kernel is issue-bound and the extra instructions cost more than the overlap buys)
    pdl_wait();
    pdl_launch_dependents();
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < B; e += stride) {
        TTTEnv s;
        TTTOut o;
        ttt_decode(s, ld_stream(in + e));
        if ((flags & CRL_FLAG_AUTO_RESET) && ttt_is_terminal<NP>(s)) ttt_new_state(s);
        const int mover = s.mover;
        ttt_step_env<NP>(s, (int)actions[e], o);
        st_stream(out + e, ttt_encode(s));
        if (flags & CRL_FLAG_COMPACT_RESULT)         // 1-byte record: flags | (winner + 1) << 3 | the player who moved << 6
            ((uint8_t *)result)[e] = (uint8_t)((o.terminal | o.error << 1 | o.placed << 2) | s.winner1 << 3 | mover << 6);
        else
            result[e] = ttt_pack_result<NP>(o);
        if (valid_after) valid_after[e] = o.valid_after;
        if (stats) acc.add<NP>(o, mover, s.ep_len);
    }
    if (stats) {
        acc.flush<NP, TTT_STATS_GLOBAL_STEP != 0>(sm_stat, TTT_STAT_LANE[threadIdx.x & 31], row);
        if (!TTT_STATS_GLOBAL_STEP) {
            __syncthreads();
            stats_flush_row(sm_stat, stats);
        }
    }
}

// One-hot mask of the k-th (0-based) set bit of a <= 27-bit mask: binary search on popcounts, written so that only
// TWO instructions per level use the ALU pipe (the binding pipe of the fused rollout kernel,
// profiles/r02_ttt_rollout_full.md): the search window is a constant times the running one-hot position (IMAD, FMA
// pipe), the count is a POPC (XU pipe), and the updates are predicated IMADs.  (The first version -- shift the mask
// down, SEL the three values -- spent 5 ALU instructions per level plus a final 1 << pos.)
__device__ __forceinline__ uint32_t ttt_kth_bit_onehot(uint32_t mask, uint32_t k) {
    uint32_t bit = 1u;
#ifndef CRL_HOSTSIM
#define TTT_KTH_LEVEL(WIN, MUL)                                                                                          \
    "mul.lo.u32 t, %0, " WIN ";\n\tand.b32 t, t, %2;\n\tpopc.b32 c, t;\n\tsetp.ge.u32 p, %1, c;\n\t"                      \
    "@p sub.u32 %1, %1, c;\n\t@p mul.lo.u32 %0, %0, " MUL ";\n\t"
    asm("{\n\t.reg .pred p;\n\t.reg .u32 c, t;\n\t"
        TTT_KTH_LEVEL("0xffff", "0x10000") TTT_KTH_LEVEL("0xff", "0x100") TTT_KTH_LEVEL("0xf", "0x10")
        TTT_KTH_LEVEL("0x3", "0x4") TTT_KTH_LEVEL("0x1", "0x2")
        "}" : "+r"(bit), "+r"(k) : "r"(mask));
#undef TTT_KTH_LEVEL
#else
    for (uint32_t w = 16; w >= 1; w >>= 1) {
        const uint32_t c = (uint32_t)__popc(mask & (((1u << w) - 1u) * bit));
        if (k >= c) { k -= c; bit <<= w; }
    }
#endif
    return bit;
}

// Exact r % n for n <= 27 without the generic 32-bit division (~20 instructions): lane l holds floor(2^32 / l), a
// shuffle fetches the entry of the lane's own n, q' = umulhi(r, M[n]) is the quotient or one less, one correction.
// (n = 1: M = 2^32 - 1, q' = r - 1, the correction gives 0.)  Warp-collective: call with all lanes.
__device__ const uint32_t TTT_RCP_G[32] = {      // floor(2^32 / l); l < 2: 2^32 - 1   (global: one coalesced load per warp)
    0xffffffffu, 0xffffffffu, 0x80000000u, 0x55555555u, 0x40000000u, 0x33333333u, 0x2aaaaaaau, 0x24924924u,
    0x20000000u, 0x1c71c71cu, 0x19999999u, 0x1745d174u, 0x15555555u, 0x13b13b13u, 0x12492492u, 0x11111111u,
    0x10000000u, 0x0f0f0f0fu, 0x0e38e38eu, 0x0d79435eu, 0x0cccccccu, 0x0c30c30cu, 0x0ba2e8bau, 0x0b21642cu,
    0x0aaaaaaau, 0x0a3d70a3u, 0x09d89d89u, 0x097b425eu, 0x09249249u, 0x08d3dcb0u, 0x08888888u, 0x08421084u};
__device__ __forceinline__ uint32_t ttt_rcp_lane() { return TTT_RCP_G[threadIdx.x & 31u]; }
__device__ __forceinline__ uint32_t ttt_mod_small(uint32_t r, uint32_t n, uint32_t rcp_lane) {
    const uint32_t m = __shfl_sync(0xffffffffu, rcp_lane, (int)n);
    uint32_t rem = r - __umulhi(r, m) * n;
#ifndef CRL_HOSTSIM
    asm("{\n\t.reg .pred p;\n\tsetp.ge.u32 p, %0, %1;\n\t@p sub.u32 %0, %0, %1;\n\t}" : "+r"(rem) : "r"(n));   // (a predicated IMAD, not a SEL)
    return rem;
#else
    return rem >= n ? rem - n : rem;
#endif
}

// uniform random policy: the (r0 % n_empty)-th empty cell in C order, pass (-1) if the board is full
// (warp-collective because of ttt_mod_small)
template <int NP>
__device__ __forceinline__ int ttt_random_action(const TTTEnv &s, uint32_t r0, uint32_t rcp_lane) {
    uint32_t empty = ~(s.c[0] | s.c[1] | s.c[2] | s.c[3]) & TTTGeo<NP>::CELLMASK;
    const int n = __popc(empty);
    const uint32_t k = ttt_mod_small(r0, (uint32_t)max(n, 1), rcp_lane);
    return n ? 31 - __clz((int)ttt_kth_bit_onehot(empty, k)) : -1;
}

template <int NP>
__global__ void ttt_policy_random_kernel(const uint4 *__restrict__ st, int8_t *__restrict__ actions, long long B,
                                         int flags, crl_u64 seed, crl_u64 first_env, uint32_t step) {
    long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = e < B;
    TTTEnv s;
    ttt_new_state(s);
    if (valid) ttt_decode(s, st[e]);
    if ((flags & CRL_FLAG_AUTO_RESET) && ttt_is_terminal<NP>(s)) ttt_new_state(s);
    uint4 r = env_words(seed, first_env + (crl_u64)e, step, CRL_TAG_TTT);
    const int a = ttt_random_action<NP>(s, r.x, ttt_rcp_lane());
    if (valid) actions[e] = (int8_t)a;
}

// ---- fused random-policy step on the RAW state words (mover-relative layout, fields in the top five bits of x / y).
// A non-terminal board has an empty cell and no winner, so the chosen cell is always free and always placed:
// next_state (tictactoe_2p_env.py:283-315) without its validity branches, sharing the empty mask with the policy.
// Written against the ALU pipe: the cells are never masked out of their words (the win test only shifts LEFT and ends
// with an AND against masks inside the cell bits, so the field bits above them cannot reach it), the move is
// x |= bit, the turn passes by renaming the four words, and the field updates are adds of disjoint bit ranges (IMAD).
struct TTTFusedOut {
    uint32_t win, terminal;      // 0 / 1
    uint32_t mover, n;           // the player who moved, number of empty cells before the move
    uint32_t ep_top;             // new (saturated) episode length << 27
};

template <int NP>
__device__ __forceinline__ void ttt_policy_step_raw(uint4 &v, uint32_t empty, uint32_t r0, uint32_t rcp_lane, TTTFusedOut &o) {
    constexpr uint32_t CM = 0x07ffffffu;                 // the cell bits of a word (the fields sit above, whatever NP)
    const uint32_t n = (uint32_t)__popc(empty);          // >= 1
    const uint32_t bit = ttt_kth_bit_onehot(empty, ttt_mod_small(r0, n, rcp_lane));
    const uint32_t mine = v.x | bit;                     // raw: mover in bits 27..28, winner bits zero
    const bool win = TTTGeo<NP>::win(mine) != 0u;
    const uint32_t mover = v.x >> 27;
    const uint32_t t1 = mover + 1u;
    uint32_t f0 = (NP == 4 ? (t1 & 3u) : (t1 == (uint32_t)NP ? 0u : t1)) << 27;           // next mover
    uint32_t top1 = v.y & ~CM;                           // episode length, saturating at 31
#ifndef CRL_HOSTSIM
    asm("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %1, 0;\n\t@p mad.lo.u32 %0, %2, 0x20000000, %0;\n\t}" : "+r"(f0) : "r"((uint32_t)win), "r"(t1));
    asm("{\n\t.reg .pred p;\n\tsetp.lt.u32 p, %0, 0xf8000000;\n\t@p add.u32 %0, %0, 0x08000000;\n\t}" : "+r"(top1));
#else
    if (win) f0 += t1 << 29;
    if (top1 < 0xf8000000u) top1 += 0x08000000u;
#endif
    o.win = win ? 1u : 0u;
    o.terminal = (win || empty == bit) ? 1u : 0u;
    o.mover = mover; o.n = n; o.ep_top = top1;
    const uint32_t back = mine & CM;                     // the mover's cells go to the back of the queue
    if (NP == 4) v = make_uint4((v.y & CM) | f0, v.z + top1, v.w, back);
    else if (NP == 3) v = make_uint4((v.y & CM) | f0, v.z + top1, back, 0u);
    else v = make_uint4((v.y & CM) | f0, back + top1, 0u, 0u);
}

// result record of a fused step (reward = 1 for a winning move, the winner is the mover)
template <int NP>
__device__ __forceinline__ uint32_t ttt_fused_result(const TTTFusedOut &o) {
    const uint32_t wm = o.win << o.mover;                                   // winners mask
    return o.win | (o.terminal | 4u) << 8 | wm << 16 | ((((1u << NP) - 1u) ^ wm) << 24);
}

// episode statistics of a fused step into the packed counters of TTTStatAcc; the reward bias the flush removes is
// added once per flush (TTTStatAcc::bias_from_steps)
// acc += v if cond (0 / 1): a predicated add (FMA pipe) instead of SEL + add (the compiler's choice for `c ? v : 0`)
__device__ __forceinline__ void ttt_add_if(uint32_t &acc, uint32_t cond, uint32_t v) {
#ifndef CRL_HOSTSIM
    asm("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %1, 0;\n\t@p add.u32 %0, %0, %2;\n\t}" : "+r"(acc) : "r"(cond), "r"(v));
#else
    if (cond) acc += v;
#endif
}
__device__ __forceinline__ void ttt_fused_stats(TTTStatAcc &acc, const TTTFusedOut &o) {
    acc.A += 1u;                                                            // steps
    ttt_add_if(acc.A, o.terminal, 0x10100u);                                // episodes << 8 | episodes without a winner << 16
    ttt_add_if(acc.A, o.win, 0u - 0x10000u);                                // ... a win is not one of those (win => terminal)
    ttt_add_if(acc.W, o.win, 1u << (8u * o.mover));                         // wins per seat, one byte each
    acc.D += o.n;                                                           // valid-action count
    ttt_add_if(acc.D, o.terminal, o.ep_top >> 15);                          // episode length << 12 (ep_top has bits 27..31 only)
    ttt_add_if(acc.R, o.win, o.mover + 1u);                                 // (mover + 1) * reward
}

// K fused random-policy steps with auto-reset; grid-stride like the step kernel (a thread owns <= TTT_ACC_MAX
// environments and keeps one of them in registers for the K steps).  STATS is a template parameter (no per-iteration
// pointer tests), the batch index is 32-bit (the launcher refuses B >= 2^31), MINB = resident CTAs per SM the register
// allocation aims at (8: 32 registers; 6: 40 registers, the Philox keys and pointers stay in registers).
template <int NP, bool STATS, int MINB>
__global__ void __launch_bounds__(256, MINB)
ttt_rollout_kernel(uint4 *__restrict__ state, uint32_t *__restrict__ result, crl_u64 *stats, int B,
                   const PhiloxKeys keys, crl_u64 first_env, uint32_t step0, int K) {
    // TTT_DBG (compile-time, timing attribution only -- statistics are wrong with any bit set): 1 no per-step
    // accumulation, 2 no warp flush, 4 no CTA flush.  Measured (us per 1,048,576-env step, 4 chains): 9.30 full, 8.75 / 8.85 /
    // 9.21 without one of the three, 8.30 without all, 7.45 with STATS = false
    constexpr int dbg = TTT_DBG;
    constexpr uint32_t CM = TTTGeo<NP>::CELLMASK;
    __shared__ int sm_stat[CRL_NSTAT];
    if (STATS && !TTT_STATS_GLOBAL_ROLLOUT) { if (threadIdx.x < CRL_NSTAT) sm_stat[threadIdx.x] = 0; __syncthreads(); }
    crl_u64 *const row = STATS ? stats + (blockIdx.x & (CRL_STAT_ROWS - 1)) * CRL_NSTAT : nullptr;
    const uint32_t lane_const = TTT_STAT_LANE[threadIdx.x & 31], rcp_lane = ttt_rcp_lane();
    TTTStatAcc acc;
    acc.clear();
    int pending = 0;                                     // env-steps accumulated since the last flush (block-uniform)
    const int stride = (int)(gridDim.x * blockDim.x), first = (int)(blockIdx.x * blockDim.x);
    pdl_wait();
    pdl_launch_dependents();
    for (int e0 = first; e0 < B; e0 += stride) {         // block-uniform trip count: the flushes are warp-collective
        const int e = e0 + (int)threadIdx.x;
        const bool valid = e < B;
        uint4 v = make_uint4(0u, 0u, 0u, 0u);            // (lanes past the end of the batch step a dummy board)
        if (valid) v = ld_stream(state + e);
        TTTFusedOut o;
        o.win = o.terminal = o.mover = o.n = o.ep_top = 0u;
        const crl_u64 ge = first_env + (crl_u64)(uint32_t)e;
        for (int k = 0; k < K; k++) {
            uint32_t empty = ~(v.x | v.y | v.z | v.w) & CM;
            if (v.x >= 0x20000000u || empty == 0u) {     // terminal (a winner, or a full board): new_state
                v = make_uint4(0u, 0u, 0u, 0u);
                empty = CM;
            }
            const uint32_t r0 = philox4x32_10_x((uint32_t)ge, (uint32_t)(ge >> 32), step0 + (uint32_t)k, CRL_TAG_TTT, keys);
            ttt_policy_step_raw<NP>(v, empty, r0, rcp_lane, o);
            if (STATS) {
                if (valid && !(dbg & 1)) ttt_fused_stats(acc, o);
                if (++pending == TTT_ACC_MAX && !(dbg & 2)) {
                    acc.bias_from_steps();
                    acc.flush<NP, TTT_STATS_GLOBAL_ROLLOUT != 0>(sm_stat, lane_const, row);
                    pending = 0;
                }
            }
        }
        if (valid) {
            st_stream(state + e, v);
            if (result) result[e] = ttt_fused_result<NP>(o);
        }
    }
    if (STATS && !(dbg & 4)) {
        if (pending && !(dbg & 2)) { acc.bias_from_steps(); acc.flush<NP, TTT_STATS_GLOBAL_ROLLOUT != 0>(sm_stat, lane_const, row); }
        if (!TTT_STATS_GLOBAL_ROLLOUT) {
            __syncthreads();
            stats_flush_row(sm_stat, stats);
        }
    }
}

__global__ void ttt_reset_kernel(uint4 *__restrict__ state, const uint8_t *__restrict__ mask, long long B) {
    long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= B || (mask && !mask[e])) return;
    state[e] = make_uint4(0, 0, 0, 0);
}

// valid_actions (tictactoe_2p_env.py:317-348): bit c set = cell c (C order) is empty; 0 <=> ['']
__global__ void ttt_valid_kernel(const uint4 *__restrict__ st, uint32_t *__restrict__ mask, long long B, TTTParams prm) {
    long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= B) return;
    uint4 v = st[e];
    mask[e] = ~(v.x | v.y | v.z | v.w) & prm.cellmask;
}

// state_to_observation (2p :382-407).  A warp unpacks 32 environments.  Lane = environment: the viewer-relative label
// of every player's cells (absolute: p; else (p - viewer) mod 2 for 2p, mod 3 for 3p AND 4p -- tictactoe_4p_env.py:50)
// is folded into two label bit-planes + the occupancy plane, four cells at a time are spread to bytes with one
// multiply each ((nibble * 0x00204081) & 0x01010101: bit i -> byte i) and combined into a word of int8 cells
// (-1 = empty), which goes to the lane's CELLS-byte slot of the warp's staging tile.  The tile (32 * CELLS bytes,
// contiguous in the output and 16-byte aligned) then leaves with 128-bit stores.
// player == -1: absolute; -2: each game seen by its current mover (CRL_PLAYER_MOVER).
// board int8[B][cells] (-1 empty); winner int8[B] (-1 None); mover int8[B].
template <int NP>
__global__ void __launch_bounds__(256)
ttt_observe_kernel(const uint4 *__restrict__ st, long long B, int player, int8_t *__restrict__ board,
                   int8_t *__restrict__ winner, int8_t *__restrict__ mover) {
    constexpr int CELLS = TTTGeo<NP>::CELLS, GROUPS = (CELLS + 3) / 4, MOD = NP == 2 ? 2 : 3;
    constexpr int TILE = 32 * CELLS;                         // 288 / 480 / 864: multiples of 16
    __shared__ __align__(16) uint8_t stage[8][TILE + 16];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const long long e0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) & ~31ll;      // first environment of the warp
    if (e0 >= B) return;
    const long long e = e0 + lane;
    TTTEnv s;
    ttt_new_state(s);
    if (e < B) {
        ttt_decode(s, ld_stream(st + e));
        if (winner) winner[e] = (int8_t)(s.winner1 - 1);
        if (mover) mover[e] = (int8_t)s.mover;
    }
    const int viewer = player == -2 ? s.mover : player;
    uint32_t b0 = 0u, b1 = 0u;
#pragma unroll
    for (int j = 0; j < NP; j++) {                           // word j = player (mover + j) % NP
        int p = s.mover + j;
        p -= p >= NP ? NP : 0;
        // ((p - viewer) mod MOD) for p - viewer in -3..3 from a 2-bit-per-entry constant (no integer modulo per lane)
        const int code = viewer < 0 ? p : (int)(((MOD == 3 ? 0x924u : 0x110u) >> (2 * (p - viewer + 3))) & 3u);
        b0 |= (code & 1) ? s.c[j] : 0u;
        b1 |= (code & 2) ? s.c[j] : 0u;
    }
    const uint32_t emp = ~(s.c[0] | s.c[1] | s.c[2] | s.c[3]);
    uint8_t *mine = stage[wid] + lane * CELLS;
#pragma unroll
    for (int j = 0; j < GROUPS; j++) {
        const uint32_t x0 = (((b0 >> (4 * j)) & 15u) * 0x00204081u) & 0x01010101u;
        const uint32_t x1 = (((b1 >> (4 * j)) & 15u) * 0x00204081u) & 0x01010101u;
        const uint32_t xe = (((emp >> (4 * j)) & 15u) * 0x00204081u) & 0x01010101u;
        const uint32_t word = x0 + 2u * x1 + 255u * xe;      // empty cells have no label bits: 0xff = -1
#pragma unroll
        for (int i = 0; i < 4; i++)
            if (4 * j + i < CELLS) mine[4 * j + i] = (uint8_t)(word >> (8 * i));
    }
    __syncwarp();
    int8_t *dst = board + e0 * CELLS;
    if (B - e0 >= 32) {
        const uint4 *src4 = (const uint4 *)stage[wid];
        for (int i = lane; i < TILE / 16; i += 32) ((uint4 *)dst)[i] = src4[i];
    } else {
        const int nbytes = (int)(B - e0) * CELLS;
        for (int i = lane; i < nbytes; i += 32) dst[i] = (int8_t)stage[wid][i];
    }
}

__global__ void ttt_pack_kernel(uint4 *__restrict__ st, long long B, TTTParams prm, const int8_t *__restrict__ board,
                                const int8_t *__restrict__ winner, const int8_t *__restrict__ mover) {
    long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= B) return;
    TTTEnv s;
    ttt_new_state(s);
    s.winner1 = winner[e] + 1;
    s.mover = mover[e];
    for (int c = 0; c < prm.cells; c++) {
        const int v = board[e * prm.cells + c];
        int j = v - s.mover;                                 // player v sits in word (v - mover) mod n
        j += j < 0 ? prm.n : 0;
#pragma unroll
        for (int q = 0; q < 4; q++) s.c[q] |= (v >= 0 && q == j) ? (1u << c) : 0u;
    }
    st[e] = ttt_encode(s);
}

// ---- one learner against uniform random opponents (crl_ttt_advance; the rule is stated in
// include/colosseum_b200_learner.h).  One thread per environment, grid-stride with a block-uniform trip count like the
// rollout kernel, because the statistics flushes are warp-collective.  Every lane runs the same 2NP - 2 opponent
// slots; slot j is active while the game's mover is not `seat` (a game is restarted as soon as a move ends it, so the
// active slots are exactly the first j and their index is the opponent move index of the rule).  The pick is a plain
// `%`: ttt_mod_small shuffles, and the active slots of the lanes differ.
//   Statistics bound (the packed fields of TTTStatAcc, 32 lanes per flush): an environment is at most 2NP - 1
//   env-steps (the learner's move and 2NP - 2 opponent moves), each with nvalid <= CELLS, with at most one finished
//   episode.  Flushed once per environment, the 12-bit nvalid field would hold up to 32 x 27 x 7 = 6048 for NP = 4,
//   so 4-player flushes twice: after the learner's move and slots 0..2 (<= 4 env-steps: nvalid <= 3456, steps <= 128,
//   reward + bias <= 8 x 128) and after slots 3..5 (<= 3).  NP = 3 (<= 5 env-steps: nvalid <= 2400) and NP = 2
//   (<= 3: 864) flush once.  Episodes, wins and episode lengths (<= 31 x 32) are bounded by one episode per lane.
template <int NP, bool STATS>
__global__ void __launch_bounds__(256)
ttt_advance_kernel(uint4 *__restrict__ state, const int8_t *__restrict__ actions, int seat, uint32_t *__restrict__ result,
                   uint32_t *__restrict__ valid_after, crl_u64 *stats, int B, crl_u64 seed, crl_u64 first_env,
                   uint32_t step) {
    constexpr int SLOTS = 2 * NP - 2;
    crl_u64 *const row = STATS ? stats + (blockIdx.x & (CRL_STAT_ROWS - 1)) * CRL_NSTAT : nullptr;
    const uint32_t lane_const = TTT_STAT_LANE[threadIdx.x & 31];
    TTTStatAcc acc;
    acc.clear();
    // unsigned: B < 2^31 and stride < 2^31, so e0 + stride stays below 2^32 at the last trip
    const uint32_t stride = gridDim.x * blockDim.x, first = blockIdx.x * blockDim.x;
    for (uint32_t e0 = first; e0 < (uint32_t)B; e0 += stride) {
        const uint32_t e = e0 + threadIdx.x;
        const bool valid = e < (uint32_t)B;
        TTTEnv s;
        ttt_new_state(s);
        if (valid) ttt_decode(s, ld_stream(state + e));
        if (ttt_is_terminal<NP>(s)) ttt_new_state(s);                    // 1. it ended in an earlier call
        uint32_t flags = 0u, winners = 0u;
        int reward = 0, j = 0;
        TTTOut o;
        ttt_zero_out(o);
        // a move that ended the game: record it for the learner, restart
        auto finish = [&]() {
            flags |= 1u;
            winners = (uint32_t)o.winners;
            reward = s.winner1 == 0 ? 0 : (s.winner1 - 1 == seat ? 1 : -1);
            ttt_new_state(s);
        };
        if (actions && s.mover == seat) {                                // 2. the learner's move
            ttt_step_env<NP>(s, valid ? (int)actions[e] : -1, o);
            flags |= (uint32_t)(o.error << 1 | o.placed << 2);
            if (STATS && valid) acc.add<NP>(o, seat, s.ep_len);
            if (o.terminal) finish();
        } else {
            flags |= 8u;
        }
        uint4 w = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
        for (int k = 0; k < SLOTS; k++) {                                // 3. the opponents
            if (STATS && NP == 4 && k == NP - 1) acc.flush<NP, true>(nullptr, lane_const, row);
            if (s.mover != seat) {
                if ((k & 3) == 0) w = env_words(seed, first_env + (crl_u64)e, step, CRL_TAG_OPPONENT + (uint32_t)(k >> 2));
                const uint32_t r = (k & 3) == 0 ? w.x : (k & 3) == 1 ? w.y : (k & 3) == 2 ? w.z : w.w;
                const uint32_t empty = ~(s.c[0] | s.c[1] | s.c[2] | s.c[3]) & TTTGeo<NP>::CELLMASK;   // non-terminal: >= 1
                const int mover = s.mover;
                ttt_step_env<NP>(s, 31 - __clz((int)ttt_kth_bit_onehot(empty, r % (uint32_t)__popc(empty))), o);
                if (STATS && valid) acc.add<NP>(o, mover, s.ep_len);
                if (o.terminal) finish();
                j++;
            }
        }
        if (STATS) acc.flush<NP, true>(nullptr, lane_const, row);
        if (valid) {
            st_stream(state + e, ttt_encode(s));
            result[e] = ((uint32_t)reward & 0xffu) | flags << 8 | winners << 16 | (uint32_t)j << 24;
            if (valid_after) valid_after[e] = ~(s.c[0] | s.c[1] | s.c[2] | s.c[3]) & TTTGeo<NP>::CELLMASK;
        }
    }
}
