// Tron: batched grid movement + collision + rewards/terminal/winners/ranking in ONE kernel (sm_100a).
//
// Replaces (reference file:line):
//   next_state_inplace            envs/tron/CyTronGrid.pyx:3-62
//   TronGridEnvironment.next_state envs/tron/TronGridEnvironment.py:265-323  (alive set, rewards, terminal, winners)
//   TronGridEnvironment.compute_ranking :483-508                            (fused; incl. the deaths[-1] wrap-around)
//   TronGridEnvironment.new_state :228-263                                  (tron_reset_kernel / auto-reset)
//   state_to_observation :363-405 + relative_player_inplace CyTronGrid.pyx:65-71 (tron_observe_kernel)
//
// HBM layout (SoA of 16-byte vectors, [13][B] uint4, 208 B per environment, of which 160 B are moved by a step):
//   A cell holds its owner code: 0 empty, q + 1 for player q.  The code is stored in binary, one 384-bit plane per bit:
//     plane c0 = players 0 and 2 (codes 1, 3), c1 = players 1 and 2 (codes 2, 3), c2 = player 3 (code 4)
//   vector v = 3*k + j (k = code bit-plane 0..2, j = 0..2): 32-bit words 4j..4j+3 of plane k,
//             bit (y*N + x) of the plane is bit k of the owner code of cell (x, y)   (N*N <= 384, N <= 19)
//   vectors 9..11 = reserved: always zero (reset, pack and an out-of-place step write zeros; the step and rollout
//             kernels never read them), so two states holding the same game are equal byte for byte
//   vector 12 = header, one BYTE LANE per player so that the four players are advanced with 32-bit SWAR
//   arithmetic:
//     .x byte p = (head x + 1) | direction << 5          (coordinates are stored biased by one: 0 and N+1 are
//     .y byte p = (head y + 1) | deaths << 5              the off-grid columns / rows a move can reach)
//     .z = cells0 | cells1 << 9 | cells2 << 18 | terminal << 27      (#cells owned = compute_ranking's score)
//     .w = cells3 | episode steps << 9
//
// Data movement: vector v of the TILE environments of a CTA is ONE contiguous global segment (TILE*16 bytes), so
// the tile travels as one 2-D tensor copy of the 9 plane vectors plus one bulk copy of the header (TMA) issued by one
// thread into shared memory, and the same two copies back; the planes are never unpacked into registers.  Each thread
// owns one environment and only touches the <= 12 bitboard words its players move into plus the 16-byte header.
//
// The step is split in three phases so that only the middle one is exposed between the loads and the stores:
//   phase 1 (header + actions have landed, planes still in flight): new directions / target cells / addresses
//   phase 2 (planes have landed): 12 board lookups, the reference's player-order-sequential resolve, <= 4 bit sets;
//           then the 9 plane vectors are already on their way back to HBM
//   phase 3 (plane stores in flight): rewards / terminal / winners / ranking / header / result record / statistics
#pragma once
#include "crl_common.cuh"
#include "philox.cuh"

#define TRON_VEC 13          // 16-byte vectors per environment in a state buffer
#define TRON_PVEC 9          // vectors 0..8: the three owner-code bit-planes
#define TRON_HVEC 12         // vector 12: the header (9..11 reserved)
#define TRON_WORDS 6
#define TRON_ONES 0x01010101u

struct TronParams {
    int N, P;
    uint32_t pmask;                     // 0x01 in byte p for p < P
    uint32_t rkmask;                    // ranking bits of the present players: (1 << 2P) - 1
    uint32_t start_hdr[4];              // header of new_state()
    uint32_t spawn_word[4];             // 32-bit word (0..11) of a plane that holds player p's spawn cell
    uint32_t spawn_bit[4];              // ... and the bit inside it (0 for absent players)
};

// unpacked header (host code, import / observation kernels); the step kernels work on the packed words
struct TronHdr {
    int hx[4], hy[4], dir[4], death[4], cells[4];
    uint32_t terminal, ep_len;
};

// Register arrays are only ever indexed with compile-time constants; run-time selection is done with masks.
__device__ __forceinline__ int tron_sel4(const int (&a)[4], int k) {
    int r = 0;
#pragma unroll
    for (int i = 0; i < 4; i++) r |= a[i] & -(int)(k == i);
    return r;
}

__host__ __device__ __forceinline__ void tron_hdr_decode(TronHdr &s, uint4 h) {
    const uint32_t ce[4] = {h.z & 511u, (h.z >> 9) & 511u, (h.z >> 18) & 511u, h.w & 511u};
#pragma unroll
    for (int p = 0; p < 4; p++) {
        const uint32_t bx = (h.x >> (8 * p)) & 255u, by = (h.y >> (8 * p)) & 255u;
        s.hx[p] = (int)(bx & 31u) - 1; s.hy[p] = (int)(by & 31u) - 1;
        s.dir[p] = (int)(bx >> 5) & 3;
        s.death[p] = (int)(by >> 5);
        s.cells[p] = (int)ce[p];
    }
    s.terminal = (h.z >> 27) & 1u;
    s.ep_len = h.w >> 9;
}

__host__ __device__ __forceinline__ uint4 tron_hdr_encode(const TronHdr &s) {
    uint32_t x = 0, y = 0;
#pragma unroll
    for (int p = 0; p < 4; p++) {
        x |= ((uint32_t)(s.hx[p] + 1) | (uint32_t)s.dir[p] << 5) << (8 * p);
        y |= ((uint32_t)(s.hy[p] + 1) | (uint32_t)s.death[p] << 5) << (8 * p);
    }
    return make_uint4(x, y, (uint32_t)s.cells[0] | (uint32_t)s.cells[1] << 9 | (uint32_t)s.cells[2] << 18 | s.terminal << 27,
                      (uint32_t)s.cells[3] | s.ep_len << 9);
}

// ---- the shared-memory tile ---------------------------------------------------------------------------------
// rows 0..8 = the plane vectors 0..8 of the buffer, row 9 = its header vector 12 (the reserved vectors stay in HBM)
template <int TILE>
struct TronTile {
    uint4 v[TRON_PVEC + 1][TILE];
    static constexpr int PL = 3 * TILE * 4;     // distance in 32-bit words between the same word of two planes
    // 32-bit view of environment t: word j (0..11) of plane k is words(t)[woff(j) + k * PL]
    __device__ __forceinline__ uint32_t *words(int t) { return reinterpret_cast<uint32_t *>(&v[0][t]); }
    __device__ __forceinline__ static int woff(int j) { return (j >> 2) * (TILE * 4) + (j & 3); }
    __device__ __forceinline__ uint4 *hdr() { return &v[TRON_PVEC][0]; }
};

template <int TILE>
__device__ __forceinline__ void tron_cta_sync() {
    if (TILE == 32) __syncwarp(); else __syncthreads();
}

// Tensor maps of the [9][B*4] uint32 plane part of a state buffer (box = 9 rows x TILE*4 words): one for the
// buffer the step reads, one for the buffer it writes.  Built on the host per call (crl_api.cu).
struct TronMaps {
#ifndef CRL_HOSTSIM
    CUtensorMap in, out;
#else
    const uint4 *in_ptr;     // (SIMT emulator: plain pointers, the copies are cooperative loops)
    uint4 *out_ptr;
#endif
};

// global -> shared, two transactions: the header vector (barrier 0, one 1-D bulk copy) and the 9 plane vectors
// (barrier 1, one 2-D tensor copy when a map is given, else 9 bulk copies)
template <int TILE>
__device__ __forceinline__ void tron_tile_load_issue(TronTile<TILE> &tile, uint64_t *bar, const TronMaps *maps,
                                                     const uint4 *__restrict__ st, long long B, long long e0, int n) {
#ifndef CRL_HOSTSIM
    if (threadIdx.x == 0) {
        mbar_init(&bar[0], 1);
        mbar_init(&bar[1], 1);
        mbar_expect_tx(&bar[0], (uint32_t)(n * 16));
        bulk_g2s(tile.hdr(), st + TRON_HVEC * B + e0, (uint32_t)(n * 16), &bar[0]);
        if (maps) {
            mbar_expect_tx(&bar[1], (uint32_t)(TRON_PVEC * TILE * 16));      // clipped columns are zero-filled and count
            tma_load_2d(&tile.v[0][0], &maps->in, (int)(e0 * 4), 0, &bar[1]);
        } else {
            mbar_expect_tx(&bar[1], (uint32_t)(TRON_PVEC * n * 16));
#pragma unroll
            for (int v = 0; v < TRON_PVEC; v++) bulk_g2s(&tile.v[v][0], st + (long long)v * B + e0, (uint32_t)(n * 16), &bar[1]);
        }
    }
    tron_cta_sync<TILE>();     // barrier initialisation visible to the waiters
#else
    if ((int)threadIdx.x < n) {
        for (int v = 0; v < TRON_PVEC; v++) tile.v[v][threadIdx.x] = st[(long long)v * B + e0 + threadIdx.x];
        tile.hdr()[threadIdx.x] = st[TRON_HVEC * B + e0 + threadIdx.x];
    }
    tron_cta_sync<TILE>();
#endif
}

__device__ __forceinline__ void tron_tile_wait(uint64_t *bar, int which) {
#ifndef CRL_HOSTSIM
    mbar_wait(&bar[which], 0);
#endif
}

// shared -> global: the 9 plane vectors (planes == true) and / or the header vector (the last store of the CTA)
template <int TILE>
__device__ __forceinline__ void tron_tile_store(TronTile<TILE> &tile, const TronMaps *maps, uint4 *__restrict__ st,
                                                long long B, long long e0, int n, bool planes, bool hdr) {
#ifndef CRL_HOSTSIM
    fence_async_smem();        // generic-proxy writes to the tile -> visible to the async proxy
    tron_cta_sync<TILE>();
    if (threadIdx.x == 0) {
        if (planes) {
            if (maps) {
                tma_store_2d(&maps->out, (int)(e0 * 4), 0, &tile.v[0][0]);
            } else {
#pragma unroll
                for (int v = 0; v < TRON_PVEC; v++) bulk_s2g(st + (long long)v * B + e0, &tile.v[v][0], (uint32_t)(n * 16));
            }
        }
        if (hdr) bulk_s2g(st + TRON_HVEC * B + e0, tile.hdr(), (uint32_t)(n * 16));
        bulk_commit();
        if (hdr) bulk_wait_read();       // the tile may be released once the copies have read it
    }
#else
    tron_cta_sync<TILE>();
    if ((int)threadIdx.x < n) {
        if (planes)
            for (int v = 0; v < TRON_PVEC; v++) st[(long long)v * B + e0 + threadIdx.x] = tile.v[v][threadIdx.x];
        if (hdr) st[TRON_HVEC * B + e0 + threadIdx.x] = tile.hdr()[threadIdx.x];
    }
    tron_cta_sync<TILE>();
#endif
}

// ---- one env-step, three phases -------------------------------------------------------------------------------
// CyTronGrid.pyx:15-62 (players strictly in index order against the already-updated board), then
// TronGridEnvironment.py:309-321 and the ranking of :483-508.
//
// The four players live in the four byte lanes of 32-bit words.  Per-player flags are "byte flags" (0x01 in byte p).
// The reference's loop is sequential in the player index, but the only things a later player can observe from an
// earlier one in the same step are (a) the single cell it just claimed, (b) its new head and (c) a head-on kill.
// So all lookups are done against the OLD board (12 independent shared-memory loads) and the sequential part runs on
// registers only.  The <= 4 bit sets are read-modify-writes of the tile, in player order: players 0 and 2 share plane
// c0, players 1 and 2 plane c1, and two movers may claim different cells of the same 32-bit word.
struct TronCtx {
    uint32_t X, Y, Z, W;            // header words (updated in place by the phases)
    uint32_t BX, BY, NX, NY;        // biased head coordinates, old / candidate (one byte per player)
    uint32_t DIR, ND, D4, ALV;      // directions old / candidate, deaths, alive byte flags
    uint32_t pos[4], hpos[4];       // candidate / old head position codes (x | y << 8)
    uint32_t bit[4], same[4];       // bit of the candidate cell inside its word; byte flags of the j < i with the same target
    int off[4];                     // word offset of the candidate cell inside a plane (tile-relative)
    bool inb[4];
    bool reset;
};

struct TronOut {
    uint32_t reward4;               // int8 reward per player
    uint32_t alive, winners, terminal, rank8;
};

// phase 1: needs the header and the actions only.  a4 = the four int8 actions (0 forward, +1 right, -1 left).
template <int TILE>
__device__ __forceinline__ void tron_phase1(TronCtx &c, uint4 h, uint32_t a4, const TronParams &prm, bool auto_reset) {
    const uint32_t N = (uint32_t)prm.N;
    c.reset = auto_reset && ((h.z >> 27) & 1u);
    if (c.reset) h = make_uint4(prm.start_hdr[0], prm.start_hdr[1], prm.start_hdr[2], prm.start_hdr[3]);
    c.X = h.x; c.Y = h.y; c.Z = h.z; c.W = h.w;
    c.D4 = (c.Y >> 5) & 0x07070707u;
    c.DIR = (c.X >> 5) & 0x03030303u;
    c.ND = (c.DIR + (a4 & 0x03030303u)) & 0x03030303u;                   // pyx:31 (-1 == +3 mod 4)
    const uint32_t odd = c.ND & TRON_ONES, hi = (c.ND >> 1) & TRON_ONES;      // 0 N(y-1) 1 E(x+1) 2 S(y+1) 3 W(x-1)
    const uint32_t oh = odd & hi, ev = odd ^ TRON_ONES, eh = ev & hi;
    c.BX = c.X & 0x1F1F1F1Fu; c.BY = c.Y & 0x1F1F1F1Fu;
    c.NX = c.BX + odd - 2u * oh;                                          // pyx:34-41; bytes stay in 0..N+1, no borrows
    c.NY = c.BY + 2u * eh - ev;
    const uint32_t nz = (c.D4 | c.D4 >> 1 | c.D4 >> 2) & TRON_ONES;
    c.ALV = (nz ^ TRON_ONES) & prm.pmask;                                 // pyx:16
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const uint32_t bx = (c.NX >> (8 * i)) & 255u, by = (c.NY >> (8 * i)) & 255u;
        c.inb[i] = (bx - 1u) < N && (by - 1u) < N;                        // pyx:47
        const int cell = c.inb[i] ? (int)(by * N + bx) - (int)(N + 1u) : 0;
        c.off[i] = TronTile<TILE>::woff(cell >> 5);
        c.bit[i] = 1u << (cell & 31);
        c.pos[i] = bx | by << 8;
        c.hpos[i] = ((c.BX >> (8 * i)) & 255u) | ((c.BY >> (8 * i)) & 255u) << 8;
        c.same[i] = 0;
#pragma unroll
        for (int j = 0; j < i; j++) c.same[i] |= (c.pos[j] == c.pos[i]) ? (1u << (8 * j)) : 0u;
    }
}

// new_state (py:228-263) in row t of the tile: empty board, code p + 1 at each spawn
template <int TILE>
__device__ __forceinline__ void tron_tile_reset(TronTile<TILE> &tile, int t, const TronParams &prm) {
    constexpr int PL = TronTile<TILE>::PL;
    uint32_t *words = tile.words(t);
#pragma unroll
    for (int v = 0; v < TRON_PVEC; v++) tile.v[v][t] = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
    for (int p = 0; p < 4; p++)                                           // spawns may share a word: OR by code p + 1
#pragma unroll
        for (int k = 0; k < 3; k++)
            if (((p + 1) >> k) & 1) words[TronTile<TILE>::woff((int)prm.spawn_word[p]) + k * PL] |= prm.spawn_bit[p];
}

// phase 2: lookups, sequential resolve, bit sets, header words X / Y / Z(cells) / W
template <int TILE>
__device__ __forceinline__ void tron_phase2(TronCtx &c, TronTile<TILE> &tile, int t, const TronParams &prm) {
    constexpr int PL = TronTile<TILE>::PL;
    uint32_t *words = tile.words(t);
    if (c.reset) tron_tile_reset(tile, t, prm);
    uint32_t own[4], HK[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const uint32_t *wp = words + c.off[i];
        const uint32_t v0 = wp[0], v1 = wp[PL], v2 = wp[2 * PL];
        const uint32_t code = (v0 & c.bit[i] ? 1u : 0u) | (v1 & c.bit[i] ? 2u : 0u) | (v2 & c.bit[i] ? 4u : 0u);
        own[i] = code ? 1u << (8 * (code - 1u)) : 0u;                     // owner of the cell (code - 1), byte flag
        const uint32_t hs = code == 4u ? c.hpos[3] : code == 3u ? c.hpos[2] : code == 2u ? c.hpos[1] : c.hpos[0];
        HK[i] = (hs == c.pos[i]) ? own[i] : 0u;                           // ... and whether the cell is that owner's (old) head
    }
    uint32_t D4 = c.D4, ALV = c.ALV, MVB = 0u, ACTB = 0u;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const uint32_t me = 1u << (8 * i);
        const bool act = (ALV & me) != 0u;                                // pyx:16 (a head-on kill by j < i counts)
        const uint32_t cl = MVB & c.same[i];                              // the j < i that claimed this very cell in this step
        const uint32_t O = cl ? cl : own[i];                              // pyx:51: owner of the target cell
        const bool coll = act && c.inb[i] && O != 0u;
        const bool mv = act && c.inb[i] && O == 0u;
        const bool oobd = act && !c.inb[i];
        // pyx:56-57: the cell is its owner's CURRENT head (no liveness check: T3).  An owner that moved in this
        // step has its head elsewhere unless it moved INTO this cell (cl).
        const uint32_t Kc = cl ? cl : (HK[i] & ~MVB);
        const uint32_t K = coll ? Kc : 0u;
        const uint32_t owner_id = (O * 0x01020304u) >> 24;                // byte flag q -> q + 1
        const uint32_t dv = oobd ? (uint32_t)(i + 1) : (coll ? owner_id : 0u);   // pyx:47-48, 51-53
        D4 |= dv << (8 * i);
        D4 = (D4 & ~(K * 0xFFu)) | (K * (uint32_t)(i + 1));
        ALV &= ~K;
        MVB |= mv ? me : 0u;                                              // pyx:60-62
        ACTB |= act ? me : 0u;
    }
#pragma unroll
    for (int i = 0; i < 4; i++)                                           // mover i sets its bit in the planes of code i + 1
        if (MVB & (1u << (8 * i)))
#pragma unroll
            for (int k = 0; k < 3; k++)
                if (((i + 1) >> k) & 1) words[c.off[i] + k * PL] |= c.bit[i];
    const uint32_t AM = ACTB * 3u, MM = MVB * 0x1Fu;
    const uint32_t dirn = (c.DIR & ~AM) | (c.ND & AM);                    // pyx:44 (also when i dies)
    c.X = (c.BX & ~MM) | (c.NX & MM) | dirn << 5;
    c.Y = (c.BY & ~MM) | (c.NY & MM) | D4 << 5;
    c.Z += (MVB * 7u) & 0x00040201u;                                      // cells0..2 += moved (byte flags 0,8,16 -> bits 0,9,18)
    c.W += (MVB >> 24) + (1u << 9);                                       // cells3 += moved, episode steps += 1
    c.D4 = D4;
}

// phase 3: rewards / terminal / winners (py:309-321), compute_ranking (py:483-508)
__device__ __forceinline__ void tron_phase3(TronCtx &c, const TronParams &prm, TronOut &o) {
    const uint32_t D4 = c.D4;
    const uint32_t nz = (D4 | D4 >> 1 | D4 >> 2) & TRON_ONES;
    const uint32_t AL = (nz ^ TRON_ONES) & prm.pmask, DEAD = nz & prm.pmask;  // py:310
    o.alive = (AL * 0x01020408u) >> 24;                                   // byte flags -> bit p
    o.terminal = __popc(AL) <= 1;                                         // py:316
    o.winners = o.terminal ? o.alive : 0u;                                // py:319
    o.reward4 = AL * (o.terminal ? 10u : 1u) + DEAD * 0xFFu;              // py:313, 320-321: +1 / -1, sole survivor 10
    // ---- compute_ranking: score = #cells owned, carried in the header
    // tie_locations (py:492): deaths[deaths - 1] == p + 1, where deaths[-1] addresses the LAST player for the alive
    const uint32_t K4 = ((D4 + 0x03030303u) & 0x03030303u) - (nz ^ TRON_ONES) * (uint32_t)(4 - prm.P);
    const uint32_t kk = K4 | K4 >> 4;
    const uint32_t G = __byte_perm(D4, 0u, __byte_perm(kk, 0u, 0x4420));  // byte p = deaths[k_p]
    const uint32_t zt = G ^ 0x04030201u;
    const uint32_t tie = (((zt | zt >> 1 | zt >> 2) & TRON_ONES) ^ TRON_ONES) & prm.pmask;
    // py:493-495 runs ascending and in place, but a tie is either a dead-dead mutual pair (both get the minimum of
    // the two original scores in either order) or an alive player (score := Counter[-1] = 0, and nobody's
    // deaths[] points at an alive player with a tie), so the original scores can be used throughout.
    const uint32_t S01 = (c.Z & 511u) | ((c.Z >> 9) & 511u) << 16, S23 = ((c.Z >> 18) & 511u) | (c.W & 511u) << 16;
    const uint32_t sel = K4 * 0x22u + 0x10101010u;                        // byte p -> the two bytes of score[k_p]
    const uint32_t M01 = __vminu2(S01, __byte_perm(S01, S23, sel)), M23 = __vminu2(S23, __byte_perm(S01, S23, sel >> 16));
    const uint32_t tb = tie * 0xFFu, td = tb & (DEAD * 0xFFu);
    const uint32_t R01 = (S01 & ~__byte_perm(tb, 0u, 0x1100)) | (M01 & __byte_perm(td, 0u, 0x1100));
    const uint32_t R23 = (S23 & ~__byte_perm(tb, 0u, 0x3322)) | (M23 & __byte_perm(td, 0u, 0x3322));
    const int s[4] = {(int)(R01 & 0xFFFFu), (int)(R01 >> 16), (int)(R23 & 0xFFFFu), (int)(R23 >> 16)};
    uint32_t rk = 0;
#pragma unroll
    for (int p = 0; p < 4; p++) {                                         // competition ranking (py:497-506)
        int r = 0;
#pragma unroll
        for (int q = 0; q < 4; q++) r += (q != p && s[q] > s[p]) ? 1 : 0; // absent players hold 0 cells: never greater
        rk |= (uint32_t)r << (2 * p);
    }
    o.rank8 = rk & prm.rkmask;
    c.Z = (c.Z & ~(1u << 27)) | o.terminal << 27;
}

__device__ __forceinline__ uint4 tron_ctx_header(const TronCtx &c) { return make_uint4(c.X, c.Y, c.Z, c.W); }

// result record, 8 bytes per environment: int8 reward[4], u8 terminal, u8 alive mask, u8 winners mask,
// u8 ranking (2 bits per player)
__device__ __forceinline__ uint2 tron_pack_result(const TronOut &o) {
    return make_uint2(o.reward4, o.terminal | o.alive << 8 | o.winners << 16 | o.rank8 << 24);
}

// Episode statistics of one step: 17 counters packed into 6 words so a warp needs 6 redux.sync, not 17; lane l < 17
// then extracts counter l from the (warp-uniform) sums and adds it to `dst` (a shared-memory partial, or the CTA's
// global row when the CTA is one warp) -- ONE atomic instruction per warp.
//   lane constants: word (0..5) | shift << 4 | bits << 10 | slot << 16
#define TRON_SL(word, shift, bits, slot) ((word) | (shift) << 4 | (bits) << 10 | (slot) << 16)
__constant__ uint32_t TRON_STAT_LANE[32] = {
    TRON_SL(0, 0, 8, ST_STEPS), TRON_SL(0, 8, 8, ST_EPISODES), TRON_SL(0, 16, 8, ST_NOWIN), TRON_SL(0, 24, 8, ST_WINS + 0),
    TRON_SL(1, 0, 8, ST_WINS + 1), TRON_SL(1, 8, 8, ST_WINS + 2), TRON_SL(1, 16, 8, ST_WINS + 3),
    TRON_SL(2, 0, 8, ST_RANK + 0), TRON_SL(2, 8, 8, ST_RANK + 1), TRON_SL(2, 16, 8, ST_RANK + 2), TRON_SL(2, 24, 8, ST_RANK + 3),
    TRON_SL(3, 0, 16, ST_EPLEN), TRON_SL(3, 16, 16, ST_REWARD),
    TRON_SL(4, 0, 16, ST_SCORE + 0), TRON_SL(4, 16, 16, ST_SCORE + 1), TRON_SL(5, 0, 16, ST_SCORE + 2), TRON_SL(5, 16, 16, ST_SCORE + 3),
    0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
#define TRON_STAT_LANES 17

template <class T, class V>
__device__ __forceinline__ void tron_stats(T *dst, bool valid, const TronOut &o, uint32_t Z, uint32_t W, uint32_t lane_const) {
    const uint32_t t = (valid && o.terminal) ? 1u : 0u;
    // sum_p (p+1) * reward_p: the rewards are +k (alive) / -1 (dead) per byte
    int rw = 0;
#pragma unroll
    for (int p = 0; p < 4; p++) rw += (p + 1) * (int)(int8_t)(o.reward4 >> (8 * p));
    const uint32_t w0 = t ? o.winners : 0u;
    // every field is a sum of <= 32 lane values and stays inside its bit range
    uint32_t A = (valid ? 1u : 0u) | t << 8 | (uint32_t)(t && o.winners == 0u) << 16 | (w0 & 1u) << 24;
    uint32_t Bw = (w0 >> 1 & 1u) | (w0 >> 2 & 1u) << 8 | (w0 >> 3 & 1u) << 16;
    uint32_t C = t ? ((o.rank8 & 3u) | (o.rank8 >> 2 & 3u) << 8 | (o.rank8 >> 4 & 3u) << 16 | (o.rank8 >> 6 & 3u) << 24) : 0u;
    uint32_t D = (t ? (W >> 9) : 0u) | (uint32_t)((valid ? rw : 0) + 16) << 16;          // reward sum biased by +16 per lane
    uint32_t E = t ? ((Z & 511u) | (Z >> 9 & 511u) << 16) : 0u;
    uint32_t F = t ? ((Z >> 18 & 511u) | (W & 511u) << 16) : 0u;
    A = __reduce_add_sync(0xffffffffu, A); Bw = __reduce_add_sync(0xffffffffu, Bw);
    C = __reduce_add_sync(0xffffffffu, C); D = __reduce_add_sync(0xffffffffu, D);
    E = __reduce_add_sync(0xffffffffu, E); F = __reduce_add_sync(0xffffffffu, F);
    // the six sums are warp-uniform; lane l picks its word with masks (no branches), then its field
    const uint32_t word = lane_const & 15u;
    const uint32_t w = (A & -(uint32_t)(word == 0u)) | (Bw & -(uint32_t)(word == 1u)) | (C & -(uint32_t)(word == 2u)) |
                       (D & -(uint32_t)(word == 3u)) | (E & -(uint32_t)(word == 4u)) | (F & -(uint32_t)(word == 5u));
    int val = (int)((w >> ((lane_const >> 4) & 31u)) & ((1u << ((lane_const >> 10) & 31u)) - 1u));
    const int slot = (int)(lane_const >> 16);
    if (slot == ST_REWARD) val -= 16 * 32;
    if ((int)(threadIdx.x & 31) < TRON_STAT_LANES && val != 0) atomicAdd(&dst[slot], (V)(long long)val);
}

__device__ __forceinline__ void tron_zero_out(TronOut &o) { o.reward4 = o.alive = o.winners = o.terminal = o.rank8 = 0u; }

// actions: int8[B][4] (0 forward, +1 right, -1 left  == STRING_TO_ACTION, TronGridEnvironment.py:62-67), one
// coalesced 32-bit load per environment.
template <int TILE>
__global__ void __launch_bounds__(TILE)
tron_step_kernel(const __grid_constant__ TronMaps maps, const uint4 *__restrict__ in, uint4 *__restrict__ out,
                 const uint32_t *__restrict__ actions, uint2 *__restrict__ result, crl_u64 *stats, long long B,
                 TronParams prm, int flags) {
    __shared__ __align__(128) TronTile<TILE> tile;
    __shared__ __align__(8) uint64_t bar[2];
    const int t = threadIdx.x;
    const long long e0 = (long long)blockIdx.x * TILE;
    const int n = (int)min((long long)TILE, B - e0);
    const bool valid = t < n;
    const uint32_t lane_const = TRON_STAT_LANE[t & 31];
    // PDL prologue: this runs while the predecessor in the stream is still executing.  Nothing may be READ yet, but the
    // tile, its header and its actions can be pulled from HBM into L2 (prefetches are hints: if the predecessor is
    // still writing these very lines, L2 already holds / will hold the coherent copy), so that the loads issued after
    // griddepcontrol.wait are L2 hits and HBM keeps streaming across the launch boundary.
    if (flags & 0x4000) pdl_launch_dependents();             // (diagnostic: trigger before the prefetch / wait)
#ifndef CRL_HOSTSIM
    if (t == 0 && !(flags & 0x2000)) {
        l2_prefetch_tensor_2d(&maps.in, (int)(e0 * 4), 0);
        l2_prefetch_bulk(in + TRON_HVEC * B + e0, (uint32_t)(n * 16));
        const uint32_t abytes = (uint32_t)((flags & CRL_FLAG_PACKED_ACTIONS) ? n : 4 * n);
        const char *ap = (const char *)actions + ((flags & CRL_FLAG_PACKED_ACTIONS) ? e0 : 4 * e0);
        if (!(abytes & 15u) && !((uintptr_t)ap & 15)) l2_prefetch_bulk(ap, abytes);
    }
#endif
    pdl_wait();                  // (programmatic dependent launch only) everything above overlapped the previous kernel's tail
    // let the successor's CTAs become resident NOW: its prologue prefetch then overlaps this launch's own traffic.  The
    // successor still blocks at its griddepcontrol.wait until this grid has completed, and ITS successor cannot start
    // before it has passed that wait -- at most two launches are ever co-resident.
    if (!(flags & 0x5000)) pdl_launch_dependents();
    uint32_t a = 0u;                                         // in flight together with the tile
    if (valid) {
        if (flags & CRL_FLAG_PACKED_ACTIONS) {               // one byte per environment, 2 bits per player
            const uint32_t b = ((const uint8_t *)actions)[e0 + t];
            a = (b & 3u) | (b & 0xcu) << 6 | (b & 0x30u) << 12 | (b & 0xc0u) << 18;
        } else {
            a = actions[e0 + t];
        }
    }
#ifndef CRL_HOSTSIM
    // (diagnostic 0x8000 / 0x10000: stagger the tile loads of the CTAs that share an SM by 100 / 200 ns per rank, to see
    // whether a launch's load and store phases can be made to overlap)
    if ((flags & 0x18000) && t == 0) __nanosleep((blockIdx.x / 148u) * ((flags & 0x8000) ? 100u : 0u) + (blockIdx.x / 148u) * ((flags & 0x10000) ? 200u : 0u));
#endif
    tron_tile_load_issue(tile, bar, &maps, in, B, e0, n);
    TronOut o;
    tron_zero_out(o);
    TronCtx c;
    c.Z = c.W = 0u;
    tron_tile_wait(bar, 0);
    // flags >= 0x100 are diagnostics (tools/tron_probe.py): 0x100 data movement only, 0x200 no phase 2, 0x400 no
    // phase 3, 0x800 no statistics -- results are meaningless with any of them; 0x1000 late PDL trigger, 0x2000 no
    // prologue prefetch (results unaffected)
    const bool work = valid && !(flags & 0x100);
    if (work) tron_phase1<TILE>(c, tile.hdr()[t], a, prm, (flags & CRL_FLAG_AUTO_RESET) != 0);
    tron_tile_wait(bar, 1);
    if (work && !(flags & 0x200)) tron_phase2(c, tile, t, prm);
    tron_tile_store(tile, &maps, out, B, e0, n, true, false);
    if (flags & 0x1000) pdl_launch_dependents();     // (diagnostic: the round-1 trigger position)
    if (work) {
        if (!(flags & 0x400)) tron_phase3(c, prm, o);
        tile.hdr()[t] = tron_ctx_header(c);
        const uint2 rec = tron_pack_result(o);
        if (flags & CRL_FLAG_COMPACT2_RESULT)                                        // 2-byte record (see the header)
            ((uint16_t *)result)[e0 + t] = (uint16_t)(((rec.y >> 8) & 0xfu) | (rec.y & 1u) << 4 | (rec.y >> 24) << 8);
        else if (flags & CRL_FLAG_COMPACT_RESULT) ((uint32_t *)result)[e0 + t] = rec.y;   // 4-byte record
        else result[e0 + t] = rec;
    }
    tron_tile_store(tile, &maps, out, B, e0, n, false, true);
    if (out != in && valid)                                  // an out-of-place step writes a whole state: reserved = 0
#pragma unroll
        for (int v = TRON_PVEC; v < TRON_HVEC; v++) out[(long long)v * B + e0 + t] = make_uint4(0u, 0u, 0u, 0u);
    // statistics: every warp adds its 17 sums straight to the CTA's row of the global buffer (fire-and-forget RED);
    // after the last store, so that the header is already draining (measured 0.1 us / step cheaper than before it)
    if (stats && !(flags & 0x800))
        tron_stats<crl_u64, crl_u64>(stats + (blockIdx.x & (CRL_STAT_ROWS - 1)) * CRL_NSTAT, valid, o, c.Z, c.W, lane_const);
}

// ---- the avoid policy --------------------------------------------------------------------------------------------
// A heuristic opponent in the shape of the reference's SimpleAvoidAgent (envs/tron/rllib.py:69-96, which asks
// env.next_cell at :85 and :91): go forward if that cell is free, else try one side, else take the other.  The
// reference's source is not part of this repository, so the exact rule below -- the coin, the noise, the order -- is
// THIS ENGINE'S DEFINITION, pinned by the C oracle (tests/oracle_tron_avoid.c) the way the random policy is.  For
// seat p of environment env at step t, on the state BEFORE the step:
//   w = philox(seed, env, t, CRL_TAG_TRON_AVOID + (p >> 2))[p & 3]
//   (w >> 16) < noise_q16 (0..65536)  ->  {0, +1, -1}[(w & 0xFFFF) % 3]
//   else forward if its cell is free (on the board and owner code 0; heads are owned cells),
//   else side s = (w & 1) ? +1 (right) : -1 (left) if its cell is free, else -s.
// `occupied(cell)` is the layout's board lookup, (hx, hy) the head, dir its direction (0 N, 1 E, 2 S, 3 W).
template <class Occupied>
__device__ __forceinline__ int tron_avoid_decide(int hx, int hy, int dir, int N, uint32_t w, uint32_t noise_q16,
                                                 const Occupied &occupied) {
    if ((w >> 16) < noise_q16) {
        const uint32_t m = (w & 0xFFFFu) % 3u;
        return m == 2u ? -1 : (int)m;
    }
    auto is_free = [&](int a) {                                           // pyx:31-41: turn, then one cell ahead
        const int d = (dir + a) & 3;
        const int x = hx + (d == 1) - (d == 3), y = hy + (d == 2) - (d == 0);
        return x >= 0 && x < N && y >= 0 && y < N && !occupied(y * N + x);
    };
    if (is_free(0)) return 0;
    const int side = (w & 1u) ? 1 : -1;
    return is_free(side) ? side : -side;
}

// The avoid actions of the seats in `mask` written into the action word `a` (byte p = seat p; the other bytes are
// kept), decided on tile row t with header h (both already reset if the game restarts in this step).  Dead seats get 0.
// Per live seat: the three code planes of <= 3 cells, i.e. up to 9 shared-memory lookups.
template <int TILE>
__device__ __forceinline__ uint32_t tron_avoid_word(TronTile<TILE> &tile, int t, uint4 h, uint32_t a, const TronParams &prm,
                                                    uint32_t mask, uint32_t noise_q16, crl_u64 seed, crl_u64 env,
                                                    uint32_t step) {
    constexpr int PL = TronTile<TILE>::PL;
    const uint32_t *words = tile.words(t);
    auto occupied = [&](int cell) {
        const int o = TronTile<TILE>::woff(cell >> 5);
        return (((words[o] | words[o + PL] | words[o + 2 * PL]) >> (cell & 31)) & 1u) != 0u;
    };
    const uint4 r = env_words(seed, env, step, CRL_TAG_TRON_AVOID);
    const uint32_t rr[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int p = 0; p < 4; p++) {
        if (!((mask >> p) & 1u)) continue;
        const uint32_t bx = (h.x >> (8 * p)) & 255u, by = (h.y >> (8 * p)) & 255u;
        const int act = (by >> 5) ? 0 : tron_avoid_decide((int)(bx & 31u) - 1, (int)(by & 31u) - 1, (int)(bx >> 5) & 3,
                                                          prm.N, rr[p], noise_q16, occupied);
        a = (a & ~(0xFFu << (8 * p))) | ((uint32_t)act & 0xFFu) << (8 * p);
    }
    return a;
}

// crl_tron_policy_avoid: one thread per environment, actions int8[B][4] read-modify-written as one 32-bit word.  The
// tile's 9 plane rows are loaded whole (bulk copies, 144 coalesced bytes per environment) rather than only the words
// the lookups touch: those are up to 36 scattered 4-byte reads per environment, each costing a whole 32-byte sector,
// and the whole rows in shared memory let the lookups be plain indexed loads.
template <int TILE>
__global__ void __launch_bounds__(TILE)
tron_policy_avoid_kernel(const uint4 *__restrict__ st, uint32_t *__restrict__ actions, long long B, TronParams prm,
                         uint32_t mask, uint32_t noise_q16, crl_u64 seed, crl_u64 first_env, uint32_t step, int flags) {
    __shared__ __align__(128) TronTile<TILE> tile;
    __shared__ __align__(8) uint64_t bar[2];
    const int t = threadIdx.x;
    const long long e0 = (long long)blockIdx.x * TILE;
    const int n = (int)min((long long)TILE, B - e0);
    tron_tile_load_issue(tile, bar, (const TronMaps *)nullptr, st, B, e0, n);
    const uint32_t a = t < n ? actions[e0 + t] : 0u;                      // in flight together with the tile
    tron_tile_wait(bar, 0);
    tron_tile_wait(bar, 1);
    if (t >= n) return;
    uint4 h = tile.hdr()[t];
    if ((flags & CRL_FLAG_AUTO_RESET) && ((h.z >> 27) & 1u)) {           // decide on the game the step will restart
        tron_tile_reset(tile, t, prm);
        h = make_uint4(prm.start_hdr[0], prm.start_hdr[1], prm.start_hdr[2], prm.start_hdr[3]);
    }
    actions[e0 + t] = tron_avoid_word(tile, t, h, a, prm, mask, noise_q16, seed, first_env + (crl_u64)(e0 + t), step);
}

// K fused steps with the in-kernel Philox random policy (action of player p = {0,+1,-1}[r_p % 3]); the tile
// stays in shared memory between steps.  Benchmark / self-play helper; semantics identical to K tron_step calls
// with CRL_FLAG_AUTO_RESET.
// AVOID: the seats of avoid_mask play the avoid policy instead (= K x policy_random -> policy_avoid(avoid_mask,
// CRL_FLAG_AUTO_RESET) -> step(CRL_FLAG_AUTO_RESET)).  The policy reads the board the step will move on, so a finished
// game is restarted here, before the policy, and phase 1 / 2 are told not to restart it again.
template <int TILE, bool AVOID = false>
__global__ void __launch_bounds__(TILE)
tron_rollout_kernel(uint4 *__restrict__ state, uint2 *__restrict__ result, crl_u64 *stats, long long B,
                    TronParams prm, crl_u64 seed, crl_u64 first_env, uint32_t step0, int K, uint32_t avoid_mask,
                    uint32_t noise_q16) {
    __shared__ __align__(128) TronTile<TILE> tile;
    __shared__ __align__(8) uint64_t bar[2];
    __shared__ int sm_stat[CRL_NSTAT];
    const int t = threadIdx.x;
    const long long e0 = (long long)blockIdx.x * TILE;
    const int n = (int)min((long long)TILE, B - e0);
    const bool valid = t < n;
    if (stats && t < CRL_NSTAT) sm_stat[t] = 0;
    const uint32_t lane_const = TRON_STAT_LANE[t & 31];
    tron_tile_load_issue(tile, bar, (const TronMaps *)nullptr, state, B, e0, n);
    tron_tile_wait(bar, 0);
    tron_tile_wait(bar, 1);
    TronOut o;
    tron_zero_out(o);
    TronCtx c;
    c.Z = c.W = 0u;
    uint4 h = valid ? tile.hdr()[t] : make_uint4(0u, 0u, 0u, 0u);
    for (int k = 0; k < K; k++) {
        if (valid) {
            uint4 r = env_words(seed, first_env + (crl_u64)(e0 + t), step0 + (uint32_t)k, CRL_TAG_TRON);
            const uint32_t rr[4] = {r.x, r.y, r.z, r.w};
            uint32_t a = 0;
#pragma unroll
            for (int p = 0; p < 4; p++) { const uint32_t m = rr[p] % 3u; a |= ((m == 2u) ? 0xffu : m) << (8 * p); }
            if constexpr (AVOID) {
                if ((h.z >> 27) & 1u) {
                    tron_tile_reset(tile, t, prm);
                    h = make_uint4(prm.start_hdr[0], prm.start_hdr[1], prm.start_hdr[2], prm.start_hdr[3]);
                }
                a = tron_avoid_word(tile, t, h, a, prm, avoid_mask, noise_q16, seed, first_env + (crl_u64)(e0 + t),
                                    step0 + (uint32_t)k);
            }
            tron_phase1<TILE>(c, h, a, prm, !AVOID);
            tron_phase2(c, tile, t, prm);
            tron_phase3(c, prm, o);
            h = tron_ctx_header(c);
        }
        if (stats) tron_stats<int, int>(sm_stat, valid, o, c.Z, c.W, lane_const);
    }
    if (valid) {
        tile.hdr()[t] = h;
        if (result) result[e0 + t] = tron_pack_result(o);
    }
    tron_tile_store(tile, (const TronMaps *)nullptr, state, B, e0, n, true, true);
    if (stats) {
        tron_cta_sync<TILE>();
        stats_flush_row(sm_stat, stats);
    }
}

__global__ void tron_policy_random_kernel(uint32_t *__restrict__ actions, long long B, crl_u64 seed,
                                          crl_u64 first_env, uint32_t step) {
    long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= B) return;
    uint4 r = env_words(seed, first_env + (crl_u64)e, step, CRL_TAG_TRON);
    uint32_t rr[4] = {r.x, r.y, r.z, r.w}, a = 0;
#pragma unroll
    for (int p = 0; p < 4; p++) { uint32_t m = rr[p] % 3u; a |= ((m == 2) ? 0xffu : m) << (8 * p); }
    actions[e] = a;
}

// new_state for all / masked environments: one thread per (vector, environment), fully coalesced stores
__global__ void tron_reset_kernel(uint4 *__restrict__ state, const uint8_t *__restrict__ mask, long long B, TronParams prm) {
    long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= B * TRON_VEC) return;
    const int v = (int)(idx / B);
    const long long e = idx - (long long)v * B;
    if (mask && !mask[e]) return;
    uint4 val = v == TRON_HVEC ? make_uint4(prm.start_hdr[0], prm.start_hdr[1], prm.start_hdr[2], prm.start_hdr[3])
                               : make_uint4(0u, 0u, 0u, 0u);        // (reserved vectors 9..11: zero)
    if (v < TRON_PVEC) {                                             // words 4j .. 4j+3 of plane k: the spawn bits of codes with bit k
        const uint32_t k = (uint32_t)v / 3u, j = (uint32_t)v - 3u * k;
#pragma unroll
        for (int p = 0; p < 4; p++) {
            const uint32_t w = prm.spawn_word[p], b = (((p + 1) >> k) & 1) ? prm.spawn_bit[p] : 0u;   // spawns may share a word
            val.x |= w == 4u * j ? b : 0u; val.y |= w == 4u * j + 1u ? b : 0u;
            val.z |= w == 4u * j + 2u ? b : 0u; val.w |= w == 4u * j + 3u ? b : 0u;
        }
    }
    state[idx] = val;
}

// state_to_observation (TronGridEnvironment.py:385-405).  A CTA handles a tile of 16 environments: 10 bulk copies
// bring their packed state into shared memory, its 4 warps unpack 4 environments each into a shared-memory image of
// the dense output, and ONE bulk copy writes the tile's boards (16 * nview * N*N contiguous bytes, always 16-byte
// aligned and a multiple of 16 bytes) back to HBM.
// Unpacking is byte-SWAR: lane l owns cells 128 k + 4 l .. + 3 (k = 0..2): the 4 bits of every code plane are spread
// to 4 bytes with one multiply + mask, which gives the owner code of each cell, and one PRMT through a per-viewer
// table relabels it -- the relabelling of CyTronGrid.pyx:65-71 costs nothing.
//   player >= 0 : that player's view (board relabelled, vectors rolled py:392)
//   player == -1: absolute view (plain unpack: board values p+1)
//   player == -3: ALL P views at once (CRL_PLAYER_ALL, nview = P)
// board int8[B][nview][N][N]; heads (y*N + x like the reference) / dirs / deaths int32[B][nview][P]; terminal u8[B].
#define TRON_OBS_TILE 16
#define TRON_OBS_MAXBYTES (TRON_OBS_TILE * 4 * 384)

// board value LUT of one view (owner 0 empty / q + 1 -> value) as the two source words of a PRMT
__device__ __forceinline__ void tron_view_lut(int viewer, int P, uint32_t &lo, uint32_t &hi) {
    uint32_t id[4];
#pragma unroll
    for (int q = 0; q < 4; q++) {
        int x = q + 1;                                       // absolute: board value = player + 1
        if (viewer >= 0) { x = q - viewer; x += x < 0 ? P : 0; x += 1; }
        id[q] = (uint32_t)(q < P ? x : 0);
    }
    lo = id[0] << 8 | id[1] << 16 | id[2] << 24;
    hi = id[3];
}

__device__ __forceinline__ void tron_obs_store4(uint8_t *o, uint32_t v, int c0, int NN, bool guard) {
    if (!guard) {
        o[0] = (uint8_t)v; o[1] = (uint8_t)(v >> 8); o[2] = (uint8_t)(v >> 16); o[3] = (uint8_t)(v >> 24);
    } else {
#pragma unroll
        for (int j = 0; j < 4; j++)
            if (c0 + j < NN) o[j] = (uint8_t)(v >> (8 * j));
    }
}

template <bool ALL>
__global__ void __launch_bounds__(128)
tron_observe_kernel(const uint4 *__restrict__ st, long long B, TronParams prm, int player,
                    int8_t *__restrict__ board, int32_t *__restrict__ heads, int32_t *__restrict__ dirs,
                    int32_t *__restrict__ deaths, uint8_t *__restrict__ terminal) {
    __shared__ __align__(128) TronTile<TRON_OBS_TILE> tile;
    CRL_DYN_SMEM(img, TRON_OBS_MAXBYTES);                 // TRON_OBS_TILE * nview * N*N bytes (rounded up to 16)
    __shared__ __align__(8) uint64_t bar[2];
    constexpr int PL = TronTile<TRON_OBS_TILE>::PL;
    const int N = prm.N, P = prm.P, NN = N * N;
    const long long e0 = (long long)blockIdx.x * TRON_OBS_TILE;
    const int n = (int)min((long long)TRON_OBS_TILE, B - e0);
#ifndef CRL_HOSTSIM
    if (threadIdx.x == 0) {
        mbar_init(&bar[0], 1);
        mbar_expect_tx(&bar[0], (uint32_t)((TRON_PVEC + 1) * n * 16));
        const uint4 *src = st + e0;
        uint4 *dst = &tile.v[0][0];
#pragma unroll 1
        for (int v = 0; v < TRON_PVEC; v++, src += B, dst += TRON_OBS_TILE) bulk_g2s(dst, src, (uint32_t)(n * 16), &bar[0]);
        bulk_g2s(tile.hdr(), st + TRON_HVEC * B + e0, (uint32_t)(n * 16), &bar[0]);
    }
    __syncthreads();
    mbar_wait(&bar[0], 0);
#else
    if ((int)threadIdx.x < n) {
        for (int v = 0; v < TRON_PVEC; v++) tile.v[v][threadIdx.x] = st[(long long)v * B + e0 + threadIdx.x];
        tile.hdr()[threadIdx.x] = st[TRON_HVEC * B + e0 + threadIdx.x];
    }
    __syncthreads();
#endif
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nview = ALL ? P : 1, chunks = (NN + 127) >> 7;
    uint32_t lut_lo[4], lut_hi[4];
#pragma unroll
    for (int pv = 0; pv < 4; pv++) tron_view_lut(ALL ? pv : player, P, lut_lo[pv], lut_hi[pv]);
    // lane l owns cells 128 k + 4 l .. + 3: word 4 k + (l >> 3) of every plane, bits (4 l & 31) .. + 3
    const int sh = (4 * lane) & 31, wl = lane >> 3;
    for (int t = warp; t < n; t += 4) {
        const uint32_t *wp = tile.words(t) + wl;
        uint8_t *out = img + t * nview * NN + 4 * lane;
        for (int k = 0; k < chunks; k++, wp += TRON_OBS_TILE * 4, out += 128) {
            // owner code (0 empty, q + 1) of the lane's 4 cells, one byte each, from the three stored code bit-planes
            const uint32_t v0 = (wp[0] >> sh) & 15u, v1 = (wp[PL] >> sh) & 15u, v2 = (wp[2 * PL] >> sh) & 15u;
            const uint32_t ow = ((v0 * 0x00204081u) & TRON_ONES) + 2u * ((v1 * 0x00204081u) & TRON_ONES) +
                                4u * ((v2 * 0x00204081u) & TRON_ONES);
            const uint32_t sel = __byte_perm(ow | ow >> 4, 0u, 0x4420);      // the 4 owners as PRMT selector nibbles
            const int c0 = 128 * k + 4 * lane;
            const bool guard = k == chunks - 1;
            if (ALL) {
#pragma unroll
                for (int pv = 0; pv < 4; pv++)
                    if (pv < P) tron_obs_store4(out + pv * NN, __byte_perm(lut_lo[pv], lut_hi[pv], sel), c0, NN, guard);
            } else {
                tron_obs_store4(out, __byte_perm(lut_lo[0], lut_hi[0], sel), c0, NN, guard);
            }
        }
    }
    // per-player vectors, rolled by the viewer (py:392-396): ONE pass over the tile -- thread i owns entry i of the
    // tile's [env][view][player] block, which is contiguous in the three output arrays (coalesced 4-byte stores).  (Done
    // per environment by the lanes of its warp, as at first, this part was 93 of the kernel's 264 warp instructions per
    // environment: integer divisions and 64-bit index arithmetic for 4..16 useful lanes.)
    {
        const int per_env = nview * P, entries = n * per_env;
        for (int i = threadIdx.x; i < entries; i += blockDim.x) {
            const int t = i / per_env, r = i - t * per_env;
            const int pv = ALL ? r / P : max(player, 0), c = ALL ? r - pv * P : r;
            int src = c + ((!ALL && player == -1) ? 0 : pv);
            src -= src >= P ? P : 0;
            const uint4 h = tile.hdr()[t];
            const uint32_t bx = (h.x >> (8 * src)) & 255u, by = (h.y >> (8 * src)) & 255u;
            const long long o = e0 * per_env + i;
            if (heads) heads[o] = ((int)(by & 31u) - 1) * N + (int)(bx & 31u) - 1;
            if (dirs) dirs[o] = (int)(bx >> 5) & 3;
            if (deaths) deaths[o] = (int)(by >> 5);
        }
        if (terminal && (int)threadIdx.x < n) terminal[e0 + threadIdx.x] = (uint8_t)((tile.hdr()[threadIdx.x].z >> 27) & 1u);
    }
    // the tile's boards: one bulk copy when the segment is 16-byte aligned and sized, a cooperative byte copy otherwise
    const int nbytes = n * nview * NN;
    int8_t *dst = board + e0 * nview * NN;
#ifndef CRL_HOSTSIM
    if ((nbytes & 15) == 0 && (((uintptr_t)dst) & 15) == 0) {
        fence_async_smem();
        __syncthreads();
        if (threadIdx.x == 0) {
            bulk_s2g(dst, img, (uint32_t)nbytes);
            bulk_commit();
            bulk_wait_read();
        }
        return;
    }
#endif
    __syncthreads();
    for (int i = threadIdx.x; i < nbytes; i += blockDim.x) dst[i] = (int8_t)img[i];
}

// compute_ranking (TronGridEnvironment.py:483-508) of an arbitrary state, without stepping it: ranking byte per
// environment (2 bits per player), same code path as the ranking fused into the step
__global__ void tron_ranking_kernel(const uint4 *__restrict__ st, long long B, TronParams prm, uint8_t *__restrict__ ranking) {
    long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= B) return;
    const uint4 h = st[TRON_HVEC * B + e];
    TronCtx c;
    c.X = h.x; c.Y = h.y; c.Z = h.z; c.W = h.w;
    c.D4 = (h.y >> 5) & 0x07070707u;
    TronOut o;
    tron_phase3(c, prm, o);
    ranking[e] = (uint8_t)o.rank8;
}

// import a reference-layout state (board int8[B][N][N], heads (y*N+x) / directions / deaths int32[B][P]);
// one thread per environment (import path, not performance critical)
__global__ void tron_pack_kernel(uint4 *__restrict__ st, long long B, TronParams prm,
                                 const int8_t *__restrict__ board, const int32_t *__restrict__ heads,
                                 const int32_t *__restrict__ dirs, const int32_t *__restrict__ deaths) {
    const int N = prm.N, P = prm.P, NN = N * N;
    long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= B) return;
    uint64_t pl[3][TRON_WORDS];                             // the three owner-code bit-planes
    TronHdr s;
#pragma unroll
    for (int k = 0; k < 3; k++)
#pragma unroll
        for (int w = 0; w < TRON_WORDS; w++) pl[k][w] = 0;
#pragma unroll
    for (int p = 0; p < 4; p++) s.hx[p] = s.hy[p] = s.dir[p] = s.death[p] = s.cells[p] = 0;
    for (int c = 0; c < NN; c++) {
        const int v = board[e * NN + c];
        const int code = (v >= 1 && v <= 4) ? v : 0;         // owner code: player v - 1
#pragma unroll
        for (int p = 0; p < 4; p++) s.cells[p] += (code == p + 1);
#pragma unroll
        for (int k = 0; k < 3; k++)
#pragma unroll
            for (int w = 0; w < TRON_WORDS; w++)
                pl[k][w] |= (((code >> k) & 1) && w == (c >> 6)) ? (1ull << (c & 63)) : 0ull;
    }
    int alive = 0;
#pragma unroll
    for (int p = 0; p < 4; p++) {
        if (p < P) {
            int h = heads[e * P + p];
            s.hx[p] = h % N; s.hy[p] = h / N;
            s.dir[p] = dirs[e * P + p] & 3;
            s.death[p] = deaths[e * P + p] & 7;
            alive += s.death[p] == 0;
        }
    }
    s.terminal = alive <= 1;
    s.ep_len = 0;
#pragma unroll
    for (int k = 0; k < 3; k++)
#pragma unroll
        for (int j = 0; j < 3; j++) {
            uint64_t a = pl[k][2 * j], b = pl[k][2 * j + 1];
            st[(long long)(3 * k + j) * B + e] = make_uint4((uint32_t)a, (uint32_t)(a >> 32), (uint32_t)b, (uint32_t)(b >> 32));
        }
#pragma unroll
    for (int v = TRON_PVEC; v < TRON_HVEC; v++) st[(long long)v * B + e] = make_uint4(0u, 0u, 0u, 0u);   // reserved
    st[(long long)TRON_HVEC * B + e] = tron_hdr_encode(s);
}
