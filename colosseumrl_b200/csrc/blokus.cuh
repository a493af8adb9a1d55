// Blokus 4-player 20x20: legal-move generation and move application on row bitboards (sm_100a).
//
// Replaces (reference file:line):
//   Board.get_all_valid_moves        envs/blokus/board.py:170-193  (anchors :114-154, orientation/shift loop :156-168)
//   check_shifted & friends          envs/blokus/computation.py:145-180, 184-246, 53-142   (numba)
//   BlokusEnvironment.valid_actions  envs/blokus/BlokusEnvironment.py:453-500 (canonical order of the flattened dict)
//   BlokusEnvironment.next_state     :357-451  (Board.update_board board.py:87-98, AI.update_player ai.py:44-54,
//                                    the terminal test `not any(p.check_moves(board, round_count))` :424 which runs on
//                                    the OLD board / OLD round with the NEW inventories, winners/reward :425-440)
//   new_state :248-289, state_to_observation :721-768
//
// HBM layout: 352 bytes per game, AoS (a warp owns a game): 22 x uint4 = 88 words
//   w[20*c + y]  row y of colour c's plane, bit x set iff colour c occupies (x, y)           (c = 0..3, 80 words)
//   w[80 + c]    inventory of player c, bit p set iff piece p (PIECE_TYPES order) is still held
//   w[84]        scores, one byte per player        w[85] round | mover << 8 | terminal << 16
//   w[86]        steps taken in this episode
//   w[87]        bit q: player q is known to have no legal move any more (a cache, 0 = unknown).  Once a player
//                who is not the mover has no move in a round >= 1 he never has one again: his cells and pieces do not
//                change while he cannot move and the empty cells only shrink, so the anchor set and every FIT board can
//                only lose bits.  (Not in round 0, where the anchor is the corner; not for the mover, whose terminal test
//                runs on the board BEFORE his own move, BlokusEnvironment.py:424.)  The step kernel sets the bit instead
//                of repeating the full negative test every step, the legal kernel answers "no moves" from it.
// Lanes 0..21 of the warp move the game with one 128-bit access each (352 contiguous bytes).
//
// Legality in bitboard form (SURVEY.md Appendix A-B2): with
//   A   = empty & ~N4(own)                                   "allowed" cells (computation.py:122-142, 89-119)
//   ANC = {corner}            if round == 0 (board.py:177-179)
//         A & D4(own)         otherwise      (board.py:114-154)
//   FIT_s[q] = AND_i A[q + cell_i(s)]                       shape s fits with its bounding-box corner at q
// action (piece, anchor a, orientation o, shift k) is legal  <=>  a in ANC  and  FIT_s[a - cell_k(s)],
// s = shape(piece, o).  The list is emitted in the reference's order piece -> anchor (row-major) -> o -> k, with
// lanes = (anchor of a group of four, orientation), a SWAR popcount + one shuffle scan per 16 anchors (blk_emit_piece).
//
// FIT boards, LANES = SHAPES: the 91 oriented shapes are exactly the fixed polyominoes of 1..5 cells.  The 27 shapes
// of 2..4 cells are built in ONE pass straight from A (blk_tree_pass_le4: lane l owns shape 1 + l and ANDs the <= 4
// shifted A rows of its cells over the 20 rows: 4 LDS, 4 shifts, 2 LOP3, 1 STS per row); a pentomino is a tetromino
// plus a cell, FIT_s[q] = FIT_parent[q + off] & A[q + c] (blk_tree_pass: 2 LDS, 2 shifts, 1 AND, 1 STS per row,
// parameters from a per-shape table), one pass per group of pentomino pieces (the groups share the same slots; a
// group is built, its pieces are emitted, the next group overwrites it).  One ballot per pass yields the non-empty
// flags of up to 32 shapes.  Shapes whose pieces are not held or whose parent fits nowhere are idle lanes; a pass
// without work is skipped.  Everything is a compact loop: the first version was 86 KB of straight-line SASS and
// spent 70 % of its cycles waiting for the instruction cache.
// The any-move test of the terminal check needs no anchor loop at all:
// piece p has a move  <=>  OR_s OR_k (ANC & shift(FIT_s, cell_k)) != 0, again with lanes = shapes, level by level
// with an early exit.
#pragma once
#include "crl_common.cuh"
#include "philox.cuh"
#include "blokus_tables.h"

#define BLK_WORDS 88
#define BLK_VEC 22
#define BLK_WARPS 1            // legal / step: ONE warp (= game) per CTA, so the game index is blockIdx.x and every
                               // vote / shuffle sits in provably uniform control flow (no BRA.DIV slow paths)
#define BLK_OBS_WARPS 4        // observation kernel: games per CTA
#define BLK_ROWMASK 0xFFFFFu
#define BLK_MAX_ANCHORS 400

#define BLK_FSLOTS (BLK_NSHAPE_LE4 + BLK_GROUP_MAX)
#define BLK_OFF_LE4 8           // bit offset of column 0 in the FIT boards of shapes of <= 4 cells
#define BLK_OFF_PENT 12         // ... and of the pentomino shapes

// per-warp shared scratch
struct BlkSmem {
    uint32_t st[BLK_WORDS];          // the game state (old board during a step)
    uint32_t A[24];                  // allowed rows << 4 (bit x + 4); rows 20..23 are zero (shapes are at most 5 rows tall)
    uint32_t anc[20];                // anchor rows (bit x)
    alignas(16) uint32_t F[BLK_FSLOTS * BLK_FROWS + 4];   // FIT boards: bit (x + BLK_OFF(n)) of word [slot * BLK_FROWS + y + 4]
                                     // with BLK_OFF = 8 for shapes of <= 4 cells and 12 for pentominoes: a board is built
                                     // with LEFT shifts only (IMADs on the FMA pipe -- the ALU pipe is this kernel's busy
                                     // one), each level landing 4 bits above its inputs.  The zero padding (rows -4..-1,
                                     // 20..24, the bits below the offset) makes FIT_s[a - cell] a plain load + shift for
                                     // every anchor a and shape cell, and a tree step branch-free
    // anchors, row-major, 16 bits each: (4 * y) << 9 | x, then >= 4 padding entries (column 24: outside every FIT
    // board).  One PRMT expands an entry to w = (4 * y) << 25 | x: the low 5 bits feed a wrap-mode funnel shift
    // directly, the top 7 are the byte offset of FIT row y.
    uint16_t anch[BLK_MAX_ANCHORS + 8];
};

__device__ __forceinline__ void blk_load(BlkSmem &sm, const uint4 *__restrict__ st, long long g, int lane) {
    if (lane < BLK_VEC) {
        uint4 v = ld_stream(st + g * BLK_VEC + lane);
        sm.st[4 * lane + 0] = v.x; sm.st[4 * lane + 1] = v.y; sm.st[4 * lane + 2] = v.z; sm.st[4 * lane + 3] = v.w;
    }
    __syncwarp();
}
__device__ __forceinline__ void blk_store(const BlkSmem &sm, uint4 *__restrict__ st, long long g, int lane) {
    __syncwarp();
    if (lane < BLK_VEC)
        st_stream(st + g * BLK_VEC + lane,
                  make_uint4(sm.st[4 * lane + 0], sm.st[4 * lane + 1], sm.st[4 * lane + 2], sm.st[4 * lane + 3]));
}
// new_state (BlokusEnvironment.py:248-289): empty board, round 0, four full inventories, player 0 to move
__device__ __forceinline__ void blk_new_state(BlkSmem &sm, int lane) {
    __syncwarp();
    for (int i = lane; i < BLK_WORDS; i += 32) sm.st[i] = (i >= 80 && i < 84) ? ((1u << BLK_NPIECE) - 1u) : 0u;
    __syncwarp();
}

// A and ANC rows of player c (0-based) for the board in sm.st; fills sm.A, sm.anc and (LIST) the row-major anchor
// list sm.anch and returns #anchors, or (!LIST) returns the mask of the rows that hold an anchor.
template <bool LIST>
__device__ __forceinline__ int blk_allowed_and_anchors(BlkSmem &sm, int c, int round, int lane) {
    __syncwarp();
    uint32_t a = 0, an = 0;
    if (lane < 20) {
        const int y = lane;
        uint32_t own = sm.st[20 * c + y];
        uint32_t occ = sm.st[y] | sm.st[20 + y] | sm.st[40 + y] | sm.st[60 + y];
        uint32_t up = y > 0 ? sm.st[20 * c + y - 1] : 0u, dn = y < 19 ? sm.st[20 * c + y + 1] : 0u;
        uint32_t n4 = up | dn | (own << 1) | (own >> 1);                       // is_valid_adjacents
        a = ~occ & ~n4 & BLK_ROWMASK;                                          // is_valid_cell
        if (round == 0) {                                                      // PLAYER_DEFAULT_CORNERS (board.py:50)
            const int cx = (c & 1) ? 19 : 0, cy = (c & 2) ? 19 : 0;
            an = (y == cy) ? (1u << cx) : 0u;
        } else {
            uint32_t d4 = (up << 1) | (up >> 1) | (dn << 1) | (dn >> 1);       // check_valid_corner (board.py:127-154)
            an = a & d4;
        }
    }
    if (lane < 24) sm.A[lane] = a << 4;
    if (lane < 20) sm.anc[lane] = an;
    if (!LIST) {                                             // callers only need "which rows hold an anchor"
        __syncwarp();
        return (int)__ballot_sync(0xffffffffu, an != 0u);
    }
    // row-major anchor list: exclusive prefix of the per-row counts
    int cnt = __popc(an), pre = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) pre = (int)warp_scan_step((uint32_t)pre, d);
    const int total = __shfl_sync(0xffffffffu, pre, 31);
    int pos = pre - cnt;
    while (an) {
        const int x = __ffs((int)an) - 1;
        an &= an - 1;
        sm.anch[pos++] = (uint16_t)((4 * lane) << 9 | x);
    }
    if (lane < 4) sm.anch[total + lane] = 24;                // padding: never fits
    __syncwarp();
    return total;
}

// ---- FIT boards, lanes = shapes ---------------------------------------------------------------------------------
// zero every board once per kernel (the passes only write rows 0..19 of the boards they build)
__device__ __forceinline__ void blk_zero_fit(BlkSmem &sm, int lane) {
    uint4 *f4 = (uint4 *)sm.F;
    for (int i = lane; i < (BLK_FSLOTS * BLK_FROWS + 4) / 4; i += 32) f4[i] = make_uint4(0u, 0u, 0u, 0u);
}

// shape 0 (the monomino): FIT = A.  Returns its non-empty flag.
__device__ __forceinline__ uint32_t blk_tree_root(BlkSmem &sm, int lane) {
    const uint32_t f = lane < 20 ? sm.A[lane] << (BLK_OFF_LE4 - 4) : 0u;
    if (lane < 20) sm.F[4 + lane] = f;
    const uint32_t ne = __any_sync(0xffffffffu, f != 0u) ? 1u : 0u;
    __syncwarp();
    return ne;
}

// One pass: lane l builds FIT of shape s0 + l (if s0 + l < s1, a held piece needs it and its parent is non-empty).
// Returns the ballot of the non-empty boards (bit l = shape s0 + l).
__device__ __forceinline__ uint32_t blk_tree_pass(BlkSmem &sm, int s0, int s1, uint32_t ne, uint32_t inv, int lane) {
    const uint4 t = BLK_SHAPE_TAB_G[s0 + lane];
    const bool active = s0 + lane < s1 && (inv & t.y) != 0u && (ne >> (t.y >> 24) & 1u) != 0u;
    if (!__any_sync(0xffffffffu, active)) return 0u;
    uint32_t acc = 0u;
    if (active) {
        const char *pp = (const char *)sm.F + (t.x & 0xffffu);      // parent row 4 + py
        const char *pa = (const char *)sm.A + (t.x >> 24);          // A row cy
        char *po = (char *)sm.F + (t.w & 0xffffu);                  // own row 4
        // parent bit (qx + px + 8) and A bit (qx + cx + 4) both land on qx + 12: two multiplies by powers of two.  No
        // mask is needed: the shape has a cell in column 0, so px == 0 or cx == 0 and that term has no bit below 12.
        const uint32_t mp = 1u << (BLK_OFF_PENT - BLK_OFF_LE4 - ((t.x >> 16) & 7u)), mc = 1u << (BLK_OFF_PENT - 4 - ((t.x >> 20) & 7u));
#pragma unroll 10
        for (int r = 0; r < 20; r++) {
            const uint32_t f = (*(const uint32_t *)(pp + 4 * r) * mp) & (*(const uint32_t *)(pa + 4 * r) * mc);
            *(uint32_t *)(po + 4 * r) = f;
            acc |= f;
        }
    }
    const uint32_t m = __ballot_sync(0xffffffffu, acc != 0u);
    __syncwarp();
    return m;
}

// ALL shapes of 2..4 cells (shapes 1..27: 2 dominoes, 6 trominoes, 19 tetrominoes) in ONE pass, straight from A:
// FIT_s[q] = AND_i A[q + cell_i(s)] with the shape's own <= 4 cells (shorter shapes repeat cell 0).  As three tree
// levels these 27 shapes cost three dependent passes that keep 2, 6 and 19 lanes busy (2 terms per row each); merged
// they are one pass with four terms per row and 27 busy lanes.  (Measured: levels 2 + 3 merged -2.5 % of the step.)
__device__ __forceinline__ uint32_t blk_tree_pass_le4(BlkSmem &sm, uint32_t ne, uint32_t inv, int lane) {
    const uint4 t = BLK_SHAPE_TAB_G[1 + lane];                      // (the table is padded past the last shape)
    const bool active = lane < BLK_NSHAPE_LE4 - 1 && (inv & t.y) != 0u && (ne & 1u) != 0u;
    if (!__any_sync(0xffffffffu, active)) return 0u;
    uint32_t acc = 0u;
    if (active) {
        const char *a0 = (const char *)sm.A + 4 * (t.z >> 3 & 7u), *a1 = (const char *)sm.A + 4 * (t.z >> 9 & 7u);
        const char *a2 = (const char *)sm.A + 4 * (t.z >> 15 & 7u), *a3 = (const char *)sm.A + 4 * (t.z >> 21 & 7u);
        // A bit (qx + dx_i + 4) lands on qx + 8: a multiply by 2^(4 - dx_i) per cell (IMAD; a right shift is an ALU-pipe SHF).
        // No mask: the cell in column 0 contributes no bit below 8.
        const uint32_t m0 = 16u >> (t.z & 7u), m1 = 16u >> (t.z >> 6 & 7u), m2 = 16u >> (t.z >> 12 & 7u), m3 = 16u >> (t.z >> 18 & 7u);
        char *po = (char *)sm.F + (t.w & 0xffffu);                  // own row 4
#pragma unroll 10
        for (int r = 0; r < 20; r++) {
            const uint32_t f = (*(const uint32_t *)(a0 + 4 * r) * m0) & (*(const uint32_t *)(a1 + 4 * r) * m1) &
                               (*(const uint32_t *)(a2 + 4 * r) * m2) & (*(const uint32_t *)(a3 + 4 * r) * m3);
            *(uint32_t *)(po + 4 * r) = f;
            acc |= f;
        }
    }
    const uint32_t m = __ballot_sync(0xffffffffu, acc != 0u);
    __syncwarp();
    return m << 1;
}

// the shapes of pentomino group g into slots 28..; returns their non-empty flags (bit = shape - group start)
__device__ __forceinline__ uint32_t blk_tree_group(BlkSmem &sm, int g, uint32_t ne, uint32_t inv, int lane) {
    __syncwarp();                // the previous group's readers are done with the shared slots
    return blk_tree_pass(sm, BLK_GROUP_S0[g], BLK_GROUP_S0[g + 1], ne, inv, lane);
}

// any-move test, lanes = the shapes [s0, s1) of n cells: does a held piece have a placement of one of these shapes
// that covers an anchor?  flags: bit l = FIT of shape s0 + l is non-empty; rows = the board rows that hold an anchor.
__device__ __forceinline__ bool blk_any_pass(BlkSmem &sm, int s0, int s1, int n, uint32_t flags, uint32_t inv, uint32_t rows,
                                             int lane) {
    const uint4 t = BLK_SHAPE_TAB_G[s0 + lane];
    const bool active = s0 + lane < s1 && (inv >> (t.w >> 16 & 31u) & 1u) != 0u && (flags >> lane & 1u) != 0u;
    if (!__any_sync(0xffffffffu, active)) return false;
    uint32_t acc = 0u;
    if (active) {
        const char *po = (const char *)sm.F + (t.w & 0xffffu);
        // OR_k shift(FIT_s, cell_k) & ANC on the anchor rows (short shapes repeat cell 0)
        const char *p0 = po - 4 * (int)(t.z >> 3 & 7u), *p1 = po - 4 * (int)(t.z >> 9 & 7u), *p2 = po - 4 * (int)(t.z >> 15 & 7u);
        const char *p3 = po - 4 * (int)(t.z >> 21 & 7u), *p4 = po - 4 * (int)(t.z >> 27 & 7u);
        const uint32_t off = n > 4 ? BLK_OFF_PENT : BLK_OFF_LE4;     // column 0 of these boards
        const uint32_t h0 = off - (t.z & 7u), h1 = off - (t.z >> 6 & 7u), h2 = off - (t.z >> 12 & 7u);
        const uint32_t h3 = off - (t.z >> 18 & 7u), h4 = off - (t.z >> 24 & 7u);
#pragma unroll 1
        for (uint32_t rm = rows; rm; rm &= rm - 1u) {
            const int r4 = 4 * (__ffs((int)rm) - 1);
            uint32_t d = __funnelshift_r(*(const uint32_t *)(p0 + r4), 0u, h0) | __funnelshift_r(*(const uint32_t *)(p1 + r4), 0u, h1);
            if (n > 2) d |= __funnelshift_r(*(const uint32_t *)(p2 + r4), 0u, h2);
            if (n > 3) d |= __funnelshift_r(*(const uint32_t *)(p3 + r4), 0u, h3);
            if (n > 4) d |= __funnelshift_r(*(const uint32_t *)(p4 + r4), 0u, h4);
            acc |= d & *(const uint32_t *)((const char *)sm.anc + r4);
        }
    }
    return __any_sync(0xffffffffu, acc != 0u) != 0;
}

// AI.check_moves (ai.py:36-42): does player c holding `inv` have any move on the board in sm.st?
__device__ __forceinline__ int blk_any_move(BlkSmem &sm, int c, int round, uint32_t inv, int lane, bool &zeroed) {
    inv = __reduce_or_sync(0xffffffffu, inv);
    if (inv == 0u) return 0;
    const uint32_t rows = (uint32_t)blk_allowed_and_anchors<false>(sm, c, round, lane);
    if (rows == 0u) return 0;
    // round 0: the anchor is the player's corner whatever it holds (board.py:177-179); every placement covers its
    // anchor, so an occupied / blocked corner means no move at all (and no tree has to be built to find that out)
    if (round == 0 && !__any_sync(0xffffffffu, lane < 20 && (sm.anc[lane] & (sm.A[lane] >> 4)) != 0u)) return 0;
    if (inv & 1u) return 1;                                  // the monomino fits on every anchor that is an allowed cell
    if (!zeroed) { blk_zero_fit(sm, lane); zeroed = true; __syncwarp(); }  // (the common case never gets here)
    uint32_t ne = blk_tree_root(sm, lane);
    ne |= blk_tree_pass_le4(sm, ne, inv, lane);              // (this is the negative path: the whole tree is needed anyway)
#pragma unroll 1
    for (int level = 2; level <= 4; level++) {
        const int s0 = BLK_LEVEL_S0[level - 1];
        if (blk_any_pass(sm, s0, BLK_LEVEL_S0[level], level, ne >> s0, inv, rows, lane)) return 1;
    }
#pragma unroll 1
    for (int g = 0; g < BLK_NGROUP; g++) {
        if (!(inv & ((1u << BLK_GROUP_P0[g + 1]) - (1u << BLK_GROUP_P0[g])))) continue;
        const uint32_t ne5 = blk_tree_group(sm, g, ne, inv, lane);
        if (ne5 != 0u && blk_any_pass(sm, BLK_GROUP_S0[g], BLK_GROUP_S0[g + 1], 5, ne5, inv, rows, lane)) return 1;
    }
    return 0;
}

// ---- emission ---------------------------------------------------------------------------------------------------
// One held piece p, anchors in groups of four.  Lanes = (anchor a = lane >> 3 of the group, orientation o = lane & 7);
// a lane tests the piece's <= 5 shifts k for its (anchor, orientation):
//   FIT_s[anchor - cell_k]  =  bit (x + 4 - dx_k) of row (y + 4 - dy_k) of the orientation's board
// = one address add, one LDS, one add, one wrap-mode shift (the anchor word's low bits are the column) and one funnel
// shift that pushes the hit bit into the lane's accumulator: no vote, no branch.  The accumulator ends up with one
// byte per group (5 hit bits), so ONE SWAR popcount and ONE shuffle scan position all hits of up to 16 anchors:
// lane order (a, o) followed by k IS the reference's order (anchor row-major -> orientation -> shift), and the action
// id is anchor code + piece * 16000 + o * 5 + k.  Each lane then stores its own <= 5 ids of a group.
// MODE (compile time):
//   BLK_STORE   store the ids into out[base..cap) and return base + the piece's count;
//   BLK_COUNT   return base + the piece's count: no scan and no store, one popcount per lane and chunk and ONE warp
//               reduction per piece;
//   BLK_SELECT  return the id at index `cap` of the piece's own list (base 0, out unused; cap < the piece's count):
//               the store phase with the stores replaced by "the lane whose range holds index cap keeps that id".
enum { BLK_STORE = 0, BLK_COUNT = 1, BLK_SELECT = 2 };
template <bool PENT, int MODE = BLK_STORE>
__device__ __forceinline__ int blk_emit_piece(BlkSmem &sm, uint32_t nemask, int p, int na, int lane, int base,
                                              int32_t *__restrict__ out, int cap) {
    // nemask: the non-empty flags the piece's table entries index (`ne`, or its pentomino group's `ne5`)
    const int n = PENT ? 5 : (int)BLK_PIECE_SIZE[p];
    const int o = lane & 7, a = lane >> 3;
    const uint4 *e = BLK_ORIENT_TAB_G[p * 8 + o];
    const uint4 e0 = e[0], e1 = e[1], e2 = e[2];
    const bool v = (nemask >> e2.z & 1u) != 0u;
    if (!__any_sync(0xffffffffu, v)) return base;            // none of the piece's shapes fits anywhere
    const char *fb = (const char *)sm.F;
    const uint32_t f0 = e0.x, f1 = e0.y, f2 = e0.z, f3 = e0.w, f4 = e1.x;          // row offsets, bytes
    const uint32_t c0 = e1.y, c1 = e1.z, c2 = e1.w, c3 = e2.x, c4 = e2.y;          // column constants
    const int val00 = p * 16000 + o * 5;
    int cnt = 0, sel = -1;                                   // BLK_COUNT: the lane's hits; BLK_SELECT: the id found
#define BLK_TEST(fk, ck) hh = __funnelshift_r(hh, __funnelshift_r(*(const uint32_t *)(fb + ((fk) + row)), 0u, w + (ck)), 1)
#pragma unroll 1
    for (int a0 = 0; a0 < na; a0 += 16) {                    // chunks of four groups (one chunk in practice: ~8 anchors)
        const int ng = min(4, (na - a0 + 3) >> 2);
        const uint16_t *al = sm.anch + a0 + a;
        uint32_t hh = 0u, wg[4];
        // both group loops are fully unrolled (the selectors become immediates, the anchor words stay in registers,
        // no loop counters); groups past the end of the list are skipped by a warp-uniform test
#pragma unroll
        for (int g = 0; g < 4; g++) {
            if (g < ng) {
                wg[g] = al[4 * g];                           // (the list is padded with never-fitting anchors)
                const uint32_t w = __byte_perm(wg[g], 0u, 0x1440u);
                const uint32_t row = w >> 25;
                BLK_TEST(f0, c0);
                if (n > 1) BLK_TEST(f1, c1);
                if (n > 2) BLK_TEST(f2, c2);
                if (n > 3) BLK_TEST(f3, c3);
                if (n > 4) BLK_TEST(f4, c4);
                hh >>= 8 - n;                                // one byte per group
            } else {
                wg[g] = 0u;
                hh >>= 8;
            }
        }
        hh = v ? hh : 0u;                                    // byte g = hits of (anchor a0 + 4 g + a, o), bit k = shift k
        if (MODE == BLK_COUNT) {
            cnt += __popc(hh);
            continue;
        }
        if (!__any_sync(0xffffffffu, hh != 0u)) continue;
        uint32_t cc = hh - ((hh >> 1) & 0x55555555u);        // per-byte popcount
        cc = (cc & 0x33333333u) + ((cc >> 2) & 0x33333333u);
        cc = (cc + (cc >> 4)) & 0x0f0f0f0fu;
        uint32_t incl = cc;                                  // per-byte inclusive scan over the lanes (sums <= 160)
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) incl = warp_scan_step(incl, d);
        const uint32_t tot = __shfl_sync(0xffffffffu, incl, 31), excl = incl - cc;
        const bool careful = base + (int)((tot * 0x01010101u) >> 24) > cap;        // rare: the caller's list is too short
#pragma unroll
        for (int g = 0; g < 4; g++) {
            const int tg = (int)((tot >> (8 * g)) & 0xffu);
            if (tg == 0) continue;                           // (warp-uniform) no hit on these four anchors / no such group
            uint32_t h = (hh >> (8 * g)) & 0xffu;
            int pos = base + (int)((excl >> (8 * g)) & 0xffu);
            base += tg;
            if (MODE == BLK_STORE && careful)                // drop the ids that do not fit (the count stays complete)
                while (h != 0u && __popc(h) > max(cap - pos, 0)) h &= ~(0x80000000u >> __clz((int)h));
            const uint32_t w = wg[g];
            const int val0 = (int)(w >> 9) * 200 + (int)(w & 31u) * 40 + val00;      // (y * 20 + x) * 40 + ...
            if (MODE == BLK_SELECT) {                        // ids pos .. pos + popc(h) - 1 are this lane's
                if (pos <= cap && cap < pos + __popc(h)) sel = val0 + (int)__fns(h, 0u, cap - pos + 1);
                continue;
            }
            // (32-bit running index: a 64-bit running pointer costs predicated 64-bit adds and moves per store)
            if (h & 1u) st_global_u32(out + pos++, val0);
            if (h & 2u) st_global_u32(out + pos++, val0 + 1);
            if (h & 4u) st_global_u32(out + pos++, val0 + 2);
            if (h & 8u) st_global_u32(out + pos++, val0 + 3);
            if (h & 16u) st_global_u32(out + pos, val0 + 4);
        }
        if (MODE == BLK_SELECT && base > cap) break;        // (warp-uniform) found
    }
#undef BLK_TEST
    if (MODE == BLK_COUNT) return base + __reduce_add_sync(0xffffffffu, cnt);
    if (MODE == BLK_SELECT) return (int)__reduce_or_sync(0xffffffffu, (uint32_t)(sel + 1)) - 1;   // one lane holds it
    return base;
}

// the monomino's id at index i of its list after round 0 (anchor i >> 3, orientation i & 7, shift 0; see below)
__device__ __forceinline__ int blk_monomino_id(const BlkSmem &sm, int i) {
    const uint32_t w = sm.anch[i >> 3];
    return (int)(w >> 9) * 200 + (int)(w & 31u) * 40 + 5 * (i & 7);
}

// Enumerate the legal moves of player c holding `inv` on the board in sm.st.
//   MODE == BLK_STORE:  action ids in the reference's order into out[0..cap), returns the full count.
//   MODE == BLK_SELECT: a uniform random pick without the list.  A count pass (the same enumeration without the store
//     phase; lane p keeps the count of piece p) gives the length n; for n > 0 the pick is the id at index rnd % n of
//     the full list, which a warp scan over the per-piece counts turns into a piece p* and an index into its ids, and
//     a select pass over p* alone finds.  *pick = that id (-1 if n == 0); returns n.  out / cap are unused.
template <int MODE = BLK_STORE>
__device__ __forceinline__ int blk_enumerate(BlkSmem &sm, int c, int round, uint32_t inv, int lane,
                                             int32_t *__restrict__ out, int cap, uint32_t rnd = 0u, int *pick = nullptr) {
    constexpr int EMIT = MODE == BLK_STORE ? BLK_STORE : BLK_COUNT;
    inv = __reduce_or_sync(0xffffffffu, inv);                // same in every lane
    if (MODE == BLK_SELECT) *pick = -1;
    const int na = blk_allowed_and_anchors<true>(sm, c, round, lane);
    if (na == 0 || inv == 0u) return 0;
    uint32_t ne = blk_tree_root(sm, lane);
    ne |= blk_tree_pass_le4(sm, ne, inv, lane);
    int base = 0, pcount = 0, glast = -1;                    // (BLK_SELECT) count of piece `lane`, last group built
    uint32_t ne5last = 0u;
    uint32_t small = inv & ((1u << BLK_GROUP_P0[0]) - 1u);                                   // pieces of <= 4 cells
    if ((small & 1u) && round != 0) {
        // the monomino needs no test after round 0: every anchor is an allowed cell (ANC = A & D4), so it fits on each
        // in all 8 orientations (k = 0) -- ids (y * 20 + x) * 40 + 5 o in anchor order, written 32 at a time
        if (MODE == BLK_STORE)
            for (int i = lane; i < 8 * na; i += 32)
                if (i < cap) st_global_u32(out + i, blk_monomino_id(sm, i));
        if (lane == 0) pcount = 8 * na;
        base = 8 * na;
        small &= ~1u;
    }
#pragma unroll 1
    for (uint32_t rest = small; rest; rest &= rest - 1u) {
        const int p = __ffs((int)rest) - 1, next = blk_emit_piece<false, EMIT>(sm, ne, p, na, lane, base, out, cap);
        if (lane == p) pcount = next - base;
        base = next;
    }
#pragma unroll 1
    for (int g = 0; g < BLK_NGROUP; g++) {                                                   // pentominoes, group by group
        uint32_t rest = inv & ((1u << BLK_GROUP_P0[g + 1]) - (1u << BLK_GROUP_P0[g]));
        if (rest == 0u) continue;
        const uint32_t ne5 = blk_tree_group(sm, g, ne, inv, lane);
        glast = g;
        ne5last = ne5;
        if (ne5 == 0u) continue;
#pragma unroll 1
        for (; rest; rest &= rest - 1u) {
            const int p = __ffs((int)rest) - 1, next = blk_emit_piece<true, EMIT>(sm, ne5, p, na, lane, base, out, cap);
            if (lane == p) pcount = next - base;
            base = next;
        }
    }
    if (MODE == BLK_STORE || base == 0) return base;
    // pick: piece p* = the first piece whose inclusive prefix count exceeds r, j = r - the ids before p*
    const uint32_t r = rnd % (uint32_t)base;
    int incl = pcount;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) incl = (int)warp_scan_step((uint32_t)incl, d);
    const int ps = __popc(__ballot_sync(0xffffffffu, (uint32_t)incl <= r));
    const int j = (int)r - __shfl_sync(0xffffffffu, incl - pcount, ps);
    if (ps == 0 && round != 0) {
        *pick = blk_monomino_id(sm, j);
    } else if (ps < BLK_GROUP_P0[0]) {
        *pick = blk_emit_piece<false, BLK_SELECT>(sm, ne, ps, na, lane, 0, out, j);   // the <= 4-cell boards are intact
    } else {
        const int g = BLK_PIECE_GROUP[ps];
        if (g != glast) ne5last = blk_tree_group(sm, g, ne, inv, lane);          // a later group overwrote its boards
        *pick = blk_emit_piece<true, BLK_SELECT>(sm, ne5last, ps, na, lane, 0, out, j);
    }
    return base;
}

// Is action id `aid` a legal move of player c holding `minv` on the board in sm.st?  (== membership in the valid
// list: the piece is held, the anchor is an anchor, every cell of the placement is allowed.)  Warp-uniform result;
// `add` receives the lane's row of the placement, `pc` / `size` the piece.  Leaves sm.A / sm.anc of player c behind.
__device__ __forceinline__ bool blk_validate(BlkSmem &sm, int c, int round, uint32_t minv, int aid, int lane,
                                             uint32_t &add, int &pc, int &size) {
    // decode ((piece*400 + y*20 + x)*8 + o)*5 + k   (string form: BlokusEnvironment.py:55-106)
    const int piece = aid / 16000, rem = aid - piece * 16000, cell = rem / 40, ok = rem - cell * 40;
    const int o = ok / 5, k = ok - o * 5;
    bool legal = aid >= 0 && piece < BLK_NPIECE;
    pc = legal ? piece : 0;
    size = BLK_PIECE_SIZE[pc];
    legal = legal && k < size && (minv >> pc & 1u);
    const uint32_t e = BLK_ID_TAB[BLK_PIECE_ID0[pc] + (legal ? o * size + k : 0)];
    const uint32_t cells = BLK_SHAPE_CELLS[e & 127u];
    const int ay = legal ? cell / 20 : 0, ax = legal ? cell - ay * 20 : 0;
    const int qx = ax - (int)((e >> 7) & 7u), qy = ay - (int)((e >> 10) & 7u);
    blk_allowed_and_anchors<false>(sm, c, round, lane);              // A / ANC of the player
    legal = legal && qx >= 0 && qy >= 0 && (sm.anc[ay] >> ax & 1u);
    add = 0u;
#pragma unroll
    for (int i = 0; i < 5; i++) {
        const uint32_t cd = cells >> (6 * i);
        const int x = qx + (int)(cd & 7u), y = qy + (int)((cd >> 3) & 7u);
        // y <= 23 by construction (rows 20..23 of A are zero), x may exceed 19 -> bit not in A
        legal = legal && x >= 0 && y >= 0 && x < 20 && (sm.A[min(max(y, 0), 23)] >> (max(x, 0) + 4) & 1u);
        add |= (y == lane && x >= 0 && x < 20) ? (1u << x) : 0u;
    }
    return legal;
}

// ---- is_valid_action (BlokusEnvironment.py:667-719): is actions[g] in the valid list of `player` (< 0: the game's
// mover)?  '' (-1) is not.  One warp per game, no enumeration.
__global__ void __launch_bounds__(32 * BLK_WARPS)
blokus_is_valid_kernel(const uint4 *__restrict__ st, const int32_t *__restrict__ actions, uint8_t *__restrict__ valid,
                       long long B, int player, int flags) {
    __shared__ BlkSmem smem[BLK_WARPS];
    const int lane = BLK_WARPS == 1 ? (int)threadIdx.x : (int)(threadIdx.x & 31), wid = BLK_WARPS == 1 ? 0 : (int)(threadIdx.x >> 5);
    const long long g = (long long)blockIdx.x * BLK_WARPS + wid;
    if (g >= B) return;
    BlkSmem &sm = smem[wid];
    blk_load(sm, st, g, lane);
    if ((flags & CRL_FLAG_AUTO_RESET) && (sm.st[85] >> 16 & 1u)) blk_new_state(sm, lane);
    const uint32_t meta = sm.st[85];
    const int c = player >= 0 ? player : (int)(meta >> 8 & 3u);
    uint32_t add;
    int pc, size;
    const bool legal = blk_validate(sm, c, (int)(meta & 0xffu), sm.st[80 + c], actions[g], lane, add, pc, size);
    if (lane == 0) valid[g] = legal ? 1 : 0;
}

// ---- valid_actions: one warp per game.  player < 0: the game's current mover.
__global__ void __launch_bounds__(32 * BLK_WARPS)
blokus_legal_kernel(const uint4 *__restrict__ st, int32_t *__restrict__ counts, int32_t *__restrict__ ids, int cap,
                    crl_u64 *stats, long long B, int player, int flags) {
    __shared__ BlkSmem smem[BLK_WARPS];
    __shared__ int sm_stat[CRL_NSTAT];
    BlockStats bs{sm_stat};
    if (stats) bs.init();
    const int lane = BLK_WARPS == 1 ? (int)threadIdx.x : (int)(threadIdx.x & 31), wid = BLK_WARPS == 1 ? 0 : (int)(threadIdx.x >> 5);
    const long long g = (long long)blockIdx.x * BLK_WARPS + wid;
    if (g < B) {
        BlkSmem &sm = smem[wid];
        blk_load(sm, st, g, lane);
        if ((flags & CRL_FLAG_AUTO_RESET) && (sm.st[85] >> 16 & 1u)) blk_new_state(sm, lane);
        const uint32_t meta = sm.st[85];
        const int c = player >= 0 ? player : (int)(meta >> 8 & 3u);
        const bool stuck = (sm.st[87] >> c & 1u) != 0u;       // cached by the step kernel: no move any more
        int32_t *out = ids + g * cap;
#ifndef CRL_HOSTSIM
        asm volatile("" : "+l"(out));         // keep the game's list base in one register pair: a store is IMAD.WIDE + STG
#endif
        int n = 0;
        if (!stuck) {
            blk_zero_fit(sm, lane);
            __syncwarp();
            n = blk_enumerate(sm, c, (int)(meta & 0xffu), sm.st[80 + c], lane, out, cap);
        }
        if (lane == 0) {
            counts[g] = n;
            if (stats) atomicAdd(&sm_stat[ST_NVALID], n);
        }
    }
    if (stats) bs.flush(stats);
}

// ---- next_state: one warp per game.
// BlkStepOut: what one next_state produced, every field warp-uniform.
// result record, 8 bytes: int8 reward | u8 flags (1 terminal, 2 illegal action, 4 placed) | u8 winners mask |
//                         u8 ranking bits (bit p = rank of p: winners 0, others 1) | u8 next mover |
//                         u8 next-players mask (1 << next mover) | u8 terminal (0 / 1) | 1 unused
//                         (the last two repeat information as plain bytes so that the host layer returns VIEWS of the
//                         record -- next_state's new_players and terminal -- without any element-wise decoding launch)
struct BlkStepOut {
    int mover, reward, terminal, error, placed, winners;
    uint32_t scores, ep_len;                                 // the new scores (one byte per player), episode steps
};
__device__ __forceinline__ uint2 blk_result(const BlkStepOut &o) {
    const uint32_t rank = 0xfu & ~(uint32_t)o.winners;
    const int nmover = (o.mover + 1) & 3;
    return make_uint2(((uint32_t)o.reward & 0xffu) | (uint32_t)(o.terminal | o.error << 1 | o.placed << 2) << 8 |
                          (uint32_t)o.winners << 16 | rank << 24,
                      (uint32_t)nmover | (1u << nmover) << 8 | (uint32_t)o.terminal << 16);
}

// next_state of the game in sm.st with action id `aid` (-1 = pass): the new state is committed into sm.st (the caller
// stores it).  `zeroed`: the FIT boards have been zeroed in this kernel (blk_any_move zeroes them on first use).
__device__ __forceinline__ BlkStepOut blk_step_apply(BlkSmem &sm, int aid, int lane, bool &zeroed) {
    const uint32_t meta = sm.st[85];
    const int round = (int)(meta & 0xffu), mover = (int)(meta >> 8 & 3u);
    uint32_t inv[4] = {sm.st[80], sm.st[81], sm.st[82], sm.st[83]};
    uint32_t scores = sm.st[84];
    uint32_t new_row = lane < 20 ? sm.st[20 * mover + lane] : 0u;
    int error = 0, placed = 0;
    if (aid >= 0) {
        uint32_t minv = 0, add;
#pragma unroll
        for (int q = 0; q < 4; q++) minv |= (q == mover) ? inv[q] : 0u;
        int pc, size;
        const bool legal = blk_validate(sm, mover, round, minv, aid, lane, add, pc, size);
        if (legal) {
            placed = 1;
            new_row |= add;                                                     // Board.update_board
            const uint32_t left = minv & ~(1u << pc);
            int gain = size + (left == 0 ? (pc == 0 ? 20 : 15) : 0);            // AI.update_player (ai.py:44-54)
#pragma unroll
            for (int q = 0; q < 4; q++) {
                if (q == mover) {
                    inv[q] = left;
                    scores = (scores & ~(0xffu << (8 * q))) | ((((scores >> (8 * q)) & 0xffu) + gain) & 0xffu) << (8 * q);
                }
            }
        } else {
            error = 1;                                                          // illegal id: flagged, applied as a pass
        }
    }
    // terminal test on the OLD board / OLD round with the NEW inventories (BlokusEnvironment.py:424, SURVEY B6)
    // `any` is order-independent; start with the players that have not moved yet this round (in round 0 the
    // ones that already moved have an occupied corner and would need a full, fruitless scan) and end with the mover.
    int any = 0;
    uint32_t stuck = sm.st[87] & 15u;
#pragma unroll 1
    for (int j = 1; j <= 4 && !any; j++) {
        const int q = (mover + j) & 3;
        if (stuck >> q & 1u) continue;                                          // known: no move any more
        uint32_t iq = 0;
#pragma unroll
        for (int r = 0; r < 4; r++) iq |= (r == q) ? inv[r] : 0u;
        any = blk_any_move(sm, q, round, iq, lane, zeroed);
        if (!any && j < 4 && round >= 1) stuck |= 1u << q;                      // (see the layout comment, w[87])
    }
    const int terminal = !any;
    int reward = 0, winners = 0;
    int sc[4] = {(int)(scores & 0xff), (int)(scores >> 8 & 0xff), (int)(scores >> 16 & 0xff), (int)(scores >> 24)};
    if (terminal) {                                                             // :425-440
        int mx = max(max(sc[0], sc[1]), max(sc[2], sc[3]));                     // max_score starts at 0, scores >= 0
        int ms = 0;
#pragma unroll
        for (int q = 0; q < 4; q++) ms |= (q == mover) ? sc[q] : 0;
#pragma unroll
        for (int q = 0; q < 4; q++) {
            winners |= (sc[q] == mx) ? (1 << q) : 0;
            reward += (sc[q] < ms || (sc[q] == ms && q < mover)) ? 1 : 0;       // index in the stable ascending sort
        }
    }
    const int nround = round + (mover == 3 ? 1 : 0), nmover = (mover + 1) & 3;  // :446-449
    const uint32_t ep_len = sm.st[86] + 1u;
    // commit into the shared copy (the caller stores it with 22 x 128-bit lanes)
    __syncwarp();
    if (lane < 20) sm.st[20 * mover + lane] = new_row;
    if (lane < 4) sm.st[80 + lane] = lane == 0 ? inv[0] : lane == 1 ? inv[1] : lane == 2 ? inv[2] : inv[3];
    if (lane == 4) sm.st[84] = scores;
    if (lane == 5) sm.st[85] = (uint32_t)(nround & 0xff) | (uint32_t)nmover << 8 | (uint32_t)terminal << 16;
    if (lane == 6) sm.st[86] = ep_len;
    if (lane == 7) sm.st[87] = stuck;
    return BlkStepOut{mover, reward, terminal, error, placed, winners, scores, ep_len};
}

__global__ void __launch_bounds__(32 * BLK_WARPS)
blokus_step_kernel(const uint4 *__restrict__ in, uint4 *__restrict__ outst, const int32_t *__restrict__ actions,
                   uint2 *__restrict__ result, crl_u64 *stats, long long B, int flags) {
    __shared__ BlkSmem smem[BLK_WARPS];
    __shared__ int sm_stat[CRL_NSTAT];
    BlockStats bs{sm_stat};
    if (stats) bs.init();
    const int lane = BLK_WARPS == 1 ? (int)threadIdx.x : (int)(threadIdx.x & 31), wid = BLK_WARPS == 1 ? 0 : (int)(threadIdx.x >> 5);
    const long long g = (long long)blockIdx.x * BLK_WARPS + wid;
    if (g < B) {
        BlkSmem &sm = smem[wid];
        blk_load(sm, in, g, lane);
        bool zeroed = false;
        if ((flags & CRL_FLAG_AUTO_RESET) && (sm.st[85] >> 16 & 1u)) blk_new_state(sm, lane);
        const BlkStepOut o = blk_step_apply(sm, actions[g], lane, zeroed);
        blk_store(sm, outst, g, lane);
        if (lane == 0) {
            result[g] = blk_result(o);
            if (stats) {
                atomicAdd(&sm_stat[ST_STEPS], 1);
                if (o.error) atomicAdd(&sm_stat[ST_ERRORS], 1);
                if (o.reward) atomicAdd(&sm_stat[ST_REWARD], (o.mover + 1) * o.reward);
                if (o.terminal) {
                    atomicAdd(&sm_stat[ST_EPISODES], 1);
                    atomicAdd(&sm_stat[ST_EPLEN], (int)o.ep_len);
                    if (!o.winners) atomicAdd(&sm_stat[ST_NOWIN], 1);
#pragma unroll
                    for (int q = 0; q < 4; q++) {
                        if (o.winners >> q & 1) atomicAdd(&sm_stat[ST_WINS + q], 1);
                        else atomicAdd(&sm_stat[ST_RANK + q], 1);
                        atomicAdd(&sm_stat[ST_SCORE + q], (int)(q == 3 ? o.scores >> 24 : o.scores >> (8 * q) & 0xffu));
                    }
                }
            }
        }
    }
    if (stats) bs.flush(stats);
}

// uniform random policy over the generated list: the (r0 % n)-th entry, pass (-1) if n == 0
__global__ void blokus_policy_random_kernel(const int32_t *__restrict__ counts, const int32_t *__restrict__ ids, int cap,
                                            int32_t *__restrict__ actions, long long B, crl_u64 seed, crl_u64 first_env,
                                            uint32_t step) {
    long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= B) return;
    int n = min(counts[g], cap);
    uint4 r = env_words(seed, first_env + (crl_u64)g, step, CRL_TAG_BLOKUS);
    actions[g] = n > 0 ? ids[g * cap + (long long)(r.x % (uint32_t)n)] : -1;
}

// One uniform random move of the mover of the game in sm.st (not terminal): unless the mover is known to be stuck
// (w[87]), blk_enumerate<BLK_SELECT> counts its ids and finds the one at index r % n of the FULL list, r = word `word`
// of philox(seed, env, step, tag); blk_step_apply applies it (a pass if n == 0).  n = the valid-move count.
__device__ __forceinline__ BlkStepOut blk_random_move(BlkSmem &sm, crl_u64 seed, crl_u64 env, uint32_t step, uint32_t tag,
                                                      int word, int lane, bool &zeroed, int &n) {
    const uint32_t meta = sm.st[85];
    const int c = (int)(meta >> 8 & 3u);
    int aid = -1;
    n = 0;
    if (!(sm.st[87] >> c & 1u)) {                            // not known to be stuck (w[87]): enumerate
        const uint4 w = env_words(seed, env, step, tag);
        const uint32_t r = word == 0 ? w.x : word == 1 ? w.y : word == 2 ? w.z : w.w;
        n = blk_enumerate<BLK_SELECT>(sm, c, (int)(meta & 0xffu), sm.st[80 + c], lane, nullptr, 0, r, &aid);
    }
    return blk_step_apply(sm, aid, lane, zeroed);
}

// Statistics slot `lane` of one env-step: the slots the step kernel adds, and the valid-move count n (the legal
// kernel's slot; 0 for a move whose list was not built).
__device__ __forceinline__ int blk_stat_slot(const BlkStepOut &o, int n, int lane) {
    int v = lane == ST_STEPS ? 1 : lane == ST_NVALID ? n : lane == ST_ERRORS ? o.error
          : lane == ST_REWARD ? (o.mover + 1) * o.reward : 0;
    if (o.terminal) {
        const int q = (lane - ST_WINS) & 3, sq = (lane - ST_SCORE) & 3, rq = (lane - ST_RANK) & 3;
        v += lane == ST_EPISODES ? 1 : lane == ST_EPLEN ? (int)o.ep_len : lane == ST_NOWIN ? (o.winners == 0)
           : (lane >= ST_WINS && lane < ST_WINS + 4) ? (o.winners >> q & 1)
           : (lane >= ST_SCORE && lane < ST_SCORE + 4) ? (int)(o.scores >> (8 * sq) & 0xffu)
           : (lane >= ST_RANK && lane < ST_RANK + 4) ? (~o.winners >> rq & 1) : 0;
    }
    return v;
}

// ---- K fused random-policy steps with auto-reset: one warp per game, the game stays in shared memory for all K steps.
// Step t is K x (legal kernel, player -1, auto-reset -> policy_random(step0 + t) -> step kernel, auto-reset) with the
// list never materialised: blk_enumerate<BLK_SELECT> counts the mover's ids and finds the one at index
// philox(env, step0 + t, tag 2)[0] % n of the FULL list, blk_step_apply applies it.  Statistics: lane s accumulates
// slot s of this game in 64 bits (no overflow for any K) and adds it to the CTA's row once.
__global__ void __launch_bounds__(32 * BLK_WARPS)
blokus_rollout_kernel(uint4 *__restrict__ st, uint2 *__restrict__ result, crl_u64 *stats, long long B, crl_u64 seed,
                      crl_u64 first_env, uint32_t step0, int K) {
    __shared__ BlkSmem smem[BLK_WARPS];
    const int lane = BLK_WARPS == 1 ? (int)threadIdx.x : (int)(threadIdx.x & 31), wid = BLK_WARPS == 1 ? 0 : (int)(threadIdx.x >> 5);
    const long long g = (long long)blockIdx.x * BLK_WARPS + wid;
    if (g >= B) return;
    BlkSmem &sm = smem[wid];
    blk_load(sm, st, g, lane);
    // Zeroed once: the passes rewrite rows 0..19 of the boards they build and every read of a board is masked by the
    // non-empty flags of the current pass, so a stale board from an earlier step is never used.
    blk_zero_fit(sm, lane);
    bool zeroed = true;
    crl_u64 acc = 0;
    uint2 rec = make_uint2(0u, 0u);
#pragma unroll 1
    for (int t = 0; t < K; t++) {
        __syncwarp();                                        // the previous step's commit (and the zeroing) is visible
        if (sm.st[85] >> 16 & 1u) blk_new_state(sm, lane);
        int n;
        const BlkStepOut o = blk_random_move(sm, seed, first_env + (crl_u64)g, step0 + (uint32_t)t, CRL_TAG_BLOKUS, 0, lane,
                                             zeroed, n);
        rec = blk_result(o);
        if (stats) acc += (crl_u64)(long long)blk_stat_slot(o, n, lane);     // the slots the legal and step kernels add
    }
    blk_store(sm, st, g, lane);
    if (result && lane == 0) result[g] = rec;
    if (stats && acc != 0) atomicAdd(stats + (blockIdx.x & (CRL_STAT_ROWS - 1)) * CRL_NSTAT + lane, acc);
}

// ---- one learner against uniform random opponents (crl_blokus_advance; the rule is stated in
// include/colosseum_b200_learner.h): one warp per game, like the rollout.  The learner's id, then opponent moves j =
// 0, 1, ... (blk_random_move on word j & 3 of tag CRL_TAG_OPPONENT + (j >> 2)) until the mover is `seat`; a move that
// ends the game is recorded and the game restarted at once.  A fresh game cannot end within its first 3 moves (every
// colour has a move in round 0), so at most 2 x 4 - 2 = 6 opponent moves are made: the loop bound never decides.
// Record, 8 bytes: int8 learner reward | u8 flags (1 finished, 2 illegal, 4 placed, 8 the learner did not move) |
// u8 winners | u8 opponent moves, then the finished game's scores (one byte per seat) or 0.  Statistics: lane s
// accumulates slot s in 64 bits and adds it to the CTA's row once.
__global__ void __launch_bounds__(32 * BLK_WARPS)
blokus_advance_kernel(uint4 *__restrict__ st, const int32_t *__restrict__ actions, int seat, uint2 *__restrict__ result,
                      crl_u64 *stats, long long B, crl_u64 seed, crl_u64 first_env, uint32_t step) {
    __shared__ BlkSmem smem[BLK_WARPS];
    const int lane = BLK_WARPS == 1 ? (int)threadIdx.x : (int)(threadIdx.x & 31), wid = BLK_WARPS == 1 ? 0 : (int)(threadIdx.x >> 5);
    const long long g = (long long)blockIdx.x * BLK_WARPS + wid;
    if (g >= B) return;
    BlkSmem &sm = smem[wid];
    blk_load(sm, st, g, lane);
    blk_zero_fit(sm, lane);                                  // once: see blokus_rollout_kernel
    bool zeroed = true;
    crl_u64 acc = 0;
    uint32_t flags = 0u, winners = 0u, scores = 0u;
    int reward = 0, j = 0;
    // a move that ended the game: record it for the learner (its index in the stable ascending sort of the scores), restart
    auto finish = [&](const BlkStepOut &o) {
        flags |= 1u;
        winners = (uint32_t)o.winners;
        scores = o.scores;
        const int ss = (int)(o.scores >> (8 * seat) & 0xffu);
        reward = 0;
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const int sq = (int)(o.scores >> (8 * q) & 0xffu);
            reward += (sq < ss || (sq == ss && q < seat)) ? 1 : 0;
        }
        blk_new_state(sm, lane);
    };
    __syncwarp();
    if (sm.st[85] >> 16 & 1u) blk_new_state(sm, lane);       // 1. it ended in an earlier call
    if (actions && (int)(sm.st[85] >> 8 & 3u) == seat) {     // 2. the learner's move
        const BlkStepOut o = blk_step_apply(sm, actions[g], lane, zeroed);
        flags |= (uint32_t)(o.error << 1 | o.placed << 2);
        if (stats) acc += (crl_u64)(long long)blk_stat_slot(o, 0, lane);
        if (o.terminal) finish(o);
    } else {
        flags |= 8u;
    }
#pragma unroll 1
    for (; j < 2 * 4 - 2; j++) {                             // 3. the opponents
        __syncwarp();                                        // the previous commit is visible
        if ((int)(sm.st[85] >> 8 & 3u) == seat) break;
        int n;
        const BlkStepOut o = blk_random_move(sm, seed, first_env + (crl_u64)g, step, CRL_TAG_OPPONENT + (uint32_t)(j >> 2), j & 3,
                                             lane, zeroed, n);
        if (stats) acc += (crl_u64)(long long)blk_stat_slot(o, n, lane);
        if (o.terminal) finish(o);
    }
    blk_store(sm, st, g, lane);
    if (lane == 0) result[g] = make_uint2(((uint32_t)reward & 0xffu) | flags << 8 | winners << 16 | (uint32_t)j << 24, scores);
    if (stats && acc != 0) atomicAdd(stats + (blockIdx.x & (CRL_STAT_ROWS - 1)) * CRL_NSTAT + lane, acc);
}

// a host-side policy's choice: actions[g] = the choice[g]-th entry of game g's valid list, pass (-1) if choice[g] is
// negative or past the end of the list.  (The policy reads the list LENGTHS on the host and answers with an index: the
// lists themselves -- kilobytes per game -- never cross PCIe.)
__global__ void blokus_pick_kernel(const int32_t *__restrict__ counts, const int32_t *__restrict__ ids, int cap,
                                   const int32_t *__restrict__ choice, int32_t *__restrict__ actions, long long B) {
    long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= B) return;
    const int n = min(counts[g], cap), c = choice[g];
    actions[g] = (c >= 0 && c < n) ? ids[g * cap + c] : -1;
}

__global__ void blokus_reset_kernel(uint4 *__restrict__ st, const uint8_t *__restrict__ mask, long long B) {
    long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= B * BLK_VEC) return;
    long long g = idx / BLK_VEC;
    int v = (int)(idx - g * BLK_VEC);
    if (mask && !mask[g]) return;
    const uint32_t full = (1u << BLK_NPIECE) - 1u;
    st[idx] = (v == 20) ? make_uint4(full, full, full, full) : make_uint4(0, 0, 0, 0);
}

// state_to_observation (BlokusEnvironment.py:721-768): one warp per game, bit-plane work instead of per-cell work.
//  1. lanes = source rows: the cell labels (relative id (c - player) & 3, or c + 1 in the absolute view) are folded into
//     label bit-planes x0, x1, x2 + the empty plane of the row (a handful of LOP3s, the label of a colour is uniform);
//  2. 4 cells at a time are spread to bytes with one multiply per plane ((nibble * 0x00204081) & 0x01010101: bit i ->
//     byte i) and combined into a word of int8 cells, 5 words per source row;
//  3. np.rot90(k=-player) is where the row lands in the staging tile: whole words for the unrotated views, bytes at
//     base + stride * x for the rotated ones; the game's 400 board bytes then leave with 25 128-bit stores.
// (The per-cell version -- 13 passes of 32 cells with a division, four plane tests and a byte store each -- executed
// 840 warp instructions per game.)
//  player >= 0: board int8[B][20][20] of relative player ids (-1 empty) rotated by np.rot90(k=-player);
//               pieces u8[B][4][21] rows by relative id; score int32[B][4] rolled by -player.
//  player == -1: absolute unpack: board = Board.board_contents (0 empty, 1..4 colour), pieces / score in seat order.
//  player == -2: like player >= 0 with every game seen by its own current mover (CRL_PLAYER_MOVER).
//  meta (optional) int32[B][4] = round, mover, terminal, episode steps.
__global__ void __launch_bounds__(32 * BLK_OBS_WARPS)
blokus_observe_kernel(const uint4 *__restrict__ st4, long long B, int player, int8_t *__restrict__ board,
                      uint8_t *__restrict__ pieces, int32_t *__restrict__ score, int32_t *__restrict__ meta) {
    __shared__ uint32_t sst[BLK_OBS_WARPS][BLK_WORDS];
    __shared__ __align__(16) uint32_t stage[BLK_OBS_WARPS][100];
    __shared__ __align__(16) uint32_t pstage[BLK_OBS_WARPS][24];         // the game's 84 inventory bytes (+ padding)
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const long long g = (long long)blockIdx.x * BLK_OBS_WARPS + wid;
    if (g >= B) return;
    uint32_t *s = sst[wid];
    if (lane < BLK_VEC) {
        const uint4 v = ld_stream(st4 + g * BLK_VEC + lane);
        s[4 * lane + 0] = v.x; s[4 * lane + 1] = v.y; s[4 * lane + 2] = v.z; s[4 * lane + 3] = v.w;
    }
    __syncwarp();
    if (player == -2) player = (int)(s[85] >> 8 & 3u);
    const bool rel = player >= 0;
    // 1. label planes of source row `lane`
    uint32_t x0 = 0u, x1 = 0u, x2 = 0u, occ = 0u;
    if (lane < 20) {
#pragma unroll
        for (int c = 0; c < 4; c++) {
            const uint32_t row = s[20 * c + lane];
            const int code = rel ? ((c - player) & 3) : c + 1;
            x0 |= (code & 1) ? row : 0u;
            x1 |= (code & 2) ? row : 0u;
            x2 |= (code & 4) ? row : 0u;
            occ |= row;
        }
    }
    const uint32_t xe = lane < 20 ? ~occ & BLK_ROWMASK : 0u;
    // 2. source row -> 20 int8 cells (5 words);  3. np.rot90(k=-player): source cell (y, x) lands at
    //    player 0 / absolute: (y, x)    1: (x, 19 - y)    2: (19 - y, 19 - x)    3: (19 - x, y)
    //    i.e. at byte  base + stride * x  of the staging tile, with base and stride constants of the lane
    if (lane < 20) {
        // three nibble -> bytes spreads per 4 cells, not four: a relative view has labels 0..3 (no bit 2) and -1 for the
        // empty cells; the absolute view has labels 1..4 and 0 for the empty cells (no empty plane)
        const uint32_t xt = rel ? xe : x2, kt = rel ? 255u : 4u;
        uint32_t w[5];
#pragma unroll
        for (int q = 0; q < 5; q++) {
            const uint32_t b0 = (((x0 >> (4 * q)) & 15u) * 0x00204081u) & 0x01010101u;
            const uint32_t b1 = (((x1 >> (4 * q)) & 15u) * 0x00204081u) & 0x01010101u;
            const uint32_t bt = (((xt >> (4 * q)) & 15u) * 0x00204081u) & 0x01010101u;
            w[q] = b0 + 2u * b1 + kt * bt;
        }
        if (player <= 0) {
            uint32_t *o = stage[wid] + 5 * lane;
#pragma unroll
            for (int q = 0; q < 5; q++) o[q] = w[q];
        } else {
            const int base = player == 1 ? 19 - lane : player == 2 ? 20 * (19 - lane) + 19 : 380 + lane;
            const int stride = player == 1 ? 20 : player == 2 ? -1 : -20;
            uint8_t *o = (uint8_t *)stage[wid] + base;
#pragma unroll
            for (int q = 0; q < 5; q++)
#pragma unroll
                for (int i = 0; i < 4; i++) o[stride * (4 * q + i)] = (uint8_t)(w[q] >> (8 * i));
        }
    }
    __syncwarp();
    if (lane < 25) ((uint4 *)(board + g * 400))[lane] = ((const uint4 *)stage[wid])[lane];
    // pieces[rel][piece]: lane p < 21 owns piece p of the four rows (4 byte stores into the staging tile), then the 84
    // bytes leave as 21 words (a game's inventory block starts at g * 84: 4-byte aligned).  (Three passes of 32 bytes with
    // a division each cost 90 of the kernel's 410 warp instructions per game.)
    if (lane < BLK_NPIECE) {
        uint8_t *pb = (uint8_t *)pstage[wid] + lane;
#pragma unroll
        for (int r = 0; r < 4; r++) {
            const int src = player >= 0 ? ((r + player) & 3) : r;
            pb[21 * r] = (uint8_t)(s[80 + src] >> lane & 1u);
        }
    }
    __syncwarp();
    if (lane < 21) ((uint32_t *)(pieces + g * 84))[lane] = pstage[wid][lane];
    if (lane < 4) {
        const int src = player >= 0 ? ((lane + player) & 3) : lane;
        score[g * 4 + lane] = (int)(s[84] >> (8 * src) & 0xffu);
        if (meta) {
            const uint32_t m = s[85];
            meta[g * 4 + lane] = lane == 0 ? (int)(m & 0xffu) : lane == 1 ? (int)(m >> 8 & 3u)
                                 : lane == 2 ? (int)(m >> 16 & 1u) : (int)s[86];
        }
    }
}

// import a reference-layout state: board int8[B][20][20] (0..4), inventory u8[B][4][21], scores int32[B][4],
// meta int32[B][4] = round, mover, terminal, episode steps
__global__ void blokus_pack_kernel(uint4 *__restrict__ st4, long long B, const int8_t *__restrict__ board,
                                   const uint8_t *__restrict__ pieces, const int32_t *__restrict__ score,
                                   const int32_t *__restrict__ meta) {
    uint32_t *st = (uint32_t *)st4;
    long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= B * BLK_WORDS) return;
    long long g = idx / BLK_WORDS;
    int w = (int)(idx - g * BLK_WORDS);
    uint32_t v = 0;
    if (w < 80) {
        int c = w / 20, y = w - c * 20;
        for (int x = 0; x < 20; x++) v |= (board[g * 400 + y * 20 + x] == c + 1) ? (1u << x) : 0u;
    } else if (w < 84) {
        for (int p = 0; p < BLK_NPIECE; p++) v |= pieces[g * 84 + (w - 80) * 21 + p] ? (1u << p) : 0u;
    } else if (w == 84) {
        for (int q = 0; q < 4; q++) v |= ((uint32_t)score[g * 4 + q] & 0xffu) << (8 * q);
    } else if (w == 85) {
        v = ((uint32_t)meta[g * 4] & 0xffu) | ((uint32_t)meta[g * 4 + 1] & 3u) << 8 | ((uint32_t)meta[g * 4 + 2] & 1u) << 16;
    } else if (w == 86) {
        v = (uint32_t)meta[g * 4 + 3];
    }
    st[idx] = v;
}

// ---- placements (include/colosseum_b200_placement.h): placement p = s * 400 + y * 20 + x, shape s with the top-left
// corner of its bounding box at (x, y).  (s, x, y) is legal for player c  <=>  c holds the piece of s, FIT_s[(x, y)]
// (every cell allowed) and a cell is an anchor:  mask_s = FIT_s & OR_k shift(ANC, -cell_k)  -- blk_any_pass with a
// store per row instead of an OR-reduction, and no emission phase at all.
#define BLK_NPLACEMENT (BLK_NSHAPE * 400)
#define BLK_ILLEGAL_ACTION (BLK_NPIECE * 16000)     // in no valid list: the step kernels flag it and apply a pass
#define BLK_MASK_VEC (BLK_NSHAPE * 20 / 4)          // uint4 per game of the mask uint32[91][20] (7 280 bytes)

// shape -> its image in player q's rotated frame (q = 0..3), for blokus_placement_to_action_kernel.  Passed BY VALUE
// (kernel parameter space), so it adds nothing to the constant banks the other kernels address.
struct BlkRotTab {
    uint8_t img[4][BLK_NSHAPE + 1];
};

// Row `lane` (< 20; 0 in lanes 20..31) of a 20 x 20 bit board -> row `lane` of the board in player r's frame (r = 1..3),
// the frame of blokus_observe_kernel: board cell (x, y) lands on (19 - y, x), (19 - x, 19 - y), (y, 19 - x).  With the
// transpose T (T[j] bit i = B[i] bit j: 20 ballots) the rotated rows are rev(T[y]), rev(B[19 - y]) and T[19 - y].
__device__ __forceinline__ uint32_t blk_rotate_row(uint32_t v, int r, int lane) {
    if (r & 1) {
        uint32_t t = 0u;
#pragma unroll
        for (int j = 0; j < 20; j++) {
            const uint32_t b = __ballot_sync(0xffffffffu, (v >> j) & 1u);
            t = lane == j ? b : t;
        }
        v = t;
    }
    v = __shfl_sync(0xffffffffu, v, r == 1 ? lane : (19 - lane) & 31);
    if (r != 3) v = __brev(v) >> 12;
    return lane < 20 ? v : 0u;
}

// Mask rows of the shapes [s0, s1), lanes = shapes: row y of shape s is FIT_s[y] & OR_k (anc[y + dy_k] >> dx_k) for a
// shape whose piece is held and whose board `flags` marks as built and non-empty (bit lane), zero rows otherwise.  The
// lane writes its shape's 80 contiguous bytes with five 128-bit stores and returns their popcount.  anc: the anchor
// rows with rows 20..23 zero (shapes are at most 5 rows tall); off: bit of column 0 in these FIT boards.
__device__ __forceinline__ int blk_mask_pass(const BlkSmem &sm, const uint32_t *anc, int s0, int s1, uint32_t flags,
                                             uint32_t inv, uint32_t off, uint4 *__restrict__ out, int lane) {
    if (s0 + lane >= s1) return 0;
    const uint4 t = BLK_SHAPE_TAB_G[s0 + lane];
    uint4 *o = out + (s0 + lane) * 5;
    if (!((inv >> (t.w >> 16 & 31u) & 1u) && (flags >> lane & 1u))) {
#pragma unroll
        for (int q = 0; q < 5; q++) o[q] = make_uint4(0u, 0u, 0u, 0u);
        return 0;
    }
    const uint32_t *f = (const uint32_t *)((const char *)sm.F + (t.w & 0xffffu));        // own row 4 (y = 0)
    const uint32_t *a0 = anc + (t.z >> 3 & 7u), *a1 = anc + (t.z >> 9 & 7u), *a2 = anc + (t.z >> 15 & 7u);
    const uint32_t *a3 = anc + (t.z >> 21 & 7u), *a4 = anc + (t.z >> 27 & 7u);           // (short shapes repeat cell 0)
    const uint32_t d0 = t.z & 7u, d1 = t.z >> 6 & 7u, d2 = t.z >> 12 & 7u, d3 = t.z >> 18 & 7u, d4 = t.z >> 24 & 7u;
    int cnt = 0;
#pragma unroll
    for (int q = 0; q < 5; q++) {
        uint32_t m[4];
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const int r = 4 * q + i;
            const uint32_t d = (a0[r] >> d0) | (a1[r] >> d1) | (a2[r] >> d2) | (a3[r] >> d3) | (a4[r] >> d4);
            m[i] = (f[r] >> off) & d & BLK_ROWMASK;
            cnt += __popc(m[i]);
        }
        o[q] = make_uint4(m[0], m[1], m[2], m[3]);
    }
    return cnt;
}

// ---- legal-placement masks: one warp per game, as the legal kernel.  A and ANC of the player (rotated into its frame
// for frame 1: legality only asks which cells are allowed and which are anchors, so it is invariant under the rotation),
// the tree passes of the legal kernel, and one mask pass per range of shapes (the <= 4-cell shapes, then each pentomino
// group).  player < 0: the game's mover.
__global__ void __launch_bounds__(32 * BLK_WARPS)
blokus_placement_mask_kernel(const uint4 *__restrict__ st, uint4 *__restrict__ mask, int32_t *__restrict__ counts,
                             long long B, int player, int frame, int flags) {
    __shared__ BlkSmem smem[BLK_WARPS];
    __shared__ uint32_t sanc[BLK_WARPS][24];                 // anchor rows, rows 20..23 zero
    const int lane = BLK_WARPS == 1 ? (int)threadIdx.x : (int)(threadIdx.x & 31), wid = BLK_WARPS == 1 ? 0 : (int)(threadIdx.x >> 5);
    const long long g = (long long)blockIdx.x * BLK_WARPS + wid;
    if (g >= B) return;
    BlkSmem &sm = smem[wid];
    uint32_t *anc = sanc[wid];
    blk_load(sm, st, g, lane);
    if ((flags & CRL_FLAG_AUTO_RESET) && (sm.st[85] >> 16 & 1u)) blk_new_state(sm, lane);
    const uint32_t meta = sm.st[85];
    const int c = player >= 0 ? player : (int)(meta >> 8 & 3u);
    const uint32_t inv = sm.st[80 + c];
    uint4 *out = mask + g * BLK_MASK_VEC;
    uint32_t rows = 0u;
    if (!(sm.st[87] >> c & 1u) && inv != 0u) rows = (uint32_t)blk_allowed_and_anchors<false>(sm, c, (int)(meta & 0xffu), lane);
    int cnt = 0;
    if (rows == 0u) {                                        // no anchor, no piece or known to be stuck: no placement
        for (int i = lane; i < BLK_MASK_VEC; i += 32) out[i] = make_uint4(0u, 0u, 0u, 0u);
    } else {
        uint32_t a = lane < 20 ? sm.A[lane] >> 4 : 0u, an = lane < 20 ? sm.anc[lane] : 0u;
        const int r = frame ? c : 0;
        if (r) {
            a = blk_rotate_row(a, r, lane);
            an = blk_rotate_row(an, r, lane);
            if (lane < 24) sm.A[lane] = a << 4;
        }
        if (lane < 24) anc[lane] = an;
        blk_zero_fit(sm, lane);
        __syncwarp();
        uint32_t ne = blk_tree_root(sm, lane);
        ne |= blk_tree_pass_le4(sm, ne, inv, lane);
        cnt = blk_mask_pass(sm, anc, 0, BLK_NSHAPE_LE4, ne, inv, BLK_OFF_LE4, out, lane);
#pragma unroll 1
        for (int gi = 0; gi < BLK_NGROUP; gi++) {
            const bool held = (inv & ((1u << BLK_GROUP_P0[gi + 1]) - (1u << BLK_GROUP_P0[gi]))) != 0u;
            const uint32_t ne5 = held ? blk_tree_group(sm, gi, ne, inv, lane) : 0u;
            cnt += blk_mask_pass(sm, anc, BLK_GROUP_S0[gi], BLK_GROUP_S0[gi + 1], ne5, inv, BLK_OFF_PENT, out, lane);
        }
    }
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if (counts && lane == 0) counts[g] = cnt;
}

// ---- placement -> canonical action id: one warp per game, every lane computes the same (warp-uniform) answer.  A
// frame-1 placement is mapped back to the board frame (the inverse of player r's rotation is player 4 - r's); held,
// fit and anchor are checked on the A and ANC rows as blk_validate checks an id.  The id is the first one of the
// reference's list with this placement: the anchor is the row-major first anchored cell, the orientation the lowest
// one of the piece whose shape is s, the shift the index of the anchor's cell in that orientation.
__global__ void __launch_bounds__(32 * BLK_WARPS)
blokus_placement_to_action_kernel(const uint4 *__restrict__ st, const int32_t *__restrict__ placements,
                                  int32_t *__restrict__ actions, long long B, int player, int frame, int flags,
                                  BlkRotTab rot) {
    __shared__ BlkSmem smem[BLK_WARPS];
    const int lane = BLK_WARPS == 1 ? (int)threadIdx.x : (int)(threadIdx.x & 31), wid = BLK_WARPS == 1 ? 0 : (int)(threadIdx.x >> 5);
    const long long g = (long long)blockIdx.x * BLK_WARPS + wid;
    if (g >= B) return;
    BlkSmem &sm = smem[wid];
    blk_load(sm, st, g, lane);
    if ((flags & CRL_FLAG_AUTO_RESET) && (sm.st[85] >> 16 & 1u)) blk_new_state(sm, lane);
    const uint32_t meta = sm.st[85];
    const int c = player >= 0 ? player : (int)(meta >> 8 & 3u);
    const int p = placements[g];
    int aid = p == -1 ? -1 : BLK_ILLEGAL_ACTION;
    if (p >= 0 && p < BLK_NPLACEMENT && !(sm.st[87] >> c & 1u)) {
        int s = p / 400, y = (p - 400 * s) / 20, x = p % 20;
        uint32_t cells = BLK_SHAPE_CELLS[s];
        int w1 = 0, h1 = 0;                                  // bounding box - 1
#pragma unroll
        for (int i = 0; i < 5; i++) {
            w1 = max(w1, (int)(cells >> (6 * i) & 7u));
            h1 = max(h1, (int)(cells >> (6 * i + 3) & 7u));
        }
        const bool on = x + w1 <= 19 && y + h1 <= 19;
        const int q = (4 - (frame ? c : 0)) & 3;
        if (on && q) {
            const int x0 = q == 1 ? 19 - h1 - y : q == 2 ? 19 - w1 - x : y;
            const int y0 = q == 1 ? x : q == 2 ? 19 - h1 - y : 19 - w1 - x;
            s = rot.img[q][s];
            x = x0;
            y = y0;
            cells = BLK_SHAPE_CELLS[s];
        }
        const int pc = (int)(BLK_SHAPE_TAB_G[s].w >> 16 & 31u);
        if (on && (sm.st[80 + c] >> pc & 1u)) {
            blk_allowed_and_anchors<false>(sm, c, (int)(meta & 0xffu), lane);
            bool fit = true;
            int first = 400;                                 // row-major index of the first anchored cell
#pragma unroll
            for (int i = 0; i < 5; i++) {
                const int cx = x + (int)(cells >> (6 * i) & 7u), cy = y + (int)(cells >> (6 * i + 3) & 7u);
                fit = fit && (sm.A[cy] >> (cx + 4) & 1u);
                if (sm.anc[cy] >> cx & 1u) first = min(first, 20 * cy + cx);
            }
            if (fit && first < 400) {
                const int ay = first / 20, ax = first - 20 * ay, size = BLK_PIECE_SIZE[pc], id0 = BLK_PIECE_ID0[pc];
                const uint32_t key = (uint32_t)s | (uint32_t)(ax - x) << 7 | (uint32_t)(ay - y) << 10;
                int j = 0;                                   // ids of the piece in the order o * size + k
                while (j < 8 * size && (BLK_ID_TAB[id0 + j] & 0x1fffu) != key) j++;
                if (j < 8 * size) aid = pc * 16000 + first * 40 + (int)(BLK_ID_TAB[id0 + j] >> 13);   // (always found)
            }
        }
    }
    if (lane == 0) actions[g] = aid;
}
