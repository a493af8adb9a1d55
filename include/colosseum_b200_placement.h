/* colosseum_b200_placement.h -- a fixed Blokus action space of placements, with legality masks, for
 * libcolosseum_b200.so (included by colosseum_b200.h; the same conventions: device pointers, the caller's stream,
 * 0 = OK, crl_last_error() on failure).
 *
 * The reference's action ids, ((piece * 400 + anchor) * 8 + orientation) * 5 + shift, form a ragged list per position
 * in which one physical move appears once per anchor it covers and per symmetric orientation of its piece.  A policy
 * head wants a fixed set of outputs and one output per move; that is what a placement is.
 *
 *   Placement index  p = s * 400 + y * 20 + x,  0 <= p < CRL_BLOKUS_NPLACEMENT (36 400);  -1 is a pass.
 *     s:      the oriented shape, 0 <= s < 91, in the engine's shape order (blokus_tables.h: sorted by size, then by
 *             piece, then by first appearance in ORIENTATIONS order).  The 91 shapes are the fixed polyominoes of
 *             1..5 cells; each belongs to exactly one piece.  crl_blokus_shape_table lists them.
 *     (x, y): the top-left corner of the shape's bounding box.  The placement covers the cells (x, y) + cell_i(s).
 *   Legal placement, for player c: c holds the piece of s; every cell is on the board and allowed for c (empty, not
 *     edge-adjacent to c's own cells); at least one cell is an anchor of c (round 0: c's corner).  This is exactly the
 *     set {placement(id) : id in crl_blokus_legal's full list}.  A player whose "no move any more" cache bit is set
 *     (state word 87) has no legal placement.
 *   Frames (frame = 0 or 1):
 *     0: the board frame.
 *     1: player r's rotated frame, the frame of crl_blokus_observe(player = r) (np.rot90(k = -r)): the board cell
 *        (x, y) is (19 - y, x), (19 - x, 19 - y), (y, 19 - x) for r = 1, 2, 3.  A placement in frame 1 is the image of
 *        the board placement's cells, so  placement_in_frame_1(real_action_to_player_perspective(id, r)) ==
 *        rotate_r(placement(id))  for every id.
 *     player < 0 means each game's mover, and in frame 1 the mover's frame (as crl_blokus_legal / crl_blokus_observe).
 *   Canonical action of a legal placement: the first id of the reference's list whose placement it is -- the anchor is
 *     the row-major first cell of the placement that is an anchor, the orientation the lowest orientation of the piece
 *     whose shape is s, and the shift follows from those two.
 *   Illegal input: an illegal or out-of-range placement converts to CRL_BLOKUS_ILLEGAL_ACTION (21 * 16 000 =
 *     336 000).  No valid list holds that id, so crl_blokus_step and crl_blokus_advance flag it as illegal and apply a
 *     pass, as for any id outside the list.  -1 stays -1.
 */
#ifndef COLOSSEUM_B200_PLACEMENT_H
#define COLOSSEUM_B200_PLACEMENT_H
#include <stdint.h>

#define CRL_BLOKUS_NSHAPE 91
#define CRL_BLOKUS_NPLACEMENT 36400
#define CRL_BLOKUS_ILLEGAL_ACTION 336000

#ifdef __cplusplus
extern "C" {
#endif

/* Legal-placement masks of `player` (< 0: each game's mover) in `frame`.  mask: uint32[B][91][20], 7 280 bytes per
 * game (16-byte aligned): bit x of word [g][s][y] is set iff placement (s, x, y) is legal; bits 20..31 are zero.
 * counts_or_null: int32[B] number of legal placements (4-byte aligned).  flags: CRL_FLAG_AUTO_RESET as for
 * crl_blokus_legal (a terminal game is read as new_state()).  State 16-byte aligned.
 * CRL_ERR_ARG: null state or mask, B < 0, player > 3, frame not 0 or 1, a misaligned buffer.  B == 0: no-op. */
int crl_blokus_placement_mask(const void *state, int player, int frame, uint32_t *mask, int32_t *counts_or_null,
                              int64_t B, int flags, crl_stream_t stream);

/* actions[g] = the canonical action id of placements[g] (a placement of `player` in `frame`), -1 for -1, and
 * CRL_BLOKUS_ILLEGAL_ACTION for an illegal or out-of-range placement.  placements, actions: int32[B] (4-byte aligned);
 * flags and refusals as crl_blokus_placement_mask (null state, placements or actions). */
int crl_blokus_placement_to_action(const void *state, int player, int frame, const int32_t *placements,
                                   int32_t *actions, int64_t B, int flags, crl_stream_t stream);

/* Host only: the shape tables.  Returns CRL_BLOKUS_NSHAPE; every output may be NULL.
 *   shape_piece:    int32[91]           the piece (PIECE_TYPES order) of shape s
 *   shape_cells:    int32[91][5][2]     its cells (dx, dy); -1 past the shape's size
 *   shape_rotation: int32[91][4]        its image in player q's rotated frame (q = 0: s itself)
 *   action_shape:   int32[21][40][3]    per piece and o * 5 + k: (shape, dx, dy) of orientation o and of its cell k,
 *                                       the cell that sits on the anchor; -1 if k >= the piece's size
 * The placement of id ((piece * 400 + ay * 20 + ax) * 8 + o) * 5 + k is then  s * 400 + (ay - dy) * 20 + (ax - dx). */
int crl_blokus_shape_table(int32_t *shape_piece_or_null, int32_t *shape_cells_or_null,
                           int32_t *shape_rotation_or_null, int32_t *action_shape_or_null);

#ifdef __cplusplus
}
#endif
#endif
