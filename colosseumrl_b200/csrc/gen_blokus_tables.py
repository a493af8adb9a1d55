"""Generate csrc/blokus_tables.h: the 21 Blokus pieces' oriented shapes as bit-friendly tables.

Geometry (closed form of the reference, SURVEY.md Appendix A-B1): the cells of action (piece, anchor a,
orientation o, shift k) are  a + R_o(c_i) - R_o(c_k)  over the piece's default offsets c_i
(colosseumrl/envs/blokus/board.py:24-44), with R_o from computation.py:53-86.  For every (piece, o) the rotated
cell set is normalised to its bounding box's top-left corner; the 168 (piece, o) pairs collapse onto 91 distinct
normalised shapes.  An action is then  (shape s, origin q = a - cell_k(s))  and is legal iff the anchor is an
anchor and FIT_s[q] is set, where FIT_s = AND_i shift(allowed, cell_i(s)).

Run:  python colosseumrl_b200/csrc/gen_blokus_tables.py   (output is committed; deterministic)
"""
import os

PIECES = [
    ("monomino1", [(0, 0)]),
    ("domino1", [(0, 0), (1, 0)]),
    ("trominoe1", [(0, 0), (1, 0), (1, 1)]),
    ("trominoe2", [(0, 0), (1, 0), (2, 0)]),
    ("tetrominoes1", [(0, 0), (1, 0), (0, 1), (1, 1)]),
    ("tetrominoes2", [(0, 0), (1, -1), (1, 0), (2, 0)]),
    ("tetrominoes3", [(0, 0), (1, 0), (2, 0), (3, 0)]),
    ("tetrominoes4", [(0, 0), (1, 0), (2, 0), (2, -1)]),
    ("tetrominoes5", [(0, 0), (1, 0), (1, -1), (2, -1)]),
    ("pentominoe1", [(0, 0), (0, -1), (1, 0), (2, 0), (3, 0)]),
    ("pentominoe2", [(0, 0), (0, -1), (0, 1), (1, 0), (2, 0)]),
    ("pentominoe3", [(0, 0), (0, -1), (0, -2), (1, -2), (2, -2)]),
    ("pentominoe4", [(0, 0), (1, 0), (1, -1), (2, -1), (3, -1)]),
    ("pentominoe5", [(0, 0), (0, 1), (1, 0), (2, 0), (2, -1)]),
    ("pentominoe6", [(0, 0), (1, 0), (2, 0), (3, 0), (4, 0)]),
    ("pentominoe7", [(0, 0), (1, 0), (2, 0), (1, -1), (2, -1)]),
    ("pentominoe8", [(0, 0), (0, 1), (1, 0), (1, -1), (2, -1)]),
    ("pentominoe9", [(0, 0), (1, 0), (0, 1), (0, 2), (1, 2)]),
    ("pentominoe10", [(0, 0), (1, 0), (1, -1), (1, 1), (2, -1)]),
    ("pentominoe11", [(0, 0), (-1, 0), (1, 0), (0, -1), (0, 1)]),
    ("pentominoe12", [(0, 0), (1, 0), (1, -1), (2, 0), (3, 0)]),
]

# ORIENTATIONS order: north northeast east southeast south southwest west northwest (board.py:47)
ROT = [
    lambda x, y: (y, -x),    # north      (270 deg)
    lambda x, y: (x, -y),    # northeast  (0 deg, flip y)
    lambda x, y: (x, y),     # east       (identity)
    lambda x, y: (y, x),     # southeast  (90 deg, flip x)
    lambda x, y: (-y, x),    # south      (90 deg)
    lambda x, y: (-x, y),    # southwest  (180 deg, flip y)
    lambda x, y: (-x, -y),   # west       (180 deg)
    lambda x, y: (-y, -x),   # northwest  (270 deg, flip x)
]


ORIENTS = []             # (piece, orientation, shape, cells in shift order k)


def build():
    shapes = []          # list of (piece, tuple(sorted cells))
    shape_index = {}
    piece_shape0 = []
    piece_id0 = []
    ids = []             # (shape, dx, dy, o*5+k)
    ORIENTS.clear()
    for p, (_, offs) in enumerate(PIECES):
        piece_shape0.append(len(shapes))
        piece_id0.append(len(ids))
        for o in range(8):
            rot = [ROT[o](x, y) for x, y in offs]
            mx, my = min(c[0] for c in rot), min(c[1] for c in rot)
            norm = [(x - mx, y - my) for x, y in rot]
            key = (p, tuple(sorted(norm)))
            if key not in shape_index:
                shape_index[key] = len(shapes)
                shapes.append(key)
            s = shape_index[key]
            ORIENTS.append((p, o, s, list(norm)))
            for k, (dx, dy) in enumerate(norm):
                ids.append((s, dx, dy, o * 5 + k))
    piece_shape0.append(len(shapes))
    piece_id0.append(len(ids))
    return shapes, piece_shape0, piece_id0, ids


def connected(cells):
    cells = set(cells)
    seen, todo = set(), [next(iter(cells))]
    while todo:
        c = todo.pop()
        if c in seen:
            continue
        seen.add(c)
        for d in ((1, 0), (-1, 0), (0, 1), (0, -1)):
            n = (c[0] + d[0], c[1] + d[1])
            if n in cells and n not in seen:
                todo.append(n)
    return len(seen) == len(cells)


def build_tree(shapes):
    """The 91 shapes are exactly the fixed polyominoes of 1..5 cells, so every shape s of n >= 2 cells is a shape
    of n - 1 cells ("parent") plus one cell c:   FIT_s[q] = FIT_parent[q + off] & A[q + c]   with off = the parent's
    bounding-box corner inside s.  All 91 FIT boards then cost 90 AND steps instead of 414 - 91.
    need[s] = pieces whose own shapes are s or descend from s (a shape is only built if one of them is held)."""
    index = {cells: i for i, (_, cells) in enumerate(shapes)}
    tree = [None] * len(shapes)
    for i, (_, cells) in enumerate(shapes):
        if len(cells) == 1:
            continue
        best = None
        for c in cells:
            rest = [x for x in cells if x != c]
            if not connected(rest):
                continue
            mx, my = min(x for x, _ in rest), min(y for _, y in rest)
            par = index[tuple(sorted((x - mx, y - my) for x, y in rest))]
            cand = (par, mx, my, c[0], c[1])
            if best is None or cand < best:
                best = cand
        assert best is not None and best[0] < i
        tree[i] = best
    need = [1 << p for p, _ in shapes]
    for i in range(len(shapes) - 1, 0, -1):
        need[tree[i][0]] |= need[i]
    return tree, need


def emit(path):
    shapes, piece_shape0, piece_id0, ids = build()
    assert len(shapes) == 91 and len(ids) == 712
    assert sum(len(s[1]) for s in shapes) == 414
    assert [len(c) for _, c in shapes] == sorted(len(c) for _, c in shapes)       # shapes are ordered by size
    tree, need = build_tree(shapes)
    L = []
    L.append("// GENERATED by gen_blokus_tables.py -- do not edit.  See that file for the derivation.")
    L.append("#pragma once")
    L.append("#define BLK_NPIECE 21")
    L.append("#define BLK_NSHAPE %d" % len(shapes))
    L.append("#define BLK_NID %d" % len(ids))
    L.append("// cells of each normalised shape: 5 x 6 bits (dx | dy << 3), short pieces repeat cell 0 (AND/OR idempotent)")
    L.append("__constant__ uint32_t BLK_SHAPE_CELLS[BLK_NSHAPE] = {")
    row = []
    for _, cells in shapes:
        cl = list(cells) + [cells[0]] * (5 - len(cells))
        v = 0
        for i, (dx, dy) in enumerate(cl):
            assert 0 <= dx <= 4 and 0 <= dy <= 4
            v |= (dx | dy << 3) << (6 * i)
        row.append("0x%08xu" % v)
    for i in range(0, len(row), 8):
        L.append("    " + ", ".join(row[i:i + 8]) + ",")
    L.append("};")
    L.append("// piece sizes (== GAME_PIECE_VALUES, ai.py:12-22)")
    L.append("__constant__ uint8_t BLK_PIECE_SIZE[BLK_NPIECE] = {" + ", ".join(str(len(o)) for _, o in PIECES) + "};")
    L.append("// shapes of piece p are [BLK_PIECE_SHAPE0[p], BLK_PIECE_SHAPE0[p+1])")
    L.append("__constant__ uint8_t BLK_PIECE_SHAPE0[BLK_NPIECE + 1] = {" + ", ".join(map(str, piece_shape0)) + "};")
    L.append("// (orientation, shift) ids of piece p are [BLK_PIECE_ID0[p], BLK_PIECE_ID0[p+1]), ordered o*size + k")
    L.append("__constant__ uint16_t BLK_PIECE_ID0[BLK_NPIECE + 1] = {" + ", ".join(map(str, piece_id0)) + "};")
    L.append("// per id: shape (7 bits) | dx << 7 | dy << 10 | (o*5 + k) << 13 ; (dx, dy) = the shape cell that sits on the anchor")
    L.append("__constant__ uint32_t BLK_ID_TAB[BLK_NID] = {")
    row = ["0x%05xu" % (s | dx << 7 | dy << 10 | ok << 13) for s, dx, dy, ok in ids]
    for i in range(0, len(row), 8):
        L.append("    " + ", ".join(row[i:i + 8]) + ",")
    L.append("};")
    n_le4 = sum(1 for _, c in shapes if len(c) <= 4)
    FROWS = 25
    L.append("// ---- FIT-board storage: %d words per board (index y + 4: rows -4..-1 and 20 are zero, rows 21..23 are the next" % FROWS)
    L.append("// board's zero rows -4..-2; the odd stride spreads the boards over the shared-memory banks when lanes = shapes).")
    L.append("// Boards of the shapes of <= 4 cells live in slots")
    L.append("// 0..%d; the pentomino shapes are processed in groups of whole pieces that share slots %d.. :" % (n_le4 - 1, n_le4))
    L.append("#define BLK_FROWS %d" % FROWS)
    L.append("#define BLK_NSHAPE_LE4 %d" % n_le4)
    # greedy grouping of the pentomino pieces, at most GROUP_CAP shapes per group
    GROUP_CAP = int(os.environ.get("BLK_GROUP_CAP", "24"))
    groups, cur = [], None
    for pc in range(len(PIECES)):
        if len(PIECES[pc][1]) < 5:
            continue
        nsh = piece_shape0[pc + 1] - piece_shape0[pc]
        if cur is None or cur[3] + nsh > GROUP_CAP:
            cur = [pc, pc + 1, piece_shape0[pc], nsh]
            groups.append(cur)
        else:
            cur[1] = pc + 1
            cur[3] += nsh
    L.append("#define BLK_NGROUP %d" % len(groups))
    L.append("#define BLK_GROUP_MAX %d" % max(g[3] for g in groups))
    L.append("// group g: pieces [BLK_GROUP_P0[g], BLK_GROUP_P0[g+1]), shapes [BLK_GROUP_S0[g], BLK_GROUP_S0[g+1])")
    L.append("__constant__ uint8_t BLK_GROUP_P0[BLK_NGROUP + 1] = {" + ", ".join(str(g[0]) for g in groups) + ", %d};" % len(PIECES))
    L.append("__constant__ uint8_t BLK_GROUP_S0[BLK_NGROUP + 1] = {" + ", ".join(str(g[2]) for g in groups) + ", %d};" % len(shapes))
    group_of = {}
    for gi, g in enumerate(groups):
        for pc in range(g[0], g[1]):
            group_of[pc] = gi
    L.append("// pentomino piece -> its group (pieces of <= 4 cells: 255)")
    L.append("__constant__ uint8_t BLK_PIECE_GROUP[BLK_NPIECE] = {" + ", ".join(str(group_of.get(pc, 255)) for pc in range(len(PIECES))) + "};")
    sizes = [len(c) for _, c in shapes]
    lv = [sizes.index(k) for k in range(1, 6)] + [len(shapes)]
    L.append("// shapes of k cells are [BLK_LEVEL_S0[k-1], BLK_LEVEL_S0[k])")
    L.append("__constant__ uint8_t BLK_LEVEL_S0[6] = {" + ", ".join(map(str, lv)) + "};")

    def slot_flag(i):
        pc = shapes[i][0]
        if len(shapes[i][1]) == 5:
            g = groups[group_of[pc]]
            return n_le4 + i - g[2], i - g[2]
        return i, i

    L.append("// per (piece, orientation), read by the lanes that own the orientation during emission, 12 x uint16, every field")
    L.append("// directly usable (no unpacking):  [0..4] byte offset of FIT row (4 - dy_k) of the orientation's slot for shift")
    L.append("// k = 0..4 (the shape cell (dx_k, dy_k) sits on the anchor; id = o * 5 + k), [5..9] OFF - dx_k (OFF = 8 for pieces of")
    L.append("// <= 4 cells, 12 for pentominoes: the column-0 bit of their FIT boards), [10] non-empty flag")
    L.append("// index (s for <= 4 cells: bit of `ne`; s - group start for pentominoes: bit of the group's `ne5`), [11] unused")
    L.append("// (32-bit entries, three 128-bit loads per lane and piece: 16-bit entries cost eleven LDG.U16)")
    L.append("__device__ const uint4 BLK_ORIENT_TAB_G[BLK_NPIECE * 8][3] = {")
    for (pc, o, s_, cells) in ORIENTS:
        slot, flag = slot_flag(s_)
        cl = list(cells) + [cells[0]] * (5 - len(cells))
        offs = [(slot * FROWS + 4 - dy) * 4 for dx, dy in cl]
        cs = [(12 if len(cells) == 5 else 8) - dx for dx, dy in cl]    # BLK_OFF_PENT / BLK_OFF_LE4 of blokus.cuh
        v = offs + cs + [flag, 0]
        L.append("    {" + ", ".join("{%d, %d, %d, %d}" % tuple(v[4 * j:4 * j + 4]) for j in range(3)) + "},")
    L.append("};")
    L.append("// Polyomino tree (see build_tree in the generator), one entry per shape, read by the lane that owns the shape")
    L.append("// (lanes = shapes of one level / pentomino group):   FIT_s[q] = FIT_parent[q + (px, py)] & A[q + (cx, cy)]")
    L.append("//  .x = byte offset of parent row (4 + py) | px << 16 | cx << 20 | (4 * cy) << 24")
    L.append("//  .y = pieces that need s (own piece + descendants; 5-cell shapes are leaves) | parent's flag index << 24")
    L.append("//  .z = the shape's cells, 5 x 6 bits (dx | dy << 3), short shapes repeat cell 0")
    L.append("//  .w = byte offset of the shape's own row 4 (y = 0) | piece << 16 | cells << 24")
    L.append("__device__ const uint4 BLK_SHAPE_TAB_G[BLK_NSHAPE + 32] = {    // (padded: a pass reads entry s0 + lane with 32 lanes)")
    for i in range(len(shapes)):
        pc, cells = shapes[i]
        slot, flag = slot_flag(i)
        if i == 0:
            par, px, py, cx, cy = 0, 0, 0, 0, 0
        else:
            par, px, py, cx, cy = tree[i]
        assert len(shapes[par][1]) <= 4 and par < n_le4
        cl = list(cells) + [cells[0]] * (5 - len(cells))
        cw = 0
        for k, (dx, dy) in enumerate(cl):
            cw |= (dx | dy << 3) << (6 * k)
        x = ((par * FROWS + 4 + py) * 4) | px << 16 | cx << 20 | (4 * cy) << 24
        y = need[i] | par << 24
        w = ((slot * FROWS + 4) * 4) | pc << 16 | len(cells) << 24
        L.append("    {0x%08xu, 0x%08xu, 0x%08xu, 0x%08xu}," % (x, y, cw, w))
    for _ in range(32):
        L.append("    {0u, 0u, 0u, 0u},")
    L.append("};")
    emit_host_tables(L, shapes, piece_id0, ids)
    open(path, "w").write("\n".join(L) + "\n")


# Rotation q of the board frame into player q's observation frame (np.rot90(k=-q)) on cell offsets:
# (x, y) -> (19 - y, x), (19 - x, 19 - y), (y, 19 - x) for q = 1, 2, 3, i.e. these maps up to a translation.
ROT_FRAME = [lambda x, y: (x, y), lambda x, y: (-y, x), lambda x, y: (-x, -y), lambda x, y: (y, -x)]


def emit_host_tables(L, shapes, piece_id0, ids):
    """Host-only copies for crl_blokus_shape_table and the placement launchers: plain `static const` arrays, so the
    device code (and its constant banks) never sees them."""
    index = {key: i for i, key in enumerate(shapes)}
    L.append("// ---- host only (crl_blokus_shape_table, include/colosseum_b200_placement.h): no device storage")
    L.append("// shape -> piece")
    L.append("static const int8_t BLK_HOST_SHAPE_PIECE[BLK_NSHAPE] = {" + ", ".join(str(p) for p, _ in shapes) + "};")
    L.append("// shape -> its cells (dx, dy), -1 past the shape's size")
    L.append("static const int8_t BLK_HOST_SHAPE_CELLS[BLK_NSHAPE][5][2] = {")
    for _, cells in shapes:
        cl = [list(c) for c in cells] + [[-1, -1]] * (5 - len(cells))
        L.append("    {" + ", ".join("{%d, %d}" % tuple(c) for c in cl) + "},")
    L.append("};")
    L.append("// shape -> its image in player q's rotated frame, q = 0..3")
    L.append("static const int8_t BLK_HOST_SHAPE_ROT[BLK_NSHAPE][4] = {")
    for p, cells in shapes:
        img = []
        for q in range(4):
            rc = [ROT_FRAME[q](x, y) for x, y in cells]
            mx, my = min(x for x, _ in rc), min(y for _, y in rc)
            img.append(index[(p, tuple(sorted((x - mx, y - my) for x, y in rc)))])
        L.append("    {" + ", ".join(map(str, img)) + "},")
    L.append("};")
    L.append("// (piece, o * 5 + k) -> (shape, dx, dy) of the id's orientation and of the shape cell on the anchor; -1 if k >= size")
    L.append("static const int8_t BLK_HOST_ACTION_SHAPE[BLK_NPIECE][40][3] = {")
    for p in range(len(piece_id0) - 1):
        row = [[-1, -1, -1] for _ in range(40)]
        for s, dx, dy, ok in ids[piece_id0[p]:piece_id0[p + 1]]:
            row[ok] = [s, dx, dy]
        L.append("    {" + ", ".join("{%d, %d, %d}" % tuple(v) for v in row) + "},")
    L.append("};")


if __name__ == "__main__":
    out = os.path.join(os.path.dirname(os.path.abspath(__file__)), "blokus_tables.h")
    emit(out)
    print("wrote", out)
