"""Blokus placement cases (crl_blokus_placement_mask, crl_blokus_placement_to_action, crl_blokus_shape_table), written
once against the C ABI and run on both backends (tests/backends.py), bit-exact.  The oracle is the C oracle's ordered
list (orc.blokus_valid_moves) mapped through the generator's geometry (gen_blokus_tables.ORIENTS): the expected mask is
the set of the list's placements, the expected canonical id the first list entry with that placement."""
import os
import sys

import numpy as np

from oracle import oracle as orc
from colosseumrl_b200.blokus import real_action_to_player_perspective
import cases_api_contract as api
import cases_blokus as cb

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, os.path.join(ROOT, "colosseumrl_b200", "csrc"))
import gen_blokus_tables as gen  # noqa: E402

NSHAPE, NPLACE, ILLEGAL = 91, 36400, 336000
AUTO_RESET = 1

# ----------------------------------------------------------------------------------------------- geometry (generator)
_SHAPES, _, _, _ = gen.build()
ORIENT_SHAPE = np.zeros((21, 8), np.int64)
ORIENT_CELLS = np.zeros((21, 8, 5, 2), np.int64)
for _p_, _o_, _s_, _cells_ in gen.ORIENTS:
    ORIENT_SHAPE[_p_, _o_] = _s_
    for _k_, _c_ in enumerate(_cells_):
        ORIENT_CELLS[_p_, _o_, _k_] = _c_


def id_placement(ids):
    """action ids (board frame, all valid list entries) -> placements of their own frame"""
    ids = np.asarray(ids, np.int64)
    k, o, cell, piece = ids % 5, (ids // 5) % 8, (ids // 40) % 400, ids // 16000
    s = ORIENT_SHAPE[piece, o]
    dx, dy = ORIENT_CELLS[piece, o, k, 0], ORIENT_CELLS[piece, o, k, 1]
    return s * 400 + (cell // 20 - dy) * 20 + (cell % 20 - dx)


def list_placements(ids, player, frame):
    """the list's placements in `frame` (frame 1: the player's rotated frame, through the ids' rotation)"""
    ids = np.asarray(ids, np.int64)
    if frame:
        ids = real_action_to_player_perspective(ids, player)
    return id_placement(ids)


def expected(state, c, frame):
    """(sorted placements, {placement: canonical id}) of player c by the oracle"""
    lst = orc.blokus_valid_moves(state, c, cap=65536)
    pl = list_placements(lst, c, frame)
    canon = {}
    for p, a in zip(pl.tolist(), lst.tolist()):
        canon.setdefault(p, a)
    return np.array(sorted(canon), np.int64), canon


def unpack_words(words):
    """uint32 [B, 91, 20] -> bool [B, 36 400]; also asserts bits 20..31 are zero"""
    w = np.asarray(words).view(np.uint32)
    assert not (w >> 20).any()
    return ((w[..., None] >> np.arange(20, dtype=np.uint32)) & 1).astype(bool).reshape(len(w), NPLACE)


# ----------------------------------------------------------------------------------------------- device calls
def placement_mask(be, st, player=-1, frame=0, flags=0, counts=True):
    B = st.shape[0]
    words, cnt = be.zeros((B, NSHAPE, 20), np.int32), be.zeros((B,), np.int32) if counts else None
    be.check(be.lib.crl_blokus_placement_mask(be.ptr(st), player, frame, be.ptr(words), be.ptr(cnt), B, flags, be.stream))
    return (be.download(cnt) if counts else None), be.download(words)


def placement_to_action(be, st, placements, player=-1, frame=0, flags=0):
    B = st.shape[0]
    p, a = be.upload(np.ascontiguousarray(placements, np.int32)), be.zeros((B,), np.int32)
    be.check(be.lib.crl_blokus_placement_to_action(be.ptr(st), player, frame, be.ptr(p), be.ptr(a), B, flags, be.stream))
    return be.download(a)


def repeat_rows(be, st, idx):
    return be.upload(be.download(st)[np.asarray(idx, np.int64)])


# ----------------------------------------------------------------------------------------------- positions
def golden_positions(stride=1):
    """board, inventory, scores, round, mover of every position of blokus_games.npz (the state before each recorded
    step), blokus_boards.npz (arbitrary positions) and the end-game positions of blokus_wide.npz"""
    g = np.load(os.path.join(cb.GOLDEN, "blokus_games.npz"))
    board, inv, scores, rounds = cb._golden_prev(g)
    b = np.load(os.path.join(cb.GOLDEN, "blokus_boards.npz"))
    w = np.load(os.path.join(cb.GOLDEN, "blokus_wide.npz"))
    out = [np.concatenate(x)[::stride] for x in (
        (board, b["i_board"], w["e_i_board"]), (inv, b["i_inventory"], w["e_i_inventory"]),
        (scores, b["i_scores"], w["e_i_scores"]), (rounds, b["i_round"], w["e_i_round"]), (g["mover"], b["mover"], w["e_mover"]))]
    return tuple(out)


def _state(pos, i):
    board, inv, scores, rounds, _ = pos
    return (board[i].astype(np.int64), int(rounds[i]), inv[i], scores[i])


def check_masks(be, st, pos, players=(-1, 0, 1, 2, 3), frames=(0, 1), flags=0):
    """mask and counts of every position vs the oracle; returns {(i, c, frame): (placements, canon)}"""
    movers = pos[4]
    ref = {}
    for player in players:
        for frame in frames:
            counts, words = placement_mask(be, st, player, frame, flags)
            m = unpack_words(words)
            for i in range(len(movers)):
                c = int(movers[i]) if player < 0 else player
                key = (i, c, frame)
                if key not in ref:
                    ref[key] = expected(_state(pos, i), c, frame)
                pl = ref[key][0]
                got = np.flatnonzero(m[i])
                assert counts[i] == len(pl) and len(got) == len(pl) and (got == pl).all(), (i, player, frame, counts[i], len(pl))
    return ref


def case_golden_masks(be, stride=1):
    """every golden position, players -1 and 0..3, both frames"""
    pos = golden_positions(stride)
    st = cb.blk_pack(be, *pos)
    check_masks(be, st, pos)
    # a NULL counts buffer writes the same mask
    _, w1 = placement_mask(be, st, -1, 1)
    _, w2 = placement_mask(be, st, -1, 1, counts=False)
    assert (w1 == w2).all()


def case_conversion(be, stride=1, per_position=None, seed=3):
    """placement -> canonical id, for the legal placements of every golden position (all of them, or `per_position`
    drawn ones), players -1 and 0..3 and both frames: the first list entry with that placement; a frame-1 placement
    gives the board-frame id of its rotation.  Illegal and out-of-range placements give ILLEGAL, -1 gives -1."""
    pos = golden_positions(stride)
    st = cb.blk_pack(be, *pos)
    movers = pos[4]
    rng = np.random.RandomState(seed)
    n_legal = n_illegal = 0
    for player in (-1, 0, 1, 2, 3):
        for frame in (0, 1):
            rows, pls, exp = [], [], []
            for i in range(len(movers)):
                c = int(movers[i]) if player < 0 else player
                pl, canon = expected(_state(pos, i), c, frame)
                take = pl if per_position is None or len(pl) <= per_position else rng.choice(pl, per_position, replace=False)
                rows += [i] * len(take)
                pls += [int(p) for p in take]
                exp += [canon[int(p)] for p in take]
                n_legal += len(take)
                # illegal: not in the legal set (random and next to legal ones), out of range, pass
                legal = set(pl.tolist())
                cand = [int(x) for x in rng.randint(0, NPLACE, size=3)] + [int(p) + d for p in take[:2] for d in (1, 20, 400)]
                cand += [-1, -2, NPLACE, NPLACE + 5, 2 ** 31 - 1, -2 ** 31]
                for p in cand:
                    if p in legal:
                        continue
                    rows.append(i)
                    pls.append(p)
                    exp.append(-1 if p == -1 else ILLEGAL)
                    n_illegal += 1
            got = placement_to_action(be, repeat_rows(be, st, rows), pls, player, frame)
            bad = np.flatnonzero(got != np.array(exp))
            assert len(bad) == 0, (player, frame, [(rows[j], pls[j], got[j], exp[j]) for j in bad[:5]])
    assert n_legal > 100 and n_illegal > 100


def case_step_equivalence(be, stride=1, ids_per_position=None, seed=4):
    """crl_blokus_step with a placement's canonical id == with every other id of that placement (state bytes and
    record); an illegal placement converts to an id that the step flags and plays as a pass"""
    pos = golden_positions(stride)
    st = cb.blk_pack(be, *pos)
    movers = pos[4]
    rng = np.random.RandomState(seed)
    rows, ids, canon_ids = [], [], []
    for i in range(len(movers)):
        lst = orc.blokus_valid_moves(_state(pos, i), int(movers[i]), cap=65536)
        pl = id_placement(lst)
        first = {}
        for p, a in zip(pl.tolist(), lst.tolist()):
            first.setdefault(p, a)
        sel = np.arange(len(lst)) if ids_per_position is None or len(lst) <= ids_per_position else \
            rng.choice(len(lst), ids_per_position, replace=False)
        for j in sel:
            rows.append(i)
            ids.append(int(lst[j]))
            canon_ids.append(first[int(pl[j])])
    sub = repeat_rows(be, st, rows)
    pls = id_placement(ids)
    conv = placement_to_action(be, sub, pls)
    assert (conv == np.array(canon_ids)).all()
    out1, r1 = cb.blk_step(be, sub, ids)
    out2, r2 = cb.blk_step(be, sub, conv)
    assert (be.download(out1) == be.download(out2)).all()
    for k in r1:
        assert (r1[k] == r2[k]).all(), k
    assert not r1["error"].any() and r1["placed"].all()
    assert (np.array(ids) != np.array(canon_ids)).sum() > len(ids) // 4          # most placements have several ids
    # illegal placements: flagged, applied as a pass
    n = len(movers)
    bad = np.full(n, NPLACE + 1, np.int64)
    conv = placement_to_action(be, st, bad)
    assert (conv == ILLEGAL).all()
    out1, r1 = cb.blk_step(be, st, conv)
    out2, r2 = cb.blk_step(be, st, np.full(n, -1))
    assert r1["error"].all() and not r2["error"].any() and (be.download(out1) == be.download(out2)).all()


def edge_positions():
    """(name, board, inventory, scores, round, mover, terminal, stuck word) of hand-built positions"""
    g = np.load(os.path.join(cb.GOLDEN, "blokus_boards.npz"))
    z = lambda: np.zeros((20, 20), np.int8)
    full = np.ones((4, 21), np.uint8)
    out = [("new", z(), full, 0)]
    b = z()
    b[0, 0] = 2                                               # colour 2 on player 0's corner: blocked in round 0
    b[19, 19] = 1                                             # player 0's colour on player 3's corner
    out.append(("blocked corner", b, full, 0))
    inv = g["i_inventory"][40].copy()
    inv[0] = 0
    inv[2, :9] = 0                                            # player 2: pentominoes only
    out.append(("empty inventory", g["i_board"][40], inv, int(g["i_round"][40])))
    # only the I-pentomino, on a board that leaves it room along the top edge only
    b = np.full((20, 20), 3, np.int8)
    b[0] = 0
    b[1, 5] = 1
    inv = np.zeros((4, 21), np.uint8)
    inv[0, 14] = 1
    out.append(("edge only", b, inv, 3))
    return out


def case_edges(be):
    """round 0 with a free and a blocked corner, an empty inventory, an edge-only piece, the stuck cache bit, terminal
    games with and without CRL_FLAG_AUTO_RESET"""
    edges = edge_positions()
    n = len(edges)
    board = np.stack([e[1] for e in edges])
    inv = np.stack([e[2] for e in edges])
    rounds = np.array([e[3] for e in edges])
    scores, movers = np.zeros((n, 4), np.int64), np.zeros(n, np.int64)
    pos = (board, inv, scores, rounds, movers)
    st = cb.blk_pack(be, *pos)
    ref = check_masks(be, st, pos)
    assert len(ref[(0, 0, 0)][0]) == 58 and len(ref[(0, 3, 1)][0]) == 58             # 58 first placements per seat
    assert len(ref[(1, 0, 0)][0]) == 0 and len(ref[(1, 3, 0)][0]) == 0 and len(ref[(1, 1, 0)][0]) == 58
    assert len(ref[(2, 0, 1)][0]) == 0
    edge = ref[(3, 0, 0)][0]
    assert len(edge) > 0 and (edge // 400 >= 56).all() and (edge % 400 < 20).all()   # I-pentomino shapes, row 0
    # the stuck cache bit (state word 87) of a player who has moves: no placement, and its placements are illegal
    raw = be.download(st)
    for c in range(4):
        s2 = raw.copy()
        s2[:, 21, 3] = 1 << c
        s2 = be.upload(s2)
        counts, words = placement_mask(be, s2, c, 1)
        assert (counts == 0).all() and (words == 0).all()
        pl0 = ref[(0, c, 0)][0]
        assert (placement_to_action(be, s2[:1], pl0[:1], c) == ILLEGAL).all()
        other = (c + 1) & 3
        counts, _ = placement_mask(be, s2, other, 0)
        assert counts[0] == 58
    # terminal games: read as stored without the flag, as new_state() with it
    term = cb.blk_pack(be, *pos, terminal=np.ones(n, np.int32))
    check_masks(be, term, pos, players=(-1, 2), frames=(0, 1))
    fresh = (np.zeros_like(board), np.ones_like(inv), scores, np.zeros(n, np.int64), movers)
    check_masks(be, term, fresh, players=(-1, 2), frames=(0, 1), flags=AUTO_RESET)
    p0 = ref[(0, 0, 0)][0]
    got = placement_to_action(be, term, np.full(n, p0[0]), -1, 0, AUTO_RESET)
    assert (got == ref[(0, 0, 0)][1][int(p0[0])]).all()
    got = placement_to_action(be, term, np.full(n, p0[0]), -1, 0, 0)
    assert got[0] == ref[(0, 0, 0)][1][int(p0[0])] and (got[1:] == ILLEGAL).all()


def case_shape_table(lib):
    """crl_blokus_shape_table == the generator's geometry"""
    piece, cells = np.zeros(91, np.int32), np.zeros((91, 5, 2), np.int32)
    rot, act = np.zeros((91, 4), np.int32), np.zeros((21, 40, 3), np.int32)
    assert lib.crl_blokus_shape_table(piece.ctypes.data, cells.ctypes.data, rot.ctypes.data, act.ctypes.data) == 91
    assert lib.crl_blokus_shape_table(None, None, None, None) == 91
    for s, (p, cl) in enumerate(_SHAPES):
        assert piece[s] == p and [tuple(c) for c in cells[s, :len(cl)]] == list(cl) and (cells[s, len(cl):] == -1).all()
    for p, o, s, cl in gen.ORIENTS:
        for k in range(5):
            exp = [s, cl[k][0], cl[k][1]] if k < len(cl) else [-1, -1, -1]
            assert list(act[p, 5 * o + k]) == exp
    # rotation images: placement of a rotated id == the rotated shape at the rotated corner
    ids = np.concatenate([orc.blokus_valid_moves(orc.blokus_new_state(), q) for q in range(4)])
    for r in range(4):
        a = id_placement(ids)
        b = id_placement(real_action_to_player_perspective(ids.astype(np.int64), r))
        assert (rot[a // 400, r] == b // 400).all()
    assert (rot[:, 0] == np.arange(91)).all()


def case_python_helpers():
    """action_to_placement over every id (both frames) and placement_mask, on numpy arrays, tensors and ints"""
    import torch
    from colosseumrl_b200 import blokus as bl
    ids = np.arange(ILLEGAL, dtype=np.int64)
    # the ids a list can hold: shift below the piece's size and the corner on the board
    size = np.array([len(c) for _, c in gen.PIECES])[ids // 16000]
    k, cell = ids % 5, (ids // 40) % 400
    ok = k < size
    exp = np.full(ILLEGAL, -1, np.int64)
    pl = id_placement(np.where(ok, ids, 0))
    o, piece = (ids // 5) % 8, ids // 16000
    dx, dy = ORIENT_CELLS[piece, o, np.minimum(k, 4), 0], ORIENT_CELLS[piece, o, np.minimum(k, 4), 1]
    on = ok & (cell % 20 >= dx) & (cell // 20 >= dy)
    exp[on] = pl[on]
    assert (bl.action_to_placement(ids) == exp).all()
    assert (bl.action_to_placement(torch.from_numpy(ids)).numpy() == exp).all()
    assert bl.action_to_placement(-1) == -1 and bl.action_to_placement(-1, 2) == -1 and bl.action_to_placement(ILLEGAL) == -1
    lst = orc.blokus_valid_moves(orc.blokus_new_state(), 2).astype(np.int64)
    for r in range(4):
        assert (bl.action_to_placement(lst, r) == id_placement(real_action_to_player_perspective(lst, r))).all()
        assert bl.action_to_placement(int(lst[5]), r) == int(id_placement(real_action_to_player_perspective(lst[5:6], r))[0])
    rng = np.random.RandomState(0)
    words = (rng.randint(0, 1 << 20, size=(3, 91, 20))).astype(np.int32)
    assert (bl.placement_mask(torch.from_numpy(words)).numpy() == unpack_words(words)).all()


# ----------------------------------------------------------------------------------------------- API contract
PROTO_HEADER = os.path.join(ROOT, "include", "colosseum_b200_placement.h")
MASK, TO_ACTION, TABLE = "crl_blokus_placement_mask", "crl_blokus_placement_to_action", "crl_blokus_shape_table"
SCALARS = dict(api.SCALARS, frame=0)


def prototypes():
    saved = api.HEADER
    try:
        api.HEADER = PROTO_HEADER
        return api.prototypes()
    finally:
        api.HEADER = saved


def contract_rows():
    """(entry point, overrides of the valid call, return code, message).  Order: null pointers, B < 0, player > 3 ->
    frame -> B == 0 -> alignment"""
    rows = []
    for fn, out in ((MASK, "mask"), (TO_ACTION, "actions")):
        BAD, FRAME = fn + ": bad argument", fn + ": frame must be 0 or 1"
        rows += [
            (fn, dict(ALL_NULL=1), api.ARG, BAD), (fn, dict(state=None), api.ARG, BAD), (fn, {out: None}, api.ARG, BAD),
            (fn, dict(B=-1), api.ARG, BAD), (fn, dict(player=4), api.ARG, BAD), (fn, dict(player=4, B=0), api.ARG, BAD),
            (fn, dict(state=None, frame=2), api.ARG, BAD),
            (fn, dict(frame=2), api.ARG, FRAME), (fn, dict(frame=-1), api.ARG, FRAME), (fn, dict(frame=1 << 20, B=0), api.ARG, FRAME),
            (fn, dict(B=0), api.OK, None), (fn, dict(B=0, frame=1, player=3, state="D1"), api.OK, None),
            (fn, dict(B=0, player=-7), api.OK, None),
        ]
    rows += [
        (MASK, dict(state="D8"), api.ARG, MASK + ": state and mask must be 16-byte aligned"),
        (MASK, dict(mask="D4", counts_or_null="D1"), api.ARG, MASK + ": state and mask must be 16-byte aligned"),
        (MASK, dict(counts_or_null="D1"), api.ARG, MASK + ": counts must be 4-byte aligned"),
        (TO_ACTION, dict(placements=None), api.ARG, TO_ACTION + ": bad argument"),
        (TO_ACTION, dict(state="D4", placements="D1"), api.ARG, TO_ACTION + ": state must be 16-byte aligned"),
        (TO_ACTION, dict(placements="D1"), api.ARG, TO_ACTION + ": placements and actions must be 4-byte aligned"),
        (TO_ACTION, dict(actions="D4", placements="D8", B=0), api.OK, None),
        (TABLE, dict(), 91, None),
    ]
    return rows


def case_contract(lib, emulator):
    """every row: return code, message, and (emulator) nothing written to device memory; emulator = False: the rows that
    pass no device buffer, on the product library"""
    protos = prototypes()
    assert set(protos) == {MASK, TO_ACTION, TABLE}
    buffers = api.Buffers(emulator)
    ran = 0
    for fn, overrides, expect, msg in contract_rows():
        args = []
        for name, is_ptr in protos[fn]:
            if name in overrides:
                v = overrides[name]
            elif name == "stream":
                v = None
            elif not is_ptr:
                v = SCALARS[name]
            else:
                v = None if ("ALL_NULL" in overrides or name.endswith("_or_null")) else "D"
            args.append((name, v))
        if not emulator and any(isinstance(v, str) and v in api.DEVICE for _, v in args):
            continue
        assert lib.crl_ttt_cells(0) == -1             # leave a different message behind first
        rc = getattr(lib, fn)(*[buffers.value(fn, name, v) if isinstance(v, str) else v for name, v in args])
        err = lib.crl_last_error().decode()
        assert rc == expect, (fn, overrides, rc, expect, err)
        if msg is not None:
            assert err == msg, (fn, overrides, err, msg)
        if emulator:
            assert buffers.untouched(), (fn, overrides)
        ran += 1
    return ran


# ----------------------------------------------------------------------------------------------- GPU only
def case_full_size(be, B=16384, phases=(0, 6, 20, 44, 76), seed=7, cap=4096, sample=48):
    """B games advanced by crl_blokus_rollout to several phases; for every game, player -1 and 0..3 and both frames,
    the mask equals crl_blokus_legal's own list mapped to placements (the legal kernel is pinned to the oracle), and a
    sample of games equals the oracle directly"""
    import torch
    from colosseumrl_b200.blokus import placement_mask as unpack
    dev = be.dev
    ids_all = np.arange(ILLEGAL, dtype=np.int64)
    lut = torch.from_numpy(np.stack([id_placement(real_action_to_player_perspective(ids_all, r)) for r in range(4)])).to(dev)
    st = be.zeros((B, 22, 4), np.int32)
    be.check(be.lib.crl_blokus_reset(be.ptr(st), None, B, be.stream))
    done, most = 0, 0
    for K in phases:
        if K > done:
            be.check(be.lib.crl_blokus_rollout(be.ptr(st), None, None, seed, 0, done, K - done, B, be.stream))
            done = K
        mover = (st[:, 21, 1] >> 8) & 3
        for player, flags in ((-1, 0), (0, 0), (1, 0), (2, 0), (3, 0), (-1, AUTO_RESET)):
            counts, ids = be.zeros((B,), np.int32), be.zeros((B, cap), np.int32)
            be.check(be.lib.crl_blokus_legal(be.ptr(st), player, be.ptr(counts), be.ptr(ids), cap, None, B, flags, be.stream))
            assert int(counts.max()) <= cap
            c = mover if player < 0 else torch.full_like(mover, player)
            if flags & AUTO_RESET:
                c = torch.where(((st[:, 21, 1] >> 16) & 1) == 1, torch.zeros_like(c), c)
            valid = torch.arange(cap, device=dev)[None] < counts[:, None]
            for frame in (0, 1):
                mc, words = be.zeros((B,), np.int32), be.zeros((B, NSHAPE, 20), np.int32)
                be.check(be.lib.crl_blokus_placement_mask(be.ptr(st), player, frame, be.ptr(words), be.ptr(mc), B, flags,
                                                          be.stream))
                got = unpack(words)
                pl = lut[(c * frame).long()[:, None], ids.clamp(min=0).long()]
                exp = torch.zeros((B, NPLACE + 1), dtype=torch.bool, device=dev)
                exp.scatter_(1, torch.where(valid, pl, torch.full_like(pl, NPLACE)), True)
                exp = exp[:, :NPLACE]
                assert torch.equal(got, exp), (K, player, frame, int((got != exp).any(1).sum()))
                assert torch.equal(mc, exp.sum(1).to(torch.int32)), (K, player, frame)
                most = max(most, int(mc.max()))
                assert not ((words.view(torch.int32) >> 20) != 0).any()
                del exp, pl
        # a sample against the oracle directly
        board, pieces, score, meta = cb.blk_unpack(be, st[:sample])
        pos = (board, pieces, score, meta[:, 0], meta[:, 1])
        check_masks(be, st[:sample].contiguous(), pos, players=(-1,), frames=(0, 1))
    assert most > 300, most


def case_python_surface(B=64, seat=1, seed=23, env0=500, steps=200):
    """SingleAgentTurnVectorEnv(action_space="placement", perspective=True) against the learner oracle: the masks of
    every game in the seat's frame, learner placements (legal, illegal, passes) converted to the canonical ids"""
    import torch
    import cases_learner as cl
    from colosseumrl_b200.blokus import BatchedBlokusEnvironment
    from colosseumrl_b200.vector import SingleAgentTurnVectorEnv

    venv = SingleAgentTurnVectorEnv(BatchedBlokusEnvironment(batch=B, seed=seed, first_env_id=env0), seat=seat,
                                    perspective=True, action_space="placement")
    obs = venv.reset()
    ob = cl.BlokusOracle(B)
    ob.advance(None, seat, seed, env0, 0)
    rng = np.random.RandomState(6)
    done_total = illegal_total = 0
    for t in range(1, steps + 1):
        counts, mask = venv.valid_actions()
        counts, mask = counts.cpu().numpy(), mask.cpu().numpy()
        acts, oids = np.full(B, -1, np.int32), np.full(B, -1, np.int32)
        for e in range(B):
            state = (ob.board[e], int(ob.round_count[e]), ob.inventory[e], ob.scores[e])
            if e % 3 == 0:
                o = orc.blokus_observation(state, seat)
                assert (obs["board"][e].cpu().numpy() == o["board"]).all(), (t, e)
            pl, canon = expected(state, seat, 1)
            assert counts[e] == len(pl) and (np.flatnonzero(mask[e]) == pl).all(), (t, e)
            u = rng.rand()
            if len(pl) and u < 0.8:
                acts[e] = int(pl[rng.randint(len(pl))])
                oids[e] = canon[int(acts[e])]
            elif u < 0.9:
                p = int(rng.randint(0, NPLACE))
                if p not in canon:
                    acts[e], oids[e] = p, ILLEGAL
        obs, reward, done, info = venv.step(torch.tensor(acts))
        rec = ob.advance(oids, seat, seed, env0, t)
        assert (reward.cpu().numpy() == rec[:, 0].view(np.int8)).all() and (done.cpu().numpy() == (rec[:, 1] & 1)).all()
        assert (info["illegal"].cpu().numpy() == (rec[:, 1] >> 1 & 1)).all()
        assert (info["scores"].cpu().numpy() == rec[:, 4:8]).all() and (info["winners"].cpu().numpy() == rec[:, 2]).all()
        done_total += int((rec[:, 1] & 1).sum())
        illegal_total += int((rec[:, 1] >> 1 & 1).sum())
    assert done_total > 0 and illegal_total > 0
