"""Single-learner advance cases (crl_ttt_advance, crl_blokus_advance), written once against the C ABI and run on both
backends (tests/backends.py), bit-exact against the C oracle tests/oracle_learner.c, which restates the rule of
include/colosseum_b200_learner.h."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle import oracle as orc
from colosseumrl_b200 import philox
from colosseumrl_b200._lib import STAT_ROWS
import cases_api_contract as api
import cases_blokus as cb
import cases_ttt as ct

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CELLS = {2: 9, 3: 15, 4: 27}
NPIECE_IDS = 21 * 16000                 # action ids 0 .. 335 999 (string form: BlokusEnvironment.py:55-106)
FINISHED, ILLEGAL, PLACED, NO_MOVE = 1, 2, 4, 8

# ----------------------------------------------------------------------------------------------- the oracle
_ORC = None


def oracle_lib():
    """tests/oracle_learner.c + oracle/oracle_ttt.c + oracle/oracle_blokus.c, compiled once per source version into the
    temp directory"""
    global _ORC
    if _ORC is None:
        srcs = [os.path.join(HERE, "oracle_learner.c")] + [os.path.join(ROOT, "oracle", f) for f in ("oracle_ttt.c", "oracle_blokus.c")]
        digest = hashlib.sha1(b"".join(open(s, "rb").read() for s in srcs)).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), "crl_oracle_learner_%s_%d.so" % (digest, os.getuid()))
        if not os.path.exists(so):
            tmp = so + ".%d.tmp" % os.getpid()
            subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-pthread", "-shared", "-o", tmp] + srcs + ["-lm"])
            os.replace(tmp, so)
        _ORC = C.CDLL(so)
    return _ORC


def _p(a, t):
    return None if a is None else a.ctypes.data_as(C.POINTER(t))


class TTTOracle:
    """B games in the reference's layout (board int8 [B, cells], -1 empty; winner -1 = None), driven by the rule.  The
    episode lengths start at 0, as those of a state from crl_ttt_reset or crl_ttt_pack do."""

    def __init__(self, n, B, board=None, winner=None, mover=None):
        self.n, self.B = n, B
        self.board = np.full((B, CELLS[n]), -1, np.int8) if board is None else np.array(board, np.int8).reshape(B, -1)
        self.winner = np.full(B, -1, np.int32) if winner is None else np.array(winner, np.int32)
        self.mover = np.zeros(B, np.int32) if mover is None else np.array(mover, np.int32)
        self.ep_len = np.zeros(B, np.int32)
        self.stats = np.zeros(32, np.int64)

    def advance(self, actions, seat, seed, env0, t):
        rec = np.zeros((self.B, 4), np.uint8)
        act = None if actions is None else np.ascontiguousarray(actions, np.int8)
        oracle_lib().orc_ttt_advance_batch(self.n, seat, _p(act, C.c_int8), C.c_uint64(seed), C.c_int64(env0),
                                           C.c_int64(self.B), C.c_uint32(t), _p(self.board, C.c_int8),
                                           _p(self.winner, C.c_int32), _p(self.mover, C.c_int32), _p(self.ep_len, C.c_int32),
                                           _p(rec, C.c_uint8), _p(self.stats, C.c_int64), 0)
        return rec


class BlokusOracle:
    """B games in the reference's layout (oracle.BlokusBatch's arrays plus the stored terminal flag), driven by the rule"""

    def __init__(self, B, board=None, inventory=None, scores=None, round_count=None, mover=None, terminal=None, ep_len=None):
        self.B = B
        z = lambda a, shape, dt, fill: np.full(shape, fill, dt) if a is None else np.array(a, dt).reshape(shape)
        self.board = z(board, (B, 20, 20), np.int64, 0)
        self.inventory = z(inventory, (B, 4, 21), np.uint8, 1)
        self.scores = z(scores, (B, 4), np.int64, 0)
        self.round_count = z(round_count, (B,), np.int32, 0)
        self.mover = z(mover, (B,), np.int32, 0)
        self.terminal = z(terminal, (B,), np.uint8, 0)
        self.ep_len = z(ep_len, (B,), np.int32, 0)
        self.stats = np.zeros(32, np.int64)

    def advance(self, actions, seat, seed, env0, t):
        rec = np.zeros((self.B, 8), np.uint8)
        act = None if actions is None else np.ascontiguousarray(actions, np.int32)
        oracle_lib().orc_blokus_advance_batch(seat, _p(act, C.c_int32), C.c_uint64(seed), C.c_int64(env0), C.c_int64(self.B),
                                              C.c_uint32(t), _p(self.board, C.c_int64), _p(self.round_count, C.c_int32),
                                              _p(self.inventory, C.c_uint8), _p(self.scores, C.c_int64),
                                              _p(self.mover, C.c_int32), _p(self.terminal, C.c_uint8),
                                              _p(self.ep_len, C.c_int32), _p(rec, C.c_uint8), _p(self.stats, C.c_int64), 0)
        return rec


# ----------------------------------------------------------------------------------------------- device calls
def ttt_advance(be, st, actions, seat, seed, env0, t, n, stats=None, valid_after=True):
    """crl_ttt_advance in place; returns (records uint8 [B, 4], valid_after uint32 [B], or None with valid_after=False:
    the call gets a NULL buffer)"""
    B = st.shape[0]
    a = None if actions is None else be.upload(np.ascontiguousarray(actions, np.int8))
    res, va = be.zeros((B, 4), np.uint8), be.zeros((B,), np.uint32) if valid_after else None
    be.check(be.lib.crl_ttt_advance(be.ptr(st), be.ptr(a), seat, be.ptr(res), be.ptr(va), be.ptr(stats), seed, env0, t, B, n,
                                    be.stream))
    return be.download(res), None if va is None else be.download(va).view(np.uint32)


def blokus_advance(be, st, actions, seat, seed, env0, t, stats=None):
    B = st.shape[0]
    a = None if actions is None else be.upload(np.ascontiguousarray(actions, np.int32))
    res = be.zeros((B, 8), np.uint8)
    be.check(be.lib.crl_blokus_advance(be.ptr(st), be.ptr(a), seat, be.ptr(res), be.ptr(stats), seed, env0, t, B, be.stream))
    return be.download(res)


def ttt_check(be, st, ob, rec, orec, valid):
    """absolute state (board, winner, mover), records and valid_after (unless None) against the oracle"""
    board, winner, mover = ct.ttt_unpack(be, st, ob.n)
    bad = np.flatnonzero((board != ob.board).any(1) | (winner != ob.winner) | (mover != ob.mover) | (rec != orec).any(1))
    assert len(bad) == 0, (bad[:5], rec[bad[:3]], orec[bad[:3]])
    if valid is not None:
        exp = ((ob.board == -1).astype(np.uint64) << np.arange(CELLS[ob.n], dtype=np.uint64)[None]).sum(1)
        assert (valid == exp).all()


def blokus_check(be, st, ob, rec, orec):
    board, pieces, score, meta = cb.blk_unpack(be, st)
    bad = np.flatnonzero((board != ob.board).reshape(ob.B, -1).any(1) | (pieces != ob.inventory).reshape(ob.B, -1).any(1) |
                         (score != ob.scores).any(1) | (meta[:, 0] != ob.round_count) | (meta[:, 1] != ob.mover) |
                         (meta[:, 2] != ob.terminal) | (meta[:, 3] != ob.ep_len) | (rec != orec).any(1))
    assert len(bad) == 0, (bad[:5], rec[bad[:3]], orec[bad[:3]])


# ----------------------------------------------------------------------------------------------- learner actions
def ttt_learner_actions(rng, board):
    """mostly empty cells, some occupied or out-of-range cells, some passes"""
    B, cells = board.shape
    key = rng.rand(B, cells) + (board == -1)                 # an empty cell wins the argmax whenever there is one
    a = key.argmax(1).astype(np.int64)
    u = rng.rand(B)
    occupied = (board != -1)
    occ_pick = (rng.rand(B, cells) + occupied).argmax(1)
    a = np.where((u < 0.08) & occupied.any(1), occ_pick, a)
    a = np.where((u >= 0.08) & (u < 0.12), rng.randint(cells, 128, size=B), a)
    a = np.where((u >= 0.12) & (u < 0.18), -1, a)
    return a.astype(np.int8)


def blokus_learner_actions(rng, counts, ids):
    """an index drawn into the learner's list (crl_blokus_legal(player = seat)), some illegal ids, some passes"""
    B = len(counts)
    pick = np.where(counts > 0, ids[np.arange(B), (rng.rand(B) * np.maximum(counts, 1)).astype(np.int64)], -1)
    u = rng.rand(B)
    pick = np.where(u < 0.1, rng.randint(0, NPIECE_IDS, size=B), pick)
    pick = np.where((u >= 0.1) & (u < 0.16), -1, pick)
    return pick.astype(np.int32)


# ----------------------------------------------------------------------------------------------- cases
def case_ttt_calls(be, n, seat, B, calls, seed=3, env0=100, check_every=1):
    """Seeded learner actions from new_state over `calls` calls: state, record and valid_after after every call (every
    `check_every`-th at scale), the statistics sums at the end.  Returns the oracle and the records seen."""
    st = be.zeros((B, 4), np.int32)
    be.check(be.lib.crl_ttt_reset(be.ptr(st), None, B, n, be.stream))
    ob, stats = TTTOracle(n, B), be.zeros((STAT_ROWS, 32), np.int64)
    rng = np.random.RandomState(seed * 7 + n * 3 + seat)
    recs = []
    for t in range(calls):
        act = ttt_learner_actions(rng, ob.board)
        rec, va = ttt_advance(be, st, act, seat, seed, env0, t, n, stats, valid_after=t % 5 != 4)    # some: NULL valid_after
        orec = ob.advance(act, seat, seed, env0, t)
        if t % check_every == 0 or t == calls - 1:
            ttt_check(be, st, ob, rec, orec, va)
        else:
            assert (rec == orec).all(), t
        recs.append(rec)
    s = be.download(stats).sum(0)
    assert (s == ob.stats).all(), (s, ob.stats)
    recs = np.stack(recs)
    flags = recs[..., 1]
    assert (flags & FINISHED).any() and (flags & ILLEGAL).any() and (flags & PLACED).any()
    assert (recs[..., 3] <= 2 * n - 2).all()
    return ob, recs


def case_blokus_calls(be, seat, B, calls, seed=5, env0=300, check_every=1):
    """Seeded learner actions (indices into its legal list, illegal ids, passes) from new_state over `calls` calls"""
    st = be.zeros((B, 22, 4), np.int32)
    be.check(be.lib.crl_blokus_reset(be.ptr(st), None, B, be.stream))
    ob, stats = BlokusOracle(B), be.zeros((STAT_ROWS, 32), np.int64)
    rng = np.random.RandomState(seed * 11 + seat)
    recs = []
    for t in range(calls):
        counts, ids = cb.blk_legal(be, st, player=seat, cap=4096)
        assert counts.max() <= 4096
        act = blokus_learner_actions(rng, counts, ids)
        rec = blokus_advance(be, st, act, seat, seed, env0, t, stats)
        orec = ob.advance(act, seat, seed, env0, t)
        if t % check_every == 0 or t == calls - 1:
            blokus_check(be, st, ob, rec, orec)
        else:
            assert (rec == orec).all(), t
        recs.append(rec)
    s = be.download(stats).sum(0)
    assert (s == ob.stats).all(), (s, ob.stats)
    recs = np.stack(recs)
    flags = recs[..., 1]
    assert (flags & FINISHED).any() and (flags & ILLEGAL).any() and (flags & PLACED).any(), "too few calls"
    assert (recs[..., 3] <= 6).all()
    if seat == 3:
        assert (recs[..., 3] == 6).any()                     # 2P - 2 opponent moves: a game ended on seat 2's move
    return ob, recs


def ttt_max_entries(n, seat, B, seed, env0):
    """Hand-built games in which every call makes 2n - 2 opponent moves and plays the most env-steps a call can
    (seat n - 1): the learner (to move) places a fixed cell, seats 0 .. n - 3 move, seat n - 2 completes a line of
    two of its cells, the game restarts and seats 0 .. n - 2 move again.  Each env id gets the first board (line,
    missing cell) for which its Philox draws do that.  Returns board, winner, mover, actions."""
    import itertools
    assert seat == n - 1
    cells = CELLS[n]
    lines = [sorted(int(c) for c in line) for line in orc.ttt_lines(n)]
    boards, acts = [], []
    for e in range(B):
        w = np.concatenate([philox.env_step_words(seed, [env0 + e], 0, 6)[0], philox.env_step_words(seed, [env0 + e], 0, 7)[0]])
        for line, miss in itertools.product(lines, range(3)):
            have = [c for i, c in enumerate(line) if i != miss]
            board = np.full(cells, -1, np.int8)
            board[have] = n - 2
            learner = next(c for c in range(cells) if board[c] == -1 and c != line[miss])
            board[learner] = seat
            ok = True
            for j in range(n - 1):                           # seats 0 .. n - 2 pick from the empty cells in C order
                empty = np.flatnonzero(board == -1)
                c = int(empty[int(w[j]) % len(empty)])
                if (c == line[miss]) != (j == n - 2):
                    ok = False
                    break
                board[c] = j
            if ok:
                board = np.full(cells, -1, np.int8)
                board[have] = n - 2
                boards.append(board)
                acts.append(learner)
                break
        else:
            raise AssertionError("no board for env %d" % (env0 + e))
    return np.array(boards), np.full(B, -1), np.full(B, seat), np.array(acts, np.int8)


def case_ttt_handbuilt(be, n, seed=9, env0=40):
    """Through crl_ttt_pack: every recorded state of tests/golden/ttt_states.npz (terminal games, carried winners, full
    boards, movers other than the seat) for every seat, with and without learner actions; and the constructed games of
    ttt_max_entries, where every lane of every warp plays 2n - 1 env-steps (the statistics fields at their maximum)."""
    g = np.load(os.path.join(ct.GOLDEN, "ttt_states.npz"))
    k = lambda name: g["p%d_%s" % (n, name)]
    board, winner, mover = k("board"), k("winner"), k("mover")
    T = len(mover)
    seen = set()
    for seat in range(n):
        for mode in ("actions", "null"):
            st = ct.ttt_pack(be, n, board, winner, mover)
            ob = TTTOracle(n, T, board, winner, mover)
            stats = be.zeros((STAT_ROWS, 32), np.int64)
            act = None if mode == "null" else ttt_learner_actions(np.random.RandomState(seat), ob.board)
            for t in range(3):
                rec, va = ttt_advance(be, st, act, seat, seed, env0, t, n, stats)
                orec = ob.advance(act, seat, seed, env0, t)
                ttt_check(be, st, ob, rec, orec, va)
                seen |= {(int(f), int(j)) for f, j in zip(rec[:, 1], rec[:, 3])}
                if act is not None:
                    act = ttt_learner_actions(np.random.RandomState(seat + 10 * t), ob.board)
            assert (be.download(stats).sum(0) == ob.stats).all()
    flags = {f for f, _ in seen}
    assert any(f & NO_MOVE for f in flags) and any(f & FINISHED for f in flags) and any(f & ILLEGAL for f in flags)
    # the maximum: 2n - 2 opponent moves in every game, 64 games = two full warps
    B, seat = 64, n - 1
    board, winner, mover, act = ttt_max_entries(n, seat, B, seed, env0)
    st, stats = ct.ttt_pack(be, n, board, winner, mover), be.zeros((STAT_ROWS, 32), np.int64)
    ob = TTTOracle(n, B, board, winner, mover)
    rec, va = ttt_advance(be, st, act, seat, seed, env0, 0, n, stats)
    orec = ob.advance(act, seat, seed, env0, 0)
    ttt_check(be, st, ob, rec, orec, va)
    assert (rec[:, 3] == 2 * n - 2).all() and (rec[:, 1] == FINISHED | PLACED).all() and (rec[:, 0].view(np.int8) == -1).all()
    s = be.download(stats).sum(0)
    assert (s == ob.stats).all(), (s, ob.stats)
    assert s[0] == B * (2 * n - 1) and s[1] == B


def _blokus_positions():
    """reference-stepped positions (blokus_boards.npz: rounds 0-3, blocked corners) and end-game positions
    (blokus_wide.npz: stuck players, terminal steps): board, inventory, scores, round, mover"""
    g = np.load(os.path.join(cb.GOLDEN, "blokus_boards.npz"))
    w = np.load(os.path.join(cb.GOLDEN, "blokus_wide.npz"))
    return tuple(np.concatenate([g[a], w[b]]) for a, b in (("i_board", "e_i_board"), ("i_inventory", "e_i_inventory"),
                                                          ("i_scores", "e_i_scores"), ("i_round", "e_i_round"),
                                                          ("mover", "e_mover")))


def case_blokus_handbuilt(be, stride=1, calls=3, seed=6, env0=70):
    """Through crl_blokus_pack: the recorded positions, every fourth one stored as terminal, for every seat, with and
    without learner actions: restarts of terminal games, movers other than the seat, players without a move."""
    board, inv, scores, rounds, movers = (x[::stride] for x in _blokus_positions())
    T = len(movers)
    terminal = (np.arange(T) % 4 == 3).astype(np.int32)
    seen = set()
    for seat in range(4):
        for mode in ("actions", "null"):
            st = cb.blk_pack(be, board, inv, scores, rounds, movers, terminal=terminal)
            ob = BlokusOracle(T, np.asarray(board, np.int64), inv, scores, rounds, movers, terminal)
            stats = be.zeros((STAT_ROWS, 32), np.int64)
            rng = np.random.RandomState(seat + 20)
            for t in range(calls):
                act = None
                if mode == "actions":
                    counts, ids = cb.blk_legal(be, st, player=seat, cap=4096)
                    act = blokus_learner_actions(rng, counts, ids)
                rec = blokus_advance(be, st, act, seat, seed, env0, t, stats)
                orec = ob.advance(act, seat, seed, env0, t)
                blokus_check(be, st, ob, rec, orec)
                seen |= {int(f) for f in rec[:, 1]}
            assert (be.download(stats).sum(0) == ob.stats).all()
    assert any(f & NO_MOVE for f in seen) and any(f & FINISHED for f in seen) and any(f & PLACED for f in seen)


def case_ttt_null_mode(be, n, B=200, seed=12, env0=5):
    """actions = NULL is the rule without a learner move: a call on games whose mover is the seat changes nothing
    (flag 8, no opponent move); on the others the opponents play up to the seat"""
    for seat in range(n):
        st = be.zeros((B, 4), np.int32)
        be.check(be.lib.crl_ttt_reset(be.ptr(st), None, B, n, be.stream))
        ob = TTTOracle(n, B)
        for t in range(4):
            before = be.download(st)
            rec, va = ttt_advance(be, st, None, seat, seed, env0, t, n, valid_after=t != 1)
            orec = ob.advance(None, seat, seed, env0, t)
            ttt_check(be, st, ob, rec, orec, va)
            assert (rec[:, 1] == NO_MOVE).all()
            assert (rec[:, 3] == (seat if t == 0 else 0)).all()
            if t > 0:
                assert (be.download(st) == before).all()


def case_blokus_null_mode(be, B=4, seed=12, env0=5):
    for seat in (0, 3):
        st = be.zeros((B, 22, 4), np.int32)
        be.check(be.lib.crl_blokus_reset(be.ptr(st), None, B, be.stream))
        ob = BlokusOracle(B)
        for t in range(2):
            before = be.download(st)
            rec = blokus_advance(be, st, None, seat, seed, env0, t)
            orec = ob.advance(None, seat, seed, env0, t)
            blokus_check(be, st, ob, rec, orec)
            assert (rec[:, 1] == NO_MOVE).all() and (rec[:, 3] == (seat if t == 0 else 0)).all()
            if t > 0:
                assert (be.download(st) == before).all()


def case_sharding(be, game, n=4, B=96, calls=12, seed=4, env0=1000, seat=1):
    """two half batches with first_env offsets == the whole batch: state, records, statistics"""
    table = np.random.RandomState(77).randint(-1, CELLS[n] + 3, size=(calls, B)).astype(np.int8)   # TTT: any cell

    def run(first, size):
        if game == "ttt":
            st = be.zeros((size, 4), np.int32)
            be.check(be.lib.crl_ttt_reset(be.ptr(st), None, size, n, be.stream))
        else:
            st = be.zeros((size, 22, 4), np.int32)
            be.check(be.lib.crl_blokus_reset(be.ptr(st), None, size, be.stream))
        stats, recs = be.zeros((STAT_ROWS, 32), np.int64), []
        for t in range(calls):
            if game == "ttt":
                recs.append(ttt_advance(be, st, table[t, first - env0:first - env0 + size], seat, seed, first, t, n, stats)[0])
            else:
                counts, ids = cb.blk_legal(be, st, player=seat, cap=4096)
                recs.append(blokus_advance(be, st, np.where(counts > 0, ids[:, 0], -1), seat, seed, first, t, stats))
        return be.download(st), np.stack(recs, 1), be.download(stats).sum(0)
    whole = run(env0, B)
    h = B // 2
    halves = [run(env0, h), run(env0 + h, B - h)]
    assert (np.concatenate([halves[0][0], halves[1][0]]) == whole[0]).all()
    assert (np.concatenate([halves[0][1], halves[1][1]]) == whole[1]).all()
    assert (halves[0][2] + halves[1][2] == whole[2]).all()


# ----------------------------------------------------------------------------------------------- API contract
PROTO_HEADER = os.path.join(ROOT, "include", "colosseum_b200_learner.h")
TTT, BLOKUS = "crl_ttt_advance", "crl_blokus_advance"
SCALARS = dict(api.SCALARS, seat=1)


def prototypes():
    saved = api.HEADER
    try:
        api.HEADER = PROTO_HEADER
        return api.prototypes()
    finally:
        api.HEADER = saved


def contract_rows():
    """(entry point, overrides of the valid call, return code, message).  Order: (TTT: n) -> null state or result ->
    B < 0 -> seat -> B == 0 -> (TTT: B >= 2^31) -> alignment of state, result (TTT: and valid_after; Blokus: actions)"""
    rows = []
    for fn, P in ((TTT, 2), (BLOKUS, 4)):
        NULL, NEG, SEAT = fn + ": null state or result", fn + ": negative batch", fn + ": seat must satisfy 0 <= seat < %s" % ("n" if fn == TTT else "4")
        rows += [
            (fn, dict(ALL_NULL=1), api.ARG, NULL), (fn, dict(state=None), api.ARG, NULL), (fn, dict(result=None), api.ARG, NULL),
            (fn, dict(state=None, B=-1, seat=9), api.ARG, NULL), (fn, dict(result=None, B=0), api.ARG, NULL),
            (fn, dict(B=-1), api.ARG, NEG), (fn, dict(B=-1, seat=-1, state="D1"), api.ARG, NEG),
            (fn, dict(seat=-1), api.ARG, SEAT), (fn, dict(seat=P), api.ARG, SEAT), (fn, dict(seat=P, B=0), api.ARG, SEAT),
            (fn, dict(seat=1 << 20, state="D4"), api.ARG, SEAT),
            (fn, dict(B=0), api.OK, None), (fn, dict(B=0, seat=0, state="D1", result="D1"), api.OK, None),
            (fn, dict(state="D8"), api.ARG, fn + ": state must be 16-byte aligned"),
            (fn, dict(state="D4", result="D1"), api.ARG, fn + ": state must be 16-byte aligned"),
        ]
    rows += [
        (TTT, dict(ALL_NULL=1, n=5), api.UNSUPPORTED, api.TTT_N), (TTT, dict(n=1, B=-1, seat=-1), api.UNSUPPORTED, api.TTT_N),
        (TTT, dict(n=4, seat=3, B=0), api.OK, None), (TTT, dict(n=3, seat=3), api.ARG, TTT + ": seat must satisfy 0 <= seat < n"),
        (TTT, dict(B=1 << 31), api.UNSUPPORTED, TTT + ": batch too large for one launch"),
        (TTT, dict(B=1 << 31, state="D8"), api.UNSUPPORTED, TTT + ": batch too large for one launch"),
        (TTT, dict(result="D1"), api.ARG, TTT + ": result and valid_after must be 4-byte aligned"),
        (TTT, dict(valid_after_or_null="D1"), api.ARG, TTT + ": result and valid_after must be 4-byte aligned"),
        (BLOKUS, dict(result="D4"), api.ARG, BLOKUS + ": result must be 8-byte aligned"),
        (BLOKUS, dict(result="D4", actions_or_null="D1"), api.ARG, BLOKUS + ": result must be 8-byte aligned"),
        (BLOKUS, dict(actions_or_null="D1"), api.ARG, BLOKUS + ": actions must be 4-byte aligned"),
        (BLOKUS, dict(actions_or_null="D4", result="D8", B=0), api.OK, None),
    ]
    return rows


def case_contract(lib, emulator):
    """every row: return code, message, and (emulator) nothing written to device memory; emulator = False: the rows that
    pass no device buffer, on the product library"""
    protos = prototypes()
    assert set(protos) == {TTT, BLOKUS}
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
