"""The packed Tron state of the tuned path (N <= 19, P <= 4, csrc/tron.cuh): vectors 0..8 hold the three bit-planes of
each cell's owner code (0 empty, q + 1 for player q), vectors 9..11 are reserved and always zero, vector 12 is the
header.  Checked against an independent numpy encoder, the oracle and the reference's recorded transitions, on the SIMT
emulator and (marked gpu) on the B200."""
import os

import numpy as np
import pytest

import backends
import cases_tron as ct
from oracle import oracle as orc

SENTINEL = np.int32(np.uint32(0xA5A5A5A5).view(np.int32))


@pytest.fixture(scope="module", params=["hostsim", pytest.param("cuda", marks=pytest.mark.gpu)])
def be(request):
    return backends.HostSim() if request.param == "hostsim" else backends.Cuda()


def encode_planes(board):
    """int8 [B, N, N] owner codes -> int32 [9, B, 4]: vector 3k + j = 32-bit words 4j..4j+3 of plane k, whose bit
    y*N + x is bit k of the code of cell (x, y)."""
    B = board.shape[0]
    code = np.asarray(board, np.int64).reshape(B, -1)
    bits = np.zeros((3, B, 384), np.uint8)
    for k in range(3):
        bits[k, :, :code.shape[1]] = (code >> k) & 1
    words = np.packbits(bits, axis=-1, bitorder="little").view("<u4")             # [3, B, 12]
    return words.reshape(3, B, 3, 4).transpose(0, 2, 1, 3).reshape(9, B, 4).view(np.int32)


def filled(be, B, value=SENTINEL):
    return be.upload(np.full((13, B, 4), value, np.int32))


def pack_into(be, st, N, P, board, heads, dirs, deaths):
    B = board.shape[0]
    b, h, d, de = (be.upload(np.ascontiguousarray(x, t)) for x, t in
                   ((board, np.int8), (heads, np.int32), (dirs, np.int32), (deaths, np.int32)))
    be.check(be.lib.crl_tron_pack(be.ptr(st), be.ptr(b), be.ptr(h), be.ptr(d), be.ptr(de), B, N, P, be.stream))
    return st


def step(be, st, out, actions, N, P, flags=0):
    B = st.shape[1]
    act = np.zeros((B, 4), np.int8)
    act[:, :actions.shape[1]] = actions
    a = be.upload(act)
    res = be.zeros((B, 8), np.uint8)
    be.check(be.lib.crl_tron_step(be.ptr(st), be.ptr(out), be.ptr(a), be.ptr(res), None, B, N, P, flags, be.stream))
    return be.download(res)


def oracle_step(boards, heads, dirs, deaths, actions):
    out = [orc.tron_next_state(s, a)[0] for s, a in zip(zip(boards, heads, dirs, deaths), actions)]
    return tuple(np.stack([o[i] for o in out]) for i in range(4))


GOLDEN_SHAPES = ["tron_N19_P4.npz", "tron_N9_P4.npz", "tron_N7_P3.npz"]


@pytest.mark.parametrize("name", GOLDEN_SHAPES)
def test_encoding_golden_steps(be, name):
    """Packed planes == the numpy encoder on the reference's recorded states, after the recorded step, and after three
    more random steps (in place) checked against the oracle."""
    g = np.load(os.path.join(ct.GOLDEN, name))
    N, P = int(g["N"]), int(g["P"])
    first = g["t"] == 0
    s0 = orc.tron_new_state(N, P)
    prev = [np.where(first.reshape((-1,) + (1,) * (g[k].ndim - 1)), s0[i][None], np.concatenate([s0[i][None], g[k][:-1]], 0))
            for i, k in enumerate(("board", "heads", "directions", "deaths"))]
    B = len(first)
    st = pack_into(be, filled(be, B), N, P, *prev)
    assert (be.download(st)[:9] == encode_planes(prev[0])).all()
    step(be, st, st, g["actions"], N, P)
    assert (be.download(st)[:9] == encode_planes(g["board"])).all()
    cur = (g["board"], g["heads"], g["directions"], g["deaths"])
    rng = np.random.RandomState(N * 10 + P)
    for t in range(3):
        a = rng.randint(-1, 2, size=(B, P))
        step(be, st, st, a, N, P)
        cur = oracle_step(*cur, a)
        assert (be.download(st)[:9] == encode_planes(cur[0])).all(), t


def test_encoding_adversarial(be):
    g = np.load(os.path.join(ct.GOLDEN, "tron_adversarial.npz"))
    for N in sorted(set(g["N"].tolist())):
        for P in sorted(set(g["P"].tolist())):
            m = (g["N"] == N) & (g["P"] == P)
            if not m.any():
                continue
            board = g["board"][m][:, :N, :N]
            st = pack_into(be, filled(be, int(m.sum())), N, P, board, g["heads"][m][:, :P], g["directions"][m][:, :P],
                           g["deaths"][m][:, :P])
            assert (be.download(st)[:9] == encode_planes(board)).all()
            step(be, st, st, g["actions"][m][:, :P], N, P)
            assert (be.download(st)[:9] == encode_planes(g["o_board"][m][:, :N, :N])).all()


def test_reserved_zero_after_reset_pack_and_out_of_place_step(be, N=19, P=4, B=70):
    ref = be.zeros((13, B, 4), np.int32)
    be.check(be.lib.crl_tron_reset(be.ptr(ref), None, B, N, P, be.stream))
    st = filled(be, B)
    be.check(be.lib.crl_tron_reset(be.ptr(st), None, B, N, P, be.stream))
    got = be.download(st)
    assert (got[9:12] == 0).all() and (got == be.download(ref)).all()
    ob = orc.tron_new_state(N, P)
    assert (got[:9] == encode_planes(np.broadcast_to(ob[0], (B, N, N)))).all()
    # pack of stepped states, then an out-of-place step into a sentinel-filled buffer
    rng = np.random.RandomState(1)
    for _ in range(5):
        step(be, ref, ref, rng.randint(-1, 2, size=(B, P)), N, P)
    board, heads, dirs, deaths, _ = ct.tron_unpack(be, ref, N, P)
    st = pack_into(be, filled(be, B), N, P, board, heads, dirs, deaths)
    got = be.download(st)
    assert (got[9:12] == 0).all() and (got[:9] == be.download(ref)[:9]).all()
    a = rng.randint(-1, 2, size=(B, P))
    out = filled(be, B)
    r_out = step(be, st, out, a, N, P, flags=1)
    r_in = step(be, st, st, a, N, P, flags=1)
    assert (r_out == r_in).all()
    assert (be.download(out) == be.download(st)).all()


def test_reserved_never_read_by_step_and_rollout(be, N=19, P=4, B=130, K=40):
    """A sentinel in vectors 9..11 changes nothing that the in-place step or the rollout computes, and stays."""
    zero = be.zeros((13, B, 4), np.int32)
    be.check(be.lib.crl_tron_reset(be.ptr(zero), None, B, N, P, be.stream))
    init = be.download(zero)
    init[9:12] = SENTINEL
    sent = be.upload(init)
    rng = np.random.RandomState(2)
    for t in range(K):
        a = rng.randint(-1, 2, size=(B, P))
        r0 = step(be, zero, zero, a, N, P, flags=1)
        r1 = step(be, sent, sent, a, N, P, flags=1)
        assert (r0 == r1).all(), t
    z, s = be.download(zero), be.download(sent)
    assert (z[9:12] == 0).all() and (s[9:12] == SENTINEL).all()
    assert (z[:9] == s[:9]).all() and (z[12] == s[12]).all()
    res0, res1 = be.zeros((B, 8), np.uint8), be.zeros((B, 8), np.uint8)
    be.check(be.lib.crl_tron_rollout(be.ptr(zero), be.ptr(res0), None, 3, 0, 0, K, B, N, P, be.stream))
    be.check(be.lib.crl_tron_rollout(be.ptr(sent), be.ptr(res1), None, 3, 0, 0, K, B, N, P, be.stream))
    assert (be.download(res0) == be.download(res1)).all()
    z, s = be.download(zero), be.download(sent)
    assert (z[9:12] == 0).all() and (s[9:12] == SENTINEL).all()
    assert (z[:9] == s[:9]).all() and (z[12] == s[12]).all()


def _shared_word_positions(rng, n, N=19):
    """Positions where all four players move (forward) into distinct empty cells of ONE 32-bit word: players 0 and 2
    share plane c0, players 1 and 2 plane c1.  The rest of the board is randomly owned."""
    boards, heads, dirs, deaths, acts = [], [], [], [], []
    moves = ((0, 1, 0), (1, 0, 3), (0, -1, 2), (-1, 0, 1))     # head offset from the target, direction toward it
    while len(boards) < n:
        w = rng.randint(0, (N * N - 1) // 32 + 1)
        cells = np.arange(32 * w, min(32 * w + 32, N * N))
        if len(cells) < 4:
            continue
        tgt = rng.choice(cells, size=4, replace=False)
        h, d = [], []
        for c in tgt:
            dx, dy, di = moves[rng.randint(4)]
            x, y = c % N + dx, c // N + dy
            h.append(y * N + x if 0 <= x < N and 0 <= y < N else -1)
            d.append(di)
        if min(h) < 0 or len(set(h) | set(tgt.tolist())) != 8:
            continue
        board = np.where(rng.rand(N * N) < 0.3, rng.randint(1, 5, size=N * N), 0)
        board[tgt] = 0
        board[h] = np.arange(1, 5)
        boards.append(board.reshape(N, N)); heads.append(h); dirs.append(d)
        deaths.append([0, 0, 0, 0]); acts.append([0, 0, 0, 0])
    return tuple(np.asarray(x, np.int64) for x in (boards, heads, dirs, deaths, acts))


def test_movers_share_a_word(be, n=300):
    N, P = 19, 4
    boards, heads, dirs, deaths, acts = _shared_word_positions(np.random.RandomState(4), n)
    st = pack_into(be, filled(be, n), N, P, boards, heads, dirs, deaths)
    res = ct.unpack_result(step(be, st, st, acts, N, P))
    exp = oracle_step(boards, heads, dirs, deaths, acts)
    assert (res["alive"] == 15).all()                             # every player moved
    assert (be.download(st)[:9] == encode_planes(exp[0])).all()
    board, h2, d2, de2, _ = ct.tron_unpack(be, st, N, P)
    assert (board == exp[0]).all() and (h2 == exp[1]).all() and (d2 == exp[2]).all() and (de2 == exp[3]).all()


@pytest.mark.parametrize("N,P", [(5, 4), (6, 4), (7, 3), (5, 2)])
def test_auto_reset_spawns_share_a_word(be, N, P, B=40):
    """Terminal states auto-reset to new_state, whose spawns lie in one 32-bit word, and are stepped from there."""
    s0 = orc.tron_new_state(N, P)
    assert len(set((s0[1] >> 5).tolist())) < P                   # at least two spawns share a word
    rng = np.random.RandomState(N * 10 + P)
    board = np.broadcast_to(s0[0], (B, N, N)).copy()
    deaths = np.ones((B, P), np.int64)
    deaths[:, 0] = 0                                               # a sole survivor: terminal
    st = pack_into(be, filled(be, B), N, P, board, np.broadcast_to(s0[1], (B, P)), np.broadcast_to(s0[2], (B, P)), deaths)
    a = rng.randint(-1, 2, size=(B, P))
    step(be, st, st, a, N, P, flags=1)
    exp = oracle_step([s0[0]] * B, [s0[1]] * B, [s0[2]] * B, [s0[3]] * B, a)
    assert (be.download(st)[:9] == encode_planes(exp[0])).all()
    got = ct.tron_unpack(be, st, N, P)
    assert all((g == e).all() for g, e in zip(got[:4], exp))
    ref = be.zeros((13, B, 4), np.int32)
    be.check(be.lib.crl_tron_reset(be.ptr(ref), None, B, N, P, be.stream))
    assert (be.download(ref)[:9] == encode_planes(np.broadcast_to(s0[0], (B, N, N)))).all()
