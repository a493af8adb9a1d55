"""Blokus fused rollout (crl_blokus_rollout) cases against the C ABI (both backends): the oracle, the three-launch
legal -> policy -> step sequence, split launches, arbitrary starting positions and sharding.  Every comparison is
bit-exact."""
import os

import numpy as np

from oracle import oracle as orc
from colosseumrl_b200._lib import STAT_ROWS
from colosseumrl_b200 import philox
import cases_blokus as cb

TAG_BLOKUS = 2
CAP = 4096                         # list capacity of the three-launch sequence


def fused(be, st, K, seed, env0, step0=0, stats=None, result=True):
    """One crl_blokus_rollout launch on st (in place); returns the result records (None if not asked for)."""
    B = st.shape[0]
    res = be.zeros((B, 8), np.uint8) if result else None
    be.check(be.lib.crl_blokus_rollout(be.ptr(st), be.ptr(res), be.ptr(stats), seed, env0, step0, K, B, be.stream))
    return res


def chain(be, st, K, seed, env0, stats, cap=CAP):
    """K x (crl_blokus_legal, crl_blokus_policy_random, crl_blokus_step) with auto-reset, in place on st.
    Returns the last step's records and the longest list seen."""
    B = st.shape[0]
    counts, ids = be.zeros((B,), np.int32), be.zeros((B, cap), np.int32)
    act, res = be.zeros((B,), np.int32), be.zeros((B, 8), np.uint8)
    most = 0
    for t in range(K):
        be.check(be.lib.crl_blokus_legal(be.ptr(st), -1, be.ptr(counts), be.ptr(ids), cap, be.ptr(stats), B, 1, be.stream))
        be.check(be.lib.crl_blokus_policy_random(be.ptr(counts), be.ptr(ids), cap, be.ptr(act), seed, env0, t, B, be.stream))
        be.check(be.lib.crl_blokus_step(be.ptr(st), be.ptr(st), be.ptr(act), be.ptr(res), be.ptr(stats), B, 1, be.stream))
        most = max(most, int(be.download(counts).max()))
    return res, most


def four_ways(be, st0, K, seed, env0, k1):
    """From the same states: one fused launch of K; launches of k1 and K - k1 steps; K single-step launches; the
    three-launch sequence.  All four must leave the same states, statistics and last records."""
    host = be.download(st0)
    runs = []
    a, sa = be.upload(host), be.zeros((STAT_ROWS, 32), np.int64)
    runs.append((a, sa, fused(be, a, K, seed, env0, stats=sa)))
    b, sb = be.upload(host), be.zeros((STAT_ROWS, 32), np.int64)
    fused(be, b, k1, seed, env0, 0, sb, result=False)
    runs.append((b, sb, fused(be, b, K - k1, seed, env0, k1, sb)))
    c, sc = be.upload(host), be.zeros((STAT_ROWS, 32), np.int64)
    for t in range(K):
        rc = fused(be, c, 1, seed, env0, t, sc)
    runs.append((c, sc, rc))
    d, sd = be.upload(host), be.zeros((STAT_ROWS, 32), np.int64)
    rd, most = chain(be, d, K, seed, env0, sd)
    assert most <= CAP, most                                  # else the sequence draws from a truncated list
    runs.append((d, sd, rd))
    ref_st, ref_stats, ref_res = (be.download(x) for x in runs[0])
    for i, (s, st, r) in enumerate(runs[1:], 1):
        assert (be.download(s) == ref_st).all(), i
        assert (be.download(st).sum(0) == ref_stats.sum(0)).all(), (i, be.download(st).sum(0), ref_stats.sum(0))
        assert (be.download(r) == ref_res).all(), i
    return a, ref_stats.sum(0), ref_res


def case_fused_vs_oracle(be, B=4, K=72, seed=3, env0=500):
    """One fused launch from new_state == the oracle's rollout: end states and all 32 statistics slots."""
    ob = orc.BlokusBatch(B)
    ob.rollout(seed, env0, 0, K, fresh=True)
    st, stats = be.zeros((B, 22, 4), np.int32), be.zeros((STAT_ROWS, 32), np.int64)
    be.check(be.lib.crl_blokus_reset(be.ptr(st), None, B, be.stream))
    res = cb.unpack_result(be.download(fused(be, st, K, seed, env0, stats=stats)))
    board, pieces, score, meta = cb.blk_unpack(be, st)
    assert (board == ob.board).all() and (pieces == ob.inventory).all() and (score == ob.scores).all()
    assert (meta[:, 0] == ob.round_count).all() and (meta[:, 1] == ob.mover).all()
    assert (meta[:, 2] == ob.terminal).all() and (meta[:, 3] == ob.ep_len).all()
    s = be.download(stats).sum(0)
    assert (s == ob.stats).all(), (s, ob.stats)
    assert (res["terminal"] == ob.terminal.astype(bool)).all() and (res["next_mover"] == ob.mover).all()
    assert ob.stats[1] > 0                                    # the run crossed an episode end


def case_fused_vs_chain(be, B=3, K=40, seed=9, env0=77, k1=13):
    """From new_state: fused (one launch, split, single steps) == the three-launch sequence."""
    st = be.zeros((B, 22, 4), np.int32)
    be.check(be.lib.crl_blokus_reset(be.ptr(st), None, B, be.stream))
    four_ways(be, st, K, seed, env0, k1)


def _positions():
    """The reference-stepped positions of blokus_boards.npz (rounds 0-3, blocked corners) and the end-game positions
    of blokus_wide.npz (bonuses, ties, terminal steps): board, inventory, scores, round, mover."""
    g = np.load(os.path.join(cb.GOLDEN, "blokus_boards.npz"))
    w = np.load(os.path.join(cb.GOLDEN, "blokus_wide.npz"))
    return tuple(np.concatenate([g[a], w[b]]) for a, b in (("i_board", "e_i_board"), ("i_inventory", "e_i_inventory"),
                                                          ("i_scores", "e_i_scores"), ("i_round", "e_i_round"),
                                                          ("mover", "e_mover")))


def case_positions(be, B, stride=1, seed=7, env0=0, strict=True):
    """Arbitrary starting positions, each replicated over env ids chosen so that the first step's draw lands on the
    first, middle and last entry of the mover's list and on the first and last entry of every piece in it; K = 1 and
    K = 3 fused == the three-launch sequence.  strict: every first / middle / last target must be placed."""
    board, inv, scores, rounds, movers = (x[::stride] for x in _positions())
    P = len(movers)
    counts, ids = cb.blk_legal(be, cb.blk_pack(be, board, inv, scores, rounds, movers), cap=CAP)
    assert counts.max() <= CAP
    r = philox.env_step_words(seed, env0 + np.arange(B, dtype=np.uint64), 0, TAG_BLOKUS)[:, 0].astype(np.int64)
    slot = np.full(B, -1, np.int64)
    placed = missed = 0
    for i in range(P):
        n = int(counts[i])
        if n == 0:
            slot[np.flatnonzero(slot < 0)[0]] = i
            continue
        piece = ids[i, :n] // 16000
        starts = np.flatnonzero(np.r_[True, piece[1:] != piece[:-1]])
        ends = np.r_[starts[1:] - 1, n - 1]
        required = {0, n // 2, n - 1}
        for t in sorted(required | set(starts.tolist()) | set(ends.tolist())):
            cand = np.flatnonzero((slot < 0) & (r % n == t))
            if len(cand):
                slot[cand[0]] = i
                placed += 1
            else:
                missed += 1
                assert not (strict and t in required), (i, n, t)
    free = np.flatnonzero(slot < 0)
    slot[free] = np.arange(len(free)) % P                    # the other env ids: every position round robin
    st = cb.blk_pack(be, board[slot], inv[slot], scores[slot], rounds[slot], movers[slot])
    for K in (1, 3):
        four_ways(be, st, K, seed, env0, K // 2)
    return placed, missed


def case_sharding(be, B=6, K=30, seed=4, env0=1000):
    """Two half-batch launches (first_env = env0 and env0 + B/2) == the whole-batch launch: trajectories depend on the
    global env id only."""
    st, stats = be.zeros((B, 22, 4), np.int32), be.zeros((STAT_ROWS, 32), np.int64)
    be.check(be.lib.crl_blokus_reset(be.ptr(st), None, B, be.stream))
    res = fused(be, st, K, seed, env0, stats=stats)
    h = B // 2
    halves, hstats, hres = [], be.zeros((STAT_ROWS, 32), np.int64), []
    for first, size in ((env0, h), (env0 + h, B - h)):
        s = be.zeros((size, 22, 4), np.int32)
        be.check(be.lib.crl_blokus_reset(be.ptr(s), None, size, be.stream))
        hres.append(be.download(fused(be, s, K, seed, first, stats=hstats)))
        halves.append(be.download(s))
    assert (np.concatenate(halves) == be.download(st)).all()
    assert (np.concatenate(hres) == be.download(res)).all()
    assert (be.download(hstats).sum(0) == be.download(stats).sum(0)).all()


def case_argument_checks(lib):
    """Refused host-side, before anything is launched: null state, B < 0, K < 0; B == 0 or K == 0 is a no-op."""
    import ctypes as C
    buf = C.create_string_buffer(352)
    assert lib.crl_blokus_rollout(None, None, None, 1, 0, 0, 4, 8, None) == 1
    assert b"null state" in lib.crl_last_error()
    assert lib.crl_blokus_rollout(buf, None, None, 1, 0, 0, 4, -1, None) == 1
    assert b"negative batch" in lib.crl_last_error()
    assert lib.crl_blokus_rollout(buf, None, None, 1, 0, 0, -1, 8, None) == 1
    assert b"negative step count" in lib.crl_last_error()
    assert lib.crl_blokus_rollout(buf, None, None, 1, 0, 0, 4, 0, None) == 0
    assert lib.crl_blokus_rollout(buf, None, None, 1, 0, 0, 0, 8, None) == 0
    assert buf.raw == b"\0" * 352                             # nothing ran


def case_python_surface(B=256, K=90, seed=5, env0=3000):
    """BatchedBlokusEnvironment.rollout == the oracle: in-place state, state.result = the last record, env.stats."""
    import torch
    from colosseumrl_b200.blokus import BatchedBlokusEnvironment
    env = BatchedBlokusEnvironment(batch=B, seed=seed, first_env_id=env0, device="cuda:0")
    st, _ = env.new_state()
    packed = st.packed
    out = env.rollout(st, 0, K)
    assert out is st and st.packed is packed
    ob = orc.BlokusBatch(B)
    ob.rollout(seed, env0, 0, K, fresh=True)
    obs = env.state_to_observation(st, -1)
    assert (obs["board"].cpu().numpy() == ob.board).all() and (obs["pieces"].cpu().numpy() == ob.inventory).all()
    assert (obs["score"].cpu().numpy() == ob.scores).all() and (obs["round"].cpu().numpy() == ob.round_count).all()
    assert (obs["mover"].cpu().numpy() == ob.mover).all() and (obs["terminal"].cpu().numpy() == ob.terminal).all()
    assert (obs["episode_steps"].cpu().numpy() == ob.ep_len).all()
    assert (env.stats.cpu().numpy() == ob.stats).all()
    # the same K steps through valid_actions -> random_actions -> step_ of an auto-resetting environment
    env2 = BatchedBlokusEnvironment(batch=B, seed=seed, first_env_id=env0, device="cuda:0", auto_reset=True)
    st2, _ = env2.new_state()
    for t in range(K):
        env2.step_(st2, env2.random_actions(env2.valid_actions(st2), t), out=st2)
    assert torch.equal(st2.packed, st.packed) and torch.equal(st2.result, st.result)
    assert torch.equal(env2.stats, env.stats)
    res = cb.unpack_result(st.result.cpu().numpy())
    assert (res["terminal"] == ob.terminal.astype(bool)).all() and (res["next_mover"] == ob.mover).all()
