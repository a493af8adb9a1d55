"""Tron avoid-policy cases (crl_tron_policy_avoid, crl_tron_rollout_avoid), written once against the C ABI and run on
both backends (tests/backends.py), against the C oracle tests/oracle_tron_avoid.c and a numpy restatement of the rule
(include/colosseum_b200_tron_policy.h)."""
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
from cases_tron import GOLDEN, tron_geom, tron_state, tron_pack, tron_unpack, unpack_result, _golden_files

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
AUTO_RESET = 1
MOVE = np.array([0, 1, -1], np.int64)
SENTINEL = 0x55                    # a byte no policy writes: marks the action bytes a call must leave alone

# ----------------------------------------------------------------------------------------------- the oracle
_ORC = None


def oracle_lib():
    """tests/oracle_tron_avoid.c + oracle/oracle_tron.c, compiled once per source version into the temp directory."""
    global _ORC
    if _ORC is None:
        srcs = [os.path.join(HERE, "oracle_tron_avoid.c"), os.path.join(ROOT, "oracle", "oracle_tron.c")]
        digest = hashlib.sha1(b"".join(open(s, "rb").read() for s in srcs)).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), "crl_oracle_tron_avoid_%s_%d.so" % (digest, os.getuid()))
        if not os.path.exists(so):
            tmp = so + ".%d.tmp" % os.getpid()
            subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-pthread", "-shared", "-o", tmp] + srcs + ["-lm"])
            os.replace(tmp, so)
        _ORC = C.CDLL(so)
    return _ORC


def _i64(a):
    return a.ctypes.data_as(C.POINTER(C.c_int64))


def _spawn_arg(spawns, P):
    return None if spawns is None else (C.c_int32 * P)(*spawns)


def orc_new_state(N, P, ring_offset=1, spawns=None):
    board, heads, dirs, deaths = np.zeros((N, N), np.int64), np.zeros(P, np.int64), np.zeros(P, np.int64), np.zeros(P, np.int64)
    assert oracle_lib().orc_tron_new_state_spawns(N, P, ring_offset, _spawn_arg(spawns, P), _i64(board), _i64(heads),
                                                  _i64(dirs), _i64(deaths)) == 0
    return board, heads, dirs, deaths


def orc_avoid(state, actions, mask, noise_q16, seed, env, t):
    """The oracle's decisions for one environment; actions int64 [P] are updated for the seats of mask only."""
    board, heads, dirs, deaths = (np.ascontiguousarray(a, np.int64) for a in state)
    act = np.array(actions, np.int64, copy=True)
    N, P = board.shape[0], heads.shape[0]
    oracle_lib().orc_tron_avoid_actions(N, P, _i64(board), _i64(heads), _i64(dirs), _i64(deaths), int(mask), int(noise_q16),
                                        C.c_uint64(seed), C.c_uint64(env), C.c_uint32(t), _i64(act))
    return act


class AvoidBatch(orc.TronBatch):
    """oracle.TronBatch driven by orc_tron_rollout_avoid (avoid mask, noise, spawns)."""

    def rollout_avoid(self, seed, env0, t0, K, mask, noise_q16, ring_offset=1, spawns=None, fresh=False, nthreads=0):
        oracle_lib().orc_tron_rollout_avoid(
            self.N, self.P, C.c_uint64(seed), C.c_int64(env0), C.c_int64(self.B), C.c_uint32(t0), K, int(fresh), int(mask),
            int(noise_q16), int(ring_offset), _spawn_arg(spawns, self.P), _i64(self.board), _i64(self.heads),
            _i64(self.directions), _i64(self.deaths), self.terminal.ctypes.data_as(C.POINTER(C.c_uint8)),
            self.ep_len.ctypes.data_as(C.POINTER(C.c_int32)), _i64(self.stats), nthreads)


# ----------------------------------------------------------------------------------------------- numpy restatement
def np_avoid(board, heads, dirs, deaths, mask, noise_q16, seed, env, t, actions):
    """The rule of include/colosseum_b200_tron_policy.h for one environment, in numpy.  Returns (actions, why) where why[p]
    names the branch taken: 'masked-out', 'dead', 'noise', 'forward', 'side', 'other-side'."""
    N, P = board.shape[0], len(heads)
    w = np.concatenate([philox.env_step_words(seed, [env], t, 4)[0], philox.env_step_words(seed, [env], t, 5)[0]])
    act, why = np.array(actions, np.int64, copy=True), []

    def free(p, a):
        d = (int(dirs[p]) + a) % 4
        x, y = int(heads[p]) % N + (d == 1) - (d == 3), int(heads[p]) // N + (d == 2) - (d == 0)
        return 0 <= x < N and 0 <= y < N and board[y, x] == 0

    for p in range(P):
        wp = int(w[p])
        if not (mask >> p) & 1:
            why.append("masked-out")
        elif deaths[p] != 0:
            act[p] = 0; why.append("dead")
        elif (wp >> 16) < noise_q16:
            act[p] = MOVE[(wp & 0xFFFF) % 3]; why.append("noise")
        elif free(p, 0):
            act[p] = 0; why.append("forward")
        else:
            side = 1 if wp & 1 else -1
            act[p] = side if free(p, side) else -side
            why.append("side" if free(p, side) else "other-side")
    return act, why


def forward_blocker(board, heads, dirs, p):
    """'wall', 'head' or 'trail': what blocks seat p's forward cell (None if it is free)"""
    N = board.shape[0]
    d = int(dirs[p])
    x, y = int(heads[p]) % N + (d == 1) - (d == 3), int(heads[p]) // N + (d == 2) - (d == 0)
    if not (0 <= x < N and 0 <= y < N):
        return "wall"
    if board[y, x] == 0:
        return None
    return "head" if y * N + x in [int(h) for h in heads] else "trail"


# ----------------------------------------------------------------------------------------------- device calls
def spawn_array(P, spawns):
    return None if spawns is None else (C.c_int32 * P)(*spawns)


def policy_avoid(be, st, actions, mask, noise_q16, seed, env0, t, N, P, flags=0, ring_offset=1, spawns=None):
    """crl_tron_policy_avoid over a [B, stride] int8 host array of prior actions; returns the updated array."""
    B = st.shape[1]
    a = be.upload(np.ascontiguousarray(actions, np.int8))
    be.check(be.lib.crl_tron_policy_avoid(be.ptr(st), be.ptr(a), mask, noise_q16, seed, env0, t, B, N, P, flags,
                                          ring_offset, spawn_array(P, spawns), be.stream))
    return be.download(a)


def expected_policy(board, heads, dirs, deaths, prior, mask, noise_q16, seed, env0, t, flags=0, ring_offset=1, spawns=None):
    """oracle and numpy decisions for a batch of reference-layout states; both must agree.  Returns (actions, whys)."""
    B, P = heads.shape
    N = board.shape[1]
    out, whys = np.array(prior, np.int8, copy=True), []
    for e in range(B):
        state = (board[e], heads[e], dirs[e], deaths[e])
        if (flags & AUTO_RESET) and (deaths[e] == 0).sum() <= 1:             # the stored terminal flag of a packed state
            state = orc_new_state(N, P, ring_offset, spawns)
        o = orc_avoid(state, prior[e, :P].astype(np.int64), mask, noise_q16, seed, env0 + e, t)
        n, why = np_avoid(*state, mask, noise_q16, seed, env0 + e, t, prior[e, :P].astype(np.int64))
        assert (o == n).all(), (e, o, n, why)
        out[e, :P] = o
        whys.append((why, [forward_blocker(state[0], state[1], state[2], p) for p in range(P)]))
    return out, whys


def crowded_boards(rng, N, P, n):
    """hand-built states: trails of every owner, heads crowded together and against the walls, dead seats"""
    boards, heads, dirs, deaths = [], [], [], []
    for i in range(n):
        board = np.zeros((N, N), np.int64)
        fill = rng.rand(N, N) < rng.uniform(0.0, 0.6)
        board[fill] = rng.randint(1, P + 1, size=int(fill.sum()))
        h = rng.choice(N * N, size=P, replace=False).astype(np.int64)
        if i % 3 == 0:                                 # heads next to each other: forward blocked by a head
            c = int(rng.randint(1, N - 1)) * N + int(rng.randint(1, N - 1))
            neigh = [c - 1, c + 1, c - N, c + N, c, c - N - 1, c - N + 1, c + N - 1, c + N + 1]
            rng.shuffle(neigh)
            h = np.asarray(neigh[:P], np.int64)
        elif i % 3 == 1:                               # heads on the border: forward into a wall
            border = [x for x in range(N * N) if x % N in (0, N - 1) or x // N in (0, N - 1)]
            h = rng.choice(border, size=P, replace=False).astype(np.int64)
        board.ravel()[h] = np.arange(1, P + 1)
        boards.append(board); heads.append(h); dirs.append(rng.randint(0, 4, size=P))
        deaths.append(np.where(rng.rand(P) < 0.2, rng.randint(1, P + 1, size=P), 0))
    return tuple(np.asarray(x, np.int64) for x in (boards, heads, dirs, deaths))


def case_rule_handbuilt(be, N=9, P=4, n=600, seed=21, env0=5):
    """The rule on hand-built boards, against the oracle and the numpy restatement: forward blocked by a wall, a trail
    and another player's head; both coin outcomes; both sides blocked; noise 0 and 65536; dead seats; the bytes of
    unmasked and absent seats surviving a sentinel; CRL_FLAG_AUTO_RESET on terminal games with non-default spawns."""
    rng = np.random.RandomState(seed)
    board, heads, dirs, deaths = crowded_boards(rng, N, P, n)
    st = tron_pack(be, N, P, board, heads, dirs, deaths)
    aw, _ = tron_geom(be, N, P)
    prior = np.full((n, aw), SENTINEL, np.int8)
    seen = set()
    full = (1 << P) - 1
    for mask in (full, full & 0b0101, 1 << (P - 1)):
        for noise in (0, 65536, 20000):
            for flags, spawns in ((0, None), (AUTO_RESET, None), (AUTO_RESET, [3, -1, 0, 5, 1, 2, 4, -2][:P])):
                got = policy_avoid(be, st, prior, mask, noise, seed, env0, 7, N, P, flags, 1, spawns)
                exp, whys = expected_policy(board, heads, dirs, deaths, prior, mask, noise, seed, env0, 7, flags, 1, spawns)
                assert (got == exp).all(), (mask, noise, flags, np.argwhere(got != exp)[:5])
                assert (got[:, P:] == SENTINEL).all()                          # absent seats untouched
                for p in range(P):
                    assert ((got[:, p] == SENTINEL) == (not (mask >> p) & 1)).all()  # unmasked seats untouched, others written
                for e, (why, blockers) in enumerate(whys):
                    for p in range(P):
                        if why[p] in ("side", "other-side"):
                            seen.add((why[p], blockers[p]))
                            w = int(philox.env_step_words(seed, [env0 + e], 7, 4 + (p >> 2))[0][p & 3])
                            seen.add(("coin", w & 1))
                        seen.add((why[p], noise))
    for blocker in ("wall", "trail", "head"):
        assert ("side", blocker) in seen or ("other-side", blocker) in seen, blocker
    assert {("coin", 0), ("coin", 1), ("noise", 65536), ("dead", 0), ("dead", 65536)} <= seen, seen
    assert any(w[0] == "other-side" for w in seen) and ("forward", 0) in seen and ("noise", 20000) in seen
    assert not any(w == ("noise", 0) for w in seen)


def case_policy_golden(be):
    """The policy on every recorded state of tests/golden (reference-stepped games, both adversarial sets), several
    masks and noise levels."""
    sets = []
    for path in _golden_files():
        g = np.load(path)
        sets.append((int(g["N"]), int(g["P"]), g["board"], g["heads"], g["directions"], g["deaths"]))
    for name in ("tron_adversarial.npz", "tron_adversarial_wide.npz"):
        g = np.load(os.path.join(GOLDEN, name))
        for N in sorted(set(g["N"].tolist())):
            for P in sorted(set(g["P"].tolist())):
                m = (g["N"] == N) & (g["P"] == P)
                if m.any():
                    sets.append((N, P, g["board"][m][:, :N, :N], g["heads"][m][:, :P], g["directions"][m][:, :P],
                                 g["deaths"][m][:, :P]))
    checked = 0
    for k, (N, P, board, heads, dirs, deaths) in enumerate(sets):
        board, heads, dirs, deaths = (np.asarray(x, np.int64) for x in (board, heads, dirs, deaths))
        st = tron_pack(be, N, P, board, heads, dirs, deaths)
        aw, _ = tron_geom(be, N, P)
        B = len(board)
        prior = np.full((B, aw), SENTINEL, np.int8)
        for mask, noise in (((1 << P) - 1, 0), (1, 6554), (((1 << P) - 1) & ~1, 32768)):
            got = policy_avoid(be, st, prior, mask, noise, 77 + k, 1000, 3, N, P, AUTO_RESET)
            exp, _ = expected_policy(board, heads, dirs, deaths, prior, mask, noise, 77 + k, 1000, 3, AUTO_RESET)
            assert (got == exp).all(), (N, P, mask, noise)
            checked += B
    assert checked > 1000, checked


# ----------------------------------------------------------------------------------------------- fused rollout
def _so(P, spawns):
    return (C.c_int32 * P)(*(spawns if spawns is not None else [2] * P))


def device_reset(be, N, P, B, ring_offset=1, spawns=None):
    st = tron_state(be, N, P, B)
    be.check(be.lib.crl_tron_reset_spawns(be.ptr(st), None, B, N, P, ring_offset, _so(P, spawns), be.stream))
    return st


def chain(be, st, seed, env0, t0, K, N, P, mask, noise_q16, ring_offset=1, spawns=None, stats=None):
    """K x (crl_tron_policy_random[_wide] -> crl_tron_policy_avoid(mask, AUTO_RESET) -> crl_tron_step_spawns(AUTO_RESET)),
    in place; returns the last result record"""
    B = st.shape[1]
    aw, rb = tron_geom(be, N, P)
    act, res = be.zeros((B, aw), np.int8), be.zeros((B, rb), np.uint8)
    random = be.lib.crl_tron_policy_random if aw == 4 else be.lib.crl_tron_policy_random_wide
    for t in range(t0, t0 + K):
        be.check(random(be.ptr(act), seed, env0, t, B, be.stream))
        be.check(be.lib.crl_tron_policy_avoid(be.ptr(st), be.ptr(act), mask, noise_q16, seed, env0, t, B, N, P, AUTO_RESET,
                                              ring_offset, spawn_array(P, spawns), be.stream))
        be.check(be.lib.crl_tron_step_spawns(be.ptr(st), be.ptr(st), be.ptr(act), be.ptr(res), be.ptr(stats), B, N, P,
                                             AUTO_RESET, ring_offset, _so(P, spawns), be.stream))
    return be.download(res)


def rollout_avoid(be, st, seed, env0, t0, K, N, P, mask, noise_q16, ring_offset=1, spawns=None, stats=None, res=None):
    B = st.shape[1]
    be.check(be.lib.crl_tron_rollout_avoid(be.ptr(st), be.ptr(res), be.ptr(stats), seed, env0, t0, K, B, N, P, mask,
                                           noise_q16, ring_offset, spawn_array(P, spawns), be.stream))


def assert_state_equals_oracle(be, st, ob, N, P):
    board, heads, dirs, deaths, term = tron_unpack(be, st, N, P)
    assert (board == ob.board).all() and (heads == ob.heads).all() and (dirs == ob.directions).all()
    assert (deaths == ob.deaths).all() and (term == ob.terminal).all()


def case_rollout_vs_oracle(be, N, P, B, K, mask, noise_q16=0, seed=3, env0=500, ring_offset=1, spawns=None, chain_too=True):
    """crl_tron_rollout_avoid in one launch == the oracle (state, all 32 statistics slots) == the same K steps in two
    launches == the three-launch chain (state, last result record, statistics)."""
    ob = AvoidBatch(B, N, P)
    ob.rollout_avoid(seed, env0, 0, K, mask, noise_q16, ring_offset, spawns, fresh=True)
    rb = tron_geom(be, N, P)[1]
    one, stats1, res1 = device_reset(be, N, P, B, ring_offset, spawns), be.zeros((STAT_ROWS, 32), np.int64), be.zeros((B, rb), np.uint8)
    rollout_avoid(be, one, seed, env0, 0, K, N, P, mask, noise_q16, ring_offset, spawns, stats1, res1)
    assert_state_equals_oracle(be, one, ob, N, P)
    assert (be.download(stats1).sum(0) == ob.stats).all(), (be.download(stats1).sum(0), ob.stats)
    two, stats2, res2 = device_reset(be, N, P, B, ring_offset, spawns), be.zeros((STAT_ROWS, 32), np.int64), be.zeros((B, rb), np.uint8)
    rollout_avoid(be, two, seed, env0, 0, K // 3, N, P, mask, noise_q16, ring_offset, spawns, stats2, None)
    rollout_avoid(be, two, seed, env0, K // 3, K - K // 3, N, P, mask, noise_q16, ring_offset, spawns, stats2, res2)
    assert (be.download(two) == be.download(one)).all() and (be.download(res2) == be.download(res1)).all()
    assert (be.download(stats2).sum(0) == ob.stats).all()
    if chain_too:
        three, stats3 = device_reset(be, N, P, B, ring_offset, spawns), be.zeros((STAT_ROWS, 32), np.int64)
        res3 = chain(be, three, seed, env0, 0, K, N, P, mask, noise_q16, ring_offset, spawns, stats3)
        assert (be.download(three) == be.download(one)).all()
        assert (res3 == be.download(res1)).all()
        assert (be.download(stats3).sum(0) == ob.stats).all()
    return ob


def case_mask_zero_is_random_rollout(be, N, P, B, K, seed=8, env0=40):
    """avoid_mask = 0 with the default spawns: crl_tron_rollout_avoid == crl_tron_rollout bit for bit (state, result,
    statistics), whatever noise_q16 says"""
    rb = tron_geom(be, N, P)[1]
    outs = []
    for fn in ("random", "avoid", "avoid-noise"):
        st, stats, res = device_reset(be, N, P, B), be.zeros((STAT_ROWS, 32), np.int64), be.zeros((B, rb), np.uint8)
        if fn == "random":
            be.check(be.lib.crl_tron_rollout(be.ptr(st), be.ptr(res), be.ptr(stats), seed, env0, 0, K, B, N, P, be.stream))
        else:
            rollout_avoid(be, st, seed, env0, 0, K, N, P, 0, 65536 if fn == "avoid-noise" else 0, 1, None, stats, res)
        outs.append((be.download(st), be.download(res), be.download(stats)))
    for o in outs[1:]:
        assert all((a == b).all() for a, b in zip(outs[0], o))


# ----------------------------------------------------------------------------------------------- meaning
SANITY = dict(N=19, P=4, B=256, K=400, seed=2024, env0=0)


def sanity_counts():
    """seats 1..3 on the avoid policy (noise 0), seat 0 random; and all four random -- on the oracle"""
    s = SANITY
    ob = AvoidBatch(s["B"], s["N"], s["P"])
    ob.rollout_avoid(s["seed"], s["env0"], 0, s["K"], 0b1110, 0, fresh=True)
    rnd = orc.TronBatch(s["B"], s["N"], s["P"])
    rnd.rollout(s["seed"], s["env0"], 0, s["K"], fresh=True)
    return ob, rnd


# the oracle's result for SANITY, from which the bounds below were set: env-steps, episodes, sum of episode lengths,
# wins of seats 0..3, episodes without a winner
SANITY_ORACLE = [102400, 2418, 95570, 3, 560, 492, 1246, 117]


def check_sanity_bounds(stats, random_stats):
    """the avoid seats win far more often than the random seat, and episodes last longer than under random play
    (oracle: 2 418 episodes, wins 3 / 560 / 492 / 1 246, mean length 39.5, against 9 956 episodes of mean length 10.1
    when all four seats play at random)"""
    episodes, eplen, wins = int(stats[1]), int(stats[2]), [int(w) for w in stats[3:7]]
    assert episodes >= 1000, episodes
    assert min(wins[1:]) >= 50 * max(wins[0], 1), wins
    assert eplen / episodes >= 3 * random_stats[2] / random_stats[1], (eplen / episodes, random_stats[2] / random_stats[1])


# ----------------------------------------------------------------------------------------------- API contract
PROTO_HEADER = os.path.join(ROOT, "include", "colosseum_b200_tron_policy.h")
POLICY = "crl_tron_policy_avoid"
ROLLOUT = "crl_tron_rollout_avoid"
SCALARS = dict(api.SCALARS, seat_mask=0b1110, avoid_mask=0b1110, noise_q16=0)


def prototypes():
    saved = api.HEADER
    try:
        api.HEADER = PROTO_HEADER
        return api.prototypes()
    finally:
        api.HEADER = saved


def contract_rows():
    """(entry point, overrides of the valid call, return code, message) in the style of cases_api_contract.py.  Order:
    range (N, P, B) -> null pointers (rollout: and K) -> seat mask -> noise -> spawns -> B == 0 (rollout: or K == 0) ->
    alignment"""
    spawns8 = (C.c_int32 * 8)(*[2] * 8)
    rows = []
    for fn, msg_null in ((POLICY, POLICY + ": null pointer"), (ROLLOUT, ROLLOUT + ": null state")):
        mask = "seat_mask" if fn == POLICY else "avoid_mask"
        MASK, NOISE = fn + ": seat mask bits must be below P", fn + ": noise_q16 must satisfy 0 <= noise_q16 <= 65536"
        rows += [
            (fn, dict(ALL_NULL=1, N=4), api.UNSUPPORTED, api.BOARD),
            (fn, dict(ALL_NULL=1, N=65, P=9), api.UNSUPPORTED, api.BOARD),
            (fn, dict(ALL_NULL=1, P=9), api.UNSUPPORTED, api.PLAYERS), (fn, dict(ALL_NULL=1, P=1, B=-1), api.UNSUPPORTED, api.PLAYERS),
            (fn, dict(ALL_NULL=1, B=-1), api.ARG, api.TRON_NEG_B), (fn, dict(B=-1, N=25, **{mask: 1 << 9}), api.ARG, api.TRON_NEG_B),
            (fn, dict(ALL_NULL=1), api.ARG, msg_null), (fn, dict(state=None, B=0), api.ARG, msg_null),
            (fn, dict(state=None, **{mask: -1, "noise_q16": -1}), api.ARG, msg_null),
            (fn, {mask: 16}, api.ARG, MASK), (fn, {mask: 4, "P": 2}, api.ARG, MASK), (fn, {mask: -1}, api.ARG, MASK),
            (fn, {mask: 1 << 8, "N": 25, "P": 8}, api.ARG, MASK), (fn, {mask: 1 << 6, "N": 11, "P": 6, "B": 0}, api.ARG, MASK),
            (fn, {mask: 16, "noise_q16": -1, "ring_offset": 9}, api.ARG, MASK),
            (fn, dict(noise_q16=-1), api.ARG, NOISE), (fn, dict(noise_q16=65537, B=0), api.ARG, NOISE),
            (fn, dict(noise_q16=1 << 30, ring_offset=9), api.ARG, NOISE),
            (fn, dict(ring_offset=9), api.ARG, api.SPAWNS), (fn, dict(ring_offset=9, B=0), api.ARG, api.SPAWNS),
            (fn, dict(ring_offset=12, N=25, P=8, B=0, **{mask: 0x80}), api.ARG, api.SPAWNS),
            (fn, dict(spawn_offsets_or_null=spawns8, N=5, P=8, ring_offset=2), api.ARG, api.SPAWNS),
            (fn, dict(B=0), api.OK, None), (fn, dict(B=0, noise_q16=65536, **{mask: 0xF}), api.OK, None),
            (fn, dict(B=0, N=64, P=8, **{mask: 0xFF}), api.OK, None), (fn, dict(B=0, state="D1"), api.OK, None),
            (fn, dict(state="D8"), api.ARG, fn + ": state must be 16-byte aligned"),
            (fn, dict(state="D4", noise_q16=65536), api.ARG, fn + ": state must be 16-byte aligned"),
        ]
    rows += [
        (POLICY, dict(actions=None), api.ARG, POLICY + ": null pointer"),
        (POLICY, dict(actions=None, N=25, B=0), api.ARG, POLICY + ": null pointer"),
        (POLICY, dict(seat_mask=0, B=0, actions="D1"), api.OK, None),
        (POLICY, dict(actions="D1"), api.ARG, POLICY + ": actions must be 4-byte aligned"),
        (POLICY, dict(actions="D4", N=25), api.ARG, POLICY + ": actions must be 8-byte aligned for wide shapes"),
        (POLICY, dict(actions="D1", N=11, P=6, seat_mask=0x3F), api.ARG, POLICY + ": actions must be 8-byte aligned for wide shapes"),
        (POLICY, dict(state="D8", actions="D1"), api.ARG, POLICY + ": state must be 16-byte aligned"),
        (ROLLOUT, dict(K=-1), api.ARG, ROLLOUT + ": negative step count K"),
        (ROLLOUT, dict(K=-1, B=0, avoid_mask=16), api.ARG, ROLLOUT + ": negative step count K"),
        (ROLLOUT, dict(K=-1, state=None), api.ARG, ROLLOUT + ": null state"),
        (ROLLOUT, dict(K=0), api.OK, None), (ROLLOUT, dict(K=0, N=25, state="D4"), api.OK, None),
        (ROLLOUT, dict(K=0, avoid_mask=16), api.ARG, ROLLOUT + ": seat mask bits must be below P"),
        (ROLLOUT, dict(K=0, state="D8"), api.OK, None),
    ]
    return rows


def case_contract(lib, emulator):
    """every row: return code, message, and (emulator) nothing written to device memory; emulator = False: the rows that
    pass no device buffer, on the product library"""
    protos = prototypes()
    assert set(protos) == {POLICY, ROLLOUT}
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
