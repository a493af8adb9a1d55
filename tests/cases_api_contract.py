"""Host-side contract of every entry point of include/colosseum_b200.h: which bad arguments it refuses, with which
return code and message, in which order when several are wrong, always before anything is launched; which calls are
accepted as no-ops; what the host-only functions return.

A row is (entry point, arguments that differ from a valid call, expected return value, expected crl_last_error() or
None).  The valid call of every entry point has B = 8, a narrow Tron shape (19 x 19, 4 players), 2-player Tic Tac Toe,
Blokus capacity 16, player -1 and K = 4; its pointer arguments are device buffers (named D; D1 / D4 / D8 = D plus that
many bytes), except parameters the header marks `_or_null`, which are NULL.  Both builds of crl_api.cu run the table
through tests/backends.py: the SIMT emulator runs every row on host arrays, the product library only the rows that pass
no device buffer."""
import ctypes as C
import os
import re

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "colosseum_b200.h")

OK, ARG, CUDA, UNSUPPORTED = 0, 1, 2, 3
COMPACT, COMPACT2, PACKED = 2, 8, 4          # CRL_FLAG_COMPACT_RESULT, CRL_FLAG_COMPACT2_RESULT, CRL_FLAG_PACKED_ACTIONS
DEVICE = ("D", "D1", "D4", "D8")             # placeholders of device buffers
ALL_NULL = "ALL_NULL"                        # as an override key: every pointer argument NULL

SCALARS = dict(device=0, seed=1, first_env=0, step=0, step0=0, tag=0, K=4, B=8, N=19, P=4, n=2, flags=0, ring_offset=1,
               spawn_offset=2, player=-1, capacity=16, accumulate=0)
HOST_ARRAYS = {                              # HOST pointer parameters: ctypes arrays instead of device buffers
    "crl_tron_start_positions": ("heads", "directions"),
    "crl_tron_start_positions_at": ("heads", "directions"),
    "crl_tron_start_positions_spawns": ("spawn_offsets", "heads", "directions"),
    "crl_tron_reset_spawns": ("spawn_offsets",),
    "crl_tron_step_spawns": ("spawn_offsets",),
}


def prototypes():
    """entry point -> [(parameter name, is a pointer)] in header order"""
    text = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    out = {}
    for name, params in re.findall(r"\b(crl_[a-z0-9_]+)\s*\(([^)]*)\)\s*;", text):
        params = [p.strip() for p in params.split(",")] if params.strip() != "void" else []
        out[name] = [(p.split()[-1].lstrip("*"), "*" in p or p.startswith("crl_stream_t")) for p in params]
    return out


# messages
BOARD = "tron: board size must satisfy 5 <= N <= 64"
PLAYERS = "tron: player count must satisfy 2 <= P <= 8"
TRON_NEG_B = "tron: negative batch"
SPAWNS = "tron: cannot place spawns for this N / P / ring_offset / spawn_offset"
NULL_SPAWNS = "tron: null spawn_offsets"
STEP_NULL = "crl_tron_step: null pointer"
STEP_FLAGS = "crl_tron_step: compact records / packed actions exist for N <= 19, P <= 4 only"
STEP_WIDE_ALIGN = "crl_tron_step: actions must be 8-byte, result 16-byte aligned"
STEP_ALIGN = "crl_tron_step: state buffers must be 16-byte aligned"
STEP_BIG = "crl_tron_step: batch too large for one launch"
TTT_N = "tictactoe: players must be 2, 3 or 4"
NO_RUNTIME = ": no CUDA runtime in the emulator build"


def bad(fn):
    return fn + ": bad argument"


def nulls(fn, names, msg, **kw):
    """one row per required pointer set to NULL"""
    return [(fn, dict(kw, **{p: None}), ARG, msg) for p in names]


def tron_rows():
    rows = []
    for fn in ("crl_tron_start_positions", "crl_tron_start_positions_at", "crl_tron_start_positions_spawns"):
        rows += [
            (fn, dict(N=4), UNSUPPORTED, BOARD), (fn, dict(N=65, heads=None), UNSUPPORTED, BOARD),
            (fn, dict(P=1), UNSUPPORTED, PLAYERS), (fn, dict(P=9, directions=None), UNSUPPORTED, PLAYERS),
            (fn, dict(N=4, P=9), UNSUPPORTED, BOARD),
        ] + nulls(fn, ("heads", "directions"), "crl_tron_start_positions: null pointer")
    rows += [
        ("crl_tron_start_positions_at", dict(ring_offset=9, spawn_offset=0), ARG, SPAWNS),      # no such ring
        ("crl_tron_start_positions_at", dict(ring_offset=-1, spawn_offset=0), ARG, SPAWNS),
        ("crl_tron_start_positions_at", dict(N=5, P=8, ring_offset=2), ARG, SPAWNS),
        ("crl_tron_start_positions_at", dict(N=64, P=8, ring_offset=31), ARG, SPAWNS),
        ("crl_tron_start_positions_spawns", dict(spawn_offsets=None), ARG, NULL_SPAWNS),
        ("crl_tron_start_positions_spawns", dict(spawn_offsets=None, heads=None), ARG, "crl_tron_start_positions: null pointer"),
        ("crl_tron_start_positions_spawns", dict(spawn_offsets=None, ring_offset=9), ARG, NULL_SPAWNS),
        ("crl_tron_start_positions_spawns", dict(ring_offset=9), ARG, SPAWNS),
    ]

    # resets: range (N, P, B) -> null state -> null spawn_offsets -> spawn ring -> B == 0
    for fn in ("crl_tron_reset", "crl_tron_reset_at", "crl_tron_reset_spawns"):
        rows += [
            (fn, dict(ALL_NULL=1, N=4), UNSUPPORTED, BOARD), (fn, dict(ALL_NULL=1, N=65, P=9), UNSUPPORTED, BOARD),
            (fn, dict(ALL_NULL=1, P=9), UNSUPPORTED, PLAYERS), (fn, dict(ALL_NULL=1, P=1, B=-1), UNSUPPORTED, PLAYERS),
            (fn, dict(ALL_NULL=1, B=-1), ARG, TRON_NEG_B), (fn, dict(B=-1), ARG, TRON_NEG_B),
            (fn, dict(ALL_NULL=1), ARG, "crl_tron_reset: null state"),
            (fn, dict(state=None, B=0), ARG, "crl_tron_reset: null state"),
            (fn, dict(B=0), OK, None), (fn, dict(B=0, N=25), OK, None), (fn, dict(B=0, P=8), OK, None),
            (fn, dict(B=0, state="D1"), OK, None),
        ]
    rows += [
        ("crl_tron_reset_at", dict(ring_offset=9), ARG, SPAWNS),
        ("crl_tron_reset_at", dict(ring_offset=9, B=0), ARG, SPAWNS),
        ("crl_tron_reset_at", dict(ring_offset=12, N=25, B=0), ARG, SPAWNS),
        ("crl_tron_reset_at", dict(ring_offset=9, state=None), ARG, "crl_tron_reset: null state"),
        ("crl_tron_reset_spawns", dict(spawn_offsets=None), ARG, NULL_SPAWNS),
        ("crl_tron_reset_spawns", dict(spawn_offsets=None, B=0), ARG, NULL_SPAWNS),
        ("crl_tron_reset_spawns", dict(spawn_offsets=None, state=None), ARG, "crl_tron_reset: null state"),
        ("crl_tron_reset_spawns", dict(spawn_offsets=None, ring_offset=9), ARG, NULL_SPAWNS),
        ("crl_tron_reset_spawns", dict(ring_offset=9, B=0), ARG, SPAWNS),
        ("crl_tron_reset_spawns", dict(ring_offset=9, P=6, N=11, B=0), ARG, SPAWNS),
    ]

    # steps: range -> (step_spawns: null spawn_offsets) -> null pointers -> wide: flags -> spawn ring -> B == 0 ->
    # wide actions / result alignment; narrow: state alignment -> batch size
    for fn in ("crl_tron_step", "crl_tron_step_spawns"):
        rows += [
            (fn, dict(ALL_NULL=1, N=4), UNSUPPORTED, BOARD), (fn, dict(ALL_NULL=1, P=9, B=-1), UNSUPPORTED, PLAYERS),
            (fn, dict(ALL_NULL=1, B=-1), ARG, TRON_NEG_B), (fn, dict(B=-1, flags=COMPACT, N=25), ARG, TRON_NEG_B),
            (fn, dict(state_in=None, state_out=None, actions=None, result=None, flags=COMPACT, N=25), ARG, STEP_NULL),
            (fn, dict(state_in=None, B=0), ARG, STEP_NULL),
            (fn, dict(state_in="D8"), ARG, STEP_ALIGN), (fn, dict(state_out="D1"), ARG, STEP_ALIGN),
            (fn, dict(state_in="D8", B=1 << 30), ARG, STEP_ALIGN),
            (fn, dict(B=1 << 29), UNSUPPORTED, STEP_BIG), (fn, dict(B=1 << 29, flags=PACKED), UNSUPPORTED, STEP_BIG),
            (fn, dict(B=0), OK, None), (fn, dict(B=0, state_in="D8", state_out="D4"), OK, None),
            (fn, dict(B=0, flags=COMPACT | COMPACT2 | PACKED), OK, None),
            # the wide layout (N > 19 or P > 4)
            (fn, dict(N=25, flags=COMPACT), UNSUPPORTED, STEP_FLAGS), (fn, dict(P=5, flags=COMPACT2), UNSUPPORTED, STEP_FLAGS),
            (fn, dict(N=64, P=8, flags=PACKED, B=0), UNSUPPORTED, STEP_FLAGS),
            (fn, dict(N=25, flags=PACKED, actions="D1"), UNSUPPORTED, STEP_FLAGS),
            (fn, dict(N=25, actions="D4"), ARG, STEP_WIDE_ALIGN), (fn, dict(N=25, result="D8"), ARG, STEP_WIDE_ALIGN),
            (fn, dict(P=6, N=11, actions="D1", result="D1"), ARG, STEP_WIDE_ALIGN),
            (fn, dict(N=25, B=0), OK, None), (fn, dict(N=25, B=0, actions="D1", result="D4"), OK, None),
            (fn, dict(N=25, B=0, state_in="D1", flags=1), OK, None),
        ] + nulls(fn, ("state_in", "state_out", "actions", "result"), STEP_NULL) \
          + nulls(fn, ("state_in", "state_out", "actions", "result"), STEP_NULL, N=25, flags=COMPACT)
    rows += [
        ("crl_tron_step_spawns", dict(ALL_NULL=1), ARG, NULL_SPAWNS),
        ("crl_tron_step_spawns", dict(spawn_offsets=None, B=0), ARG, NULL_SPAWNS),
        ("crl_tron_step_spawns", dict(spawn_offsets=None, N=25, flags=COMPACT), ARG, NULL_SPAWNS),
        ("crl_tron_step_spawns", dict(state_in=None, ring_offset=9), ARG, STEP_NULL),
        ("crl_tron_step_spawns", dict(ring_offset=9), ARG, SPAWNS),
        ("crl_tron_step_spawns", dict(ring_offset=9, B=0), ARG, SPAWNS),
        ("crl_tron_step_spawns", dict(ring_offset=9, state_in="D8"), ARG, SPAWNS),
        ("crl_tron_step_spawns", dict(ring_offset=12, N=25, B=0), ARG, SPAWNS),
        ("crl_tron_step_spawns", dict(ring_offset=12, N=25, actions="D1"), ARG, SPAWNS),
        ("crl_tron_step_spawns", dict(ring_offset=12, N=25, flags=COMPACT), UNSUPPORTED, STEP_FLAGS),
    ]

    rows += [
        ("crl_tron_policy_random", dict(actions=None), ARG, bad("crl_tron_policy_random")),
        ("crl_tron_policy_random", dict(B=-1), ARG, bad("crl_tron_policy_random")),
        ("crl_tron_policy_random", dict(B=0), OK, None), ("crl_tron_policy_random", dict(B=0, actions="D1"), OK, None),
        ("crl_tron_policy_random_wide", dict(actions=None), ARG, bad("crl_tron_policy_random_wide")),
        ("crl_tron_policy_random_wide", dict(B=-1), ARG, bad("crl_tron_policy_random_wide")),
        ("crl_tron_policy_random_wide", dict(actions="D4"), ARG, bad("crl_tron_policy_random_wide")),
        ("crl_tron_policy_random_wide", dict(actions="D1", B=0), ARG, bad("crl_tron_policy_random_wide")),
        ("crl_tron_policy_random_wide", dict(B=0), OK, None),
        ("crl_tron_policy_random_wide", dict(B=0, actions="D8"), OK, None),
    ]

    # rollout / observe / ranking / pack: range -> null pointers and other scalars -> B == 0 (rollout: or K == 0) ->
    # wide ranking alignment
    for fn in ("crl_tron_rollout", "crl_tron_observe", "crl_tron_ranking", "crl_tron_pack"):
        rows += [
            (fn, dict(ALL_NULL=1, N=4), UNSUPPORTED, BOARD), (fn, dict(ALL_NULL=1, N=65), UNSUPPORTED, BOARD),
            (fn, dict(ALL_NULL=1, P=9), UNSUPPORTED, PLAYERS), (fn, dict(ALL_NULL=1, P=1, B=-1), UNSUPPORTED, PLAYERS),
            (fn, dict(ALL_NULL=1, B=-1), ARG, TRON_NEG_B), (fn, dict(B=-1, N=25), ARG, TRON_NEG_B),
            (fn, dict(B=0), OK, None), (fn, dict(B=0, N=25), OK, None), (fn, dict(B=0, N=5, P=8), OK, None),
            (fn, dict(B=0, N=64, P=2), OK, None), (fn, dict(B=0, N=5, P=2), OK, None),
        ]
    rows += nulls("crl_tron_rollout", ("state",), bad("crl_tron_rollout")) + [
        ("crl_tron_rollout", dict(K=-1), ARG, bad("crl_tron_rollout")),
        ("crl_tron_rollout", dict(K=-1, B=0), ARG, bad("crl_tron_rollout")),
        ("crl_tron_rollout", dict(K=-1, N=25, B=0), ARG, bad("crl_tron_rollout")),
        ("crl_tron_rollout", dict(state=None, K=0), ARG, bad("crl_tron_rollout")),
        ("crl_tron_rollout", dict(K=0), OK, None), ("crl_tron_rollout", dict(K=0, N=25), OK, None),
        ("crl_tron_rollout", dict(K=0, P=6, N=11, state="D1"), OK, None),
    ]
    rows += nulls("crl_tron_observe", ("state", "board"), bad("crl_tron_observe")) + [
        ("crl_tron_observe", dict(player=4), ARG, bad("crl_tron_observe")),
        ("crl_tron_observe", dict(player=-4), ARG, bad("crl_tron_observe")),
        ("crl_tron_observe", dict(player=-2), ARG, bad("crl_tron_observe")),
        ("crl_tron_observe", dict(player=2, P=2), ARG, bad("crl_tron_observe")),
        ("crl_tron_observe", dict(player=6, P=6, N=11), ARG, bad("crl_tron_observe")),
        ("crl_tron_observe", dict(player=-2, B=0), ARG, bad("crl_tron_observe")),
        ("crl_tron_observe", dict(ALL_NULL=1, player=9, N=99), UNSUPPORTED, BOARD),
        ("crl_tron_observe", dict(B=0, player=3), OK, None), ("crl_tron_observe", dict(B=0, player=-3), OK, None),
        ("crl_tron_observe", dict(B=0, player=0, heads=None, directions=None, deaths=None), OK, None),
        ("crl_tron_observe", dict(B=0, player=5, P=6, N=11), OK, None),
        ("crl_tron_observe", dict(B=0, player=-3, P=8, N=64), OK, None),
    ]
    rows += nulls("crl_tron_ranking", ("state", "ranking"), "crl_tron_ranking: null pointer") + [
        ("crl_tron_ranking", dict(N=25, ranking="D1"), ARG, "crl_tron_ranking: ranking must be 4-byte aligned for wide shapes"),
        ("crl_tron_ranking", dict(P=5, ranking="D1"), ARG, "crl_tron_ranking: ranking must be 4-byte aligned for wide shapes"),
        ("crl_tron_ranking", dict(N=25, ranking="D1", B=0), OK, None),
        ("crl_tron_ranking", dict(ranking="D1", B=0), OK, None),
        ("crl_tron_ranking", dict(N=25, ranking=None, B=0), ARG, "crl_tron_ranking: null pointer"),
    ]
    rows += nulls("crl_tron_pack", ("state", "board", "heads", "directions", "deaths"), "crl_tron_pack: null pointer") \
        + nulls("crl_tron_pack", ("state", "deaths"), "crl_tron_pack: null pointer", N=25, B=0)
    return rows


def ttt_rows():
    rows = []
    fns = ("crl_ttt_reset", "crl_ttt_step", "crl_ttt_valid_actions", "crl_ttt_policy_random", "crl_ttt_rollout",
           "crl_ttt_observe", "crl_ttt_pack")
    required = {"crl_ttt_reset": ("state",), "crl_ttt_step": ("state_in", "state_out", "actions", "result"),
                "crl_ttt_valid_actions": ("state", "mask"), "crl_ttt_policy_random": ("state", "actions"),
                "crl_ttt_rollout": ("state",), "crl_ttt_observe": ("state", "board"),
                "crl_ttt_pack": ("state", "board", "winner", "mover")}
    # n -> null pointers and other scalars -> B == 0 (rollout: or K == 0) -> rollout batch size
    for fn in fns:
        rows += [
            (fn, dict(ALL_NULL=1, n=5), UNSUPPORTED, TTT_N), (fn, dict(n=1), UNSUPPORTED, TTT_N),
            (fn, dict(n=0, B=-1), UNSUPPORTED, TTT_N), (fn, dict(ALL_NULL=1), ARG, bad(fn)), (fn, dict(B=-1), ARG, bad(fn)),
            (fn, dict(B=0), OK, None), (fn, dict(B=0, n=3), OK, None), (fn, dict(B=0, n=4), OK, None),
            (fn, dict(B=0, ALL_NULL=1), ARG, bad(fn)),
        ] + nulls(fn, required[fn], bad(fn)) + nulls(fn, required[fn], bad(fn), n=4, B=0)
    rows += [
        ("crl_ttt_rollout", dict(K=-1), ARG, bad("crl_ttt_rollout")),
        ("crl_ttt_rollout", dict(K=-1, B=0), ARG, bad("crl_ttt_rollout")),
        ("crl_ttt_rollout", dict(K=0), OK, None), ("crl_ttt_rollout", dict(K=0, n=4, state="D1"), OK, None),
        ("crl_ttt_rollout", dict(B=1 << 31), UNSUPPORTED, "crl_ttt_rollout: batch too large for one launch"),
        ("crl_ttt_rollout", dict(B=1 << 31, K=0), OK, None),
        ("crl_ttt_rollout", dict(B=1 << 31, K=-1), ARG, bad("crl_ttt_rollout")),
        ("crl_ttt_observe", dict(player=2), ARG, bad("crl_ttt_observe")),
        ("crl_ttt_observe", dict(player=4, n=4), ARG, bad("crl_ttt_observe")),
        ("crl_ttt_observe", dict(player=-3), ARG, bad("crl_ttt_observe")),
        ("crl_ttt_observe", dict(player=-3, B=0), ARG, bad("crl_ttt_observe")),
        ("crl_ttt_observe", dict(player=3, B=0, n=4), OK, None),
        ("crl_ttt_observe", dict(player=-2, B=0), OK, None),
        ("crl_ttt_step", dict(B=0, flags=COMPACT, valid_after_or_null="D", stats_or_null="D"), OK, None),
    ]
    return rows


def blokus_rows():
    rows = []
    required = {"crl_blokus_reset": ("state",), "crl_blokus_legal": ("state", "counts", "action_ids"),
                "crl_blokus_is_valid": ("state", "actions", "valid"),
                "crl_blokus_step": ("state_in", "state_out", "actions", "result"),
                "crl_blokus_policy_random": ("counts", "action_ids", "actions"),
                "crl_blokus_pick": ("counts", "action_ids", "choice", "actions"),
                "crl_blokus_observe": ("state", "board", "pieces", "score"),
                "crl_blokus_pack": ("state", "board", "pieces", "score", "meta")}
    for fn, names in required.items():
        rows += [(fn, dict(ALL_NULL=1), ARG, bad(fn)), (fn, dict(B=-1), ARG, bad(fn)), (fn, dict(B=0), OK, None),
                 (fn, dict(B=0, ALL_NULL=1), ARG, bad(fn))] + nulls(fn, names, bad(fn)) + nulls(fn, names, bad(fn), B=0)
    for fn in ("crl_blokus_legal", "crl_blokus_policy_random", "crl_blokus_pick"):
        rows += [(fn, dict(capacity=0), ARG, bad(fn)), (fn, dict(capacity=-1), ARG, bad(fn)),
                 (fn, dict(capacity=0, B=0), ARG, bad(fn)), (fn, dict(capacity=1, B=0), OK, None)]
    for fn in ("crl_blokus_legal", "crl_blokus_is_valid", "crl_blokus_observe"):
        rows += [(fn, dict(player=4), ARG, bad(fn)), (fn, dict(player=4, B=0), ARG, bad(fn)),
                 (fn, dict(player=3, B=0), OK, None), (fn, dict(player=0, B=0), OK, None)]
    rows += [
        ("crl_blokus_legal", dict(player=-7, B=0), OK, None), ("crl_blokus_is_valid", dict(player=-7, B=0), OK, None),
        ("crl_blokus_observe", dict(player=-3), ARG, bad("crl_blokus_observe")),
        ("crl_blokus_observe", dict(player=-2, B=0), OK, None),
        ("crl_blokus_rollout", dict(ALL_NULL=1), ARG, "crl_blokus_rollout: null state"),
        ("crl_blokus_rollout", dict(state=None, B=-1, K=-1), ARG, "crl_blokus_rollout: null state"),
        ("crl_blokus_rollout", dict(state=None, B=0), ARG, "crl_blokus_rollout: null state"),
        ("crl_blokus_rollout", dict(B=-1), ARG, "crl_blokus_rollout: negative batch"),
        ("crl_blokus_rollout", dict(B=-1, K=-1), ARG, "crl_blokus_rollout: negative batch"),
        ("crl_blokus_rollout", dict(K=-1), ARG, "crl_blokus_rollout: negative step count K"),
        ("crl_blokus_rollout", dict(K=-1, B=0), ARG, "crl_blokus_rollout: negative step count K"),
        ("crl_blokus_rollout", dict(B=0), OK, None), ("crl_blokus_rollout", dict(K=0), OK, None),
        ("crl_blokus_rollout", dict(K=0, result_or_null="D", stats_or_null="D"), OK, None),
    ]
    return rows


def common_rows():
    return [
        ("crl_philox_words", dict(out=None), ARG, bad("crl_philox_words")),
        ("crl_philox_words", dict(B=-1), ARG, bad("crl_philox_words")),
        ("crl_philox_words", dict(out=None, B=0), ARG, bad("crl_philox_words")),
        ("crl_philox_words", dict(B=0), OK, None),
        ("crl_stats_reduce", dict(ALL_NULL=1), ARG, "crl_stats_reduce: null pointer"),
        ("crl_stats_reduce", dict(stats_rows=None), ARG, "crl_stats_reduce: null pointer"),
        ("crl_stats_reduce", dict(out=None, accumulate=1), ARG, "crl_stats_reduce: null pointer"),
    ]


# the emulator has no CUDA runtime: the host-policy helpers refuse, crl_init accepts any device index
EMULATOR_ONLY = [
    ("crl_init", dict(), OK, None),
    ("crl_host_graph_launch", dict(), UNSUPPORTED, "crl_host_graph_launch" + NO_RUNTIME),
    ("crl_host_graph_launch_wait", dict(), UNSUPPORTED, "crl_host_graph_launch_wait" + NO_RUNTIME),
    ("crl_host_event_wait", dict(), UNSUPPORTED, "crl_host_event_wait" + NO_RUNTIME),
]


def rows():
    return common_rows() + tron_rows() + ttt_rows() + blokus_rows()


class Buffers:
    """The device buffer D (host memory on the emulator, filled with a sentinel) and the host arrays."""

    def __init__(self, emulator):
        self.emulator = emulator
        if emulator:
            self.raw = np.full(1 << 18, 0xA5, np.uint8)
            base = self.raw.ctypes.data
            self.d = base + (-base) % 256
        self.spawns = (C.c_int32 * 8)(*[2] * 8)
        self.heads, self.dirs = (C.c_int32 * 8)(), (C.c_int32 * 8)()

    def untouched(self):
        return (self.raw == 0xA5).all()

    def value(self, fn, name, v):
        if v == "HOST":
            return {"spawn_offsets": self.spawns, "heads": self.heads, "directions": self.dirs}[name]
        if v in DEVICE:
            assert self.emulator, (fn, name)
            return self.d + {"D": 0, "D1": 1, "D4": 4, "D8": 8}[v]
        return v


def arguments(protos, fn, overrides):
    """(parameter name, value) of the valid call of `fn` with `overrides` applied; pointers as placeholders:
    a DEVICE name, "HOST" (a host array) or None"""
    out = []
    for name, is_ptr in protos[fn]:
        if name in overrides:
            v = overrides[name]
        elif name == "stream":
            v = None
        elif not is_ptr:
            v = SCALARS[name]
        elif ALL_NULL in overrides or name.endswith("_or_null"):
            v = None
        else:
            v = "HOST" if name in HOST_ARRAYS.get(fn, ()) else "D"
        out.append((name, v))
    return out


def call(lib, buffers, fn, args):
    return getattr(lib, fn)(*[buffers.value(fn, name, v) for name, v in args])


# entry points whose contract is their return value (case_host_values)
HOST_VALUE_ONLY = {"crl_version", "crl_last_error", "crl_tron_state_bytes", "crl_tron_action_stride",
                   "crl_tron_result_bytes", "crl_ttt_cells", "crl_ttt_lines", "crl_blokus_state_bytes"}


def case_contract(lib, emulator):
    """Every row: the return value, the message, and (emulator) nothing written to device memory.  emulator = False:
    the product library without a device, rows that pass no device buffer only.  Returns the number of rows run."""
    protos = prototypes()
    assert {fn for fn, *_ in rows() + EMULATOR_ONLY} | HOST_VALUE_ONLY == set(protos)     # every entry point
    buffers = Buffers(emulator)
    ran = 0
    for fn, overrides, expect, msg in rows() + (EMULATOR_ONLY if emulator else []):
        args = arguments(protos, fn, overrides)
        if not emulator and any(v in DEVICE for _, v in args):
            continue
        # leave a different message behind first, so that a refusal which sets none is caught
        assert lib.crl_ttt_cells(0) == -1 if msg != TTT_N else lib.crl_tron_state_bytes(4, 4, 1) == -1
        rc = call(lib, buffers, fn, args)
        err = lib.crl_last_error().decode()
        assert rc == expect, (fn, overrides, rc, expect, err)
        if msg is not None:
            assert err == msg, (fn, overrides, err, msg)
        if emulator:
            assert buffers.untouched(), (fn, overrides)
        ran += 1
    return ran


def case_host_values(lib):
    """Return values of the host-only functions for narrow and wide Tron shapes, the three Tic Tac Toe variants and
    Blokus, and their refusals of unsupported shapes."""
    assert lib.crl_version() == 100
    wide = lambda N, P, B: (P * ((N * N + 31) // 32) + 2 * P + 1) * 4 * B
    assert lib.crl_tron_state_bytes(19, 4, 65536) == 208 * 65536 and lib.crl_tron_state_bytes(5, 2, 1) == 208
    assert lib.crl_tron_state_bytes(19, 4, 0) == 0 and lib.crl_tron_state_bytes(25, 4, 0) == 0
    for N, P, B in ((25, 4, 1), (19, 5, 1), (20, 2, 3), (64, 8, 7), (5, 8, 2), (11, 6, 40)):
        assert lib.crl_tron_state_bytes(N, P, B) == wide(N, P, B), (N, P)
    assert lib.crl_tron_state_bytes(64, 8, 1) == (8 * 128 + 17) * 4
    for args, msg in (((65, 4, 1), BOARD), ((4, 4, 1), BOARD), ((19, 9, 1), PLAYERS), ((19, 1, 1), PLAYERS),
                      ((4, 9, -1), BOARD), ((19, 4, -1), TRON_NEG_B), ((25, 4, -1), TRON_NEG_B)):
        assert lib.crl_tron_state_bytes(*args) == -1, args
        assert lib.crl_last_error().decode() == msg, args
    for N, P, stride, rb in ((19, 4, 4, 8), (5, 2, 4, 8), (19, 3, 4, 8), (20, 2, 8, 16), (21, 4, 8, 16), (11, 6, 8, 16),
                             (19, 5, 8, 16), (64, 8, 8, 16), (65, 4, -1, -1), (19, 9, -1, -1), (4, 2, -1, -1)):
        assert (lib.crl_tron_action_stride(N, P), lib.crl_tron_result_bytes(N, P)) == (stride, rb), (N, P)
    assert lib.crl_tron_action_stride(19, 1) == -1 and lib.crl_last_error().decode() == PLAYERS

    # spawns: the default form, the _at form and the per-player form agree; values of the reference's generator
    expected = {(19, 4): ([30, 226, 330, 134], [2, 3, 0, 1]), (25, 4): ([39, 373, 585, 251], [2, 3, 0, 1]),
                (11, 6): ([17, 53, 108, 103, 78, 23], [2, 3, 0, 0, 1, 1]),
                (64, 8): ([82, 113, 1217, 3201, 4013, 3983, 2878, 958], [2, 2, 3, 3, 0, 0, 1, 1]),
                (5, 8): ([6, 7, 8, 13, 18, 17, 16, 11], [2, 2, 3, 3, 0, 0, 1, 1])}
    for (N, P), want in expected.items():
        h, d = (C.c_int32 * 8)(), (C.c_int32 * 8)()
        assert lib.crl_tron_start_positions(N, P, h, d) == 0, (N, P)
        got = (list(h)[:P], list(d)[:P])
        assert got == want, (N, P, got)
        h2, d2 = (C.c_int32 * 8)(), (C.c_int32 * 8)()
        assert lib.crl_tron_start_positions_at(N, P, 1, 2, h2, d2) == 0 and (list(h2)[:P], list(d2)[:P]) == got
        so = (C.c_int32 * 8)(*[2] * 8)
        assert lib.crl_tron_start_positions_spawns(N, P, 1, so, h2, d2) == 0 and (list(h2)[:P], list(d2)[:P]) == got
        assert len(set(got[0])) == P and all(0 <= x < N * N for x in got[0]) and all(0 <= x < 4 for x in got[1])

    assert [lib.crl_ttt_cells(n) for n in (2, 3, 4)] == [9, 15, 27]
    for n in (0, 1, 5, -2):
        assert lib.crl_ttt_cells(n) == -1 and lib.crl_last_error().decode() == TTT_N
    counts = [lib.crl_ttt_lines(n, None, 0) for n in (2, 3, 4)]
    assert counts == [8, 20, 49], counts
    for n, cnt in zip((2, 3, 4), counts):
        masks = (C.c_uint32 * 64)(*[0xFFFFFFFF] * 64)
        assert lib.crl_ttt_lines(n, masks, 64) == cnt
        assert all(bin(m).count("1") == 3 for m in masks[:cnt]) and all(m == 0xFFFFFFFF for m in masks[cnt:])
        short = (C.c_uint32 * 64)(*[0xFFFFFFFF] * 64)
        assert lib.crl_ttt_lines(n, short, 3) == cnt                                 # the count, 3 masks written
        assert list(short[:3]) == list(masks[:3]) and all(m == 0xFFFFFFFF for m in short[3:])
        assert lib.crl_ttt_lines(n, short, -1) == cnt
    assert lib.crl_ttt_lines(5, None, 0) == -1 and lib.crl_last_error().decode() == TTT_N

    assert lib.crl_blokus_state_bytes(16384) == 352 * 16384 and lib.crl_blokus_state_bytes(0) == 0
    assert lib.crl_blokus_state_bytes(-1) == -1
