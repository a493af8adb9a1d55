"""State wire format (SURVEY.md section 8 f-3): colosseumrl_b200/wire.py against the reference's own dill streams.

CPU only (the wire format is host code).  tests/golden/wire_*.dill are `env.serialize_state(state)` of the unmodified
reference (oracle/make_golden_wire.py): the bytes an untouched match server pushes every step (match_server.py:206-207).
"""
import io
import os
import pickle
import pickletools

import numpy as np
import pytest

from oracle import oracle as orc
from oracle import ref_shim

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _golden_state(step):
    """The adapter's look-alike state after recorded step `step` of game 0 of blokus_games.npz."""
    from colosseumrl_b200.single import AI, Board
    g = np.load(os.path.join(GOLDEN, "blokus_games.npz"))
    pieces = [[n for i, n in enumerate(orc.PIECE_NAMES) if g["inventory"][step][q, i]] for q in range(4)]
    state = (Board(g["board"][step]), int(g["round"][step]), [AI(q + 1, pieces[q], g["scores"][step][q]) for q in range(4)])
    return g, state


def _same_state(a, b):
    assert (np.asarray(a[0].board_contents) == np.asarray(b[0].board_contents)).all() and a[1] == b[1]
    for x, y in zip(a[2], b[2]):
        assert x.player_color == y.player_color and list(x.current_pieces) == list(y.current_pieces)
        assert int(x.player_score) == int(y.player_score)


def test_reads_the_references_own_streams():
    """wire.loads on the bytes the real reference wrote: Blokus (real class paths in the stream), TTT, Tron."""
    from colosseumrl_b200 import wire
    g, expect = _golden_state(19)
    raw = open(os.path.join(GOLDEN, "wire_blokus_step20.dill"), "rb").read()
    assert b"colosseumrl.envs.blokus.board" in raw and b"colosseumrl.envs.blokus.ai" in raw
    _same_state(wire.loads(raw), expect)
    board, winner = wire.loads(open(os.path.join(GOLDEN, "wire_ttt2_step4.dill"), "rb").read())
    assert winner is None and board.tolist() == [[1, -1, 1], [-1, 0, -1], [-1, 0, -1]]
    tb, th, td, tde = wire.loads(open(os.path.join(GOLDEN, "wire_tron_step5.dill"), "rb").read())
    assert tb.shape == (19, 19) and len(th) == len(td) == len(tde) == 4 and int((tb > 0).sum()) == 4 + int((tde == 0).sum()) * 5


def test_our_stream_names_the_reference_class_paths():
    """wire.dumps: a protocol-2 pickle whose only globals besides numpy's are the reference's Board / AI paths, written
    without the reference package being importable; round trip through wire.loads."""
    from colosseumrl_b200 import wire
    from colosseumrl_b200.single import BlokusEnvironment
    _, state = _golden_state(30)
    blob = BlokusEnvironment.serialize_state(state)
    globs = set()
    for op, arg, _ in pickletools.genops(blob):
        if op.name == "GLOBAL":
            globs.add(arg)
    assert "colosseumrl.envs.blokus.board Board" in globs and "colosseumrl.envs.blokus.ai AI" in globs
    assert not any("colosseumrl_b200" in x for x in globs), globs
    _same_state(BlokusEnvironment.deserialize_state(blob), state)
    # Tic Tac Toe / Tron states carry no class paths at all
    t = (np.array([[0, -1, 1], [-1, 0, -1], [-1, -1, -1]], np.int8), None)
    back = wire.loads(wire.dumps(t))
    assert (back[0] == t[0]).all() and back[1] is None


def _decoded(raw):
    """A stream decoded without the reference installed: every class the stream names under `colosseumrl.` becomes a
    recording stub (so the tree shows the class path the reference's loader would resolve), numpy / dill resolve
    normally.  Returns a plain tree: ("obj", module, name, {attribute: tree}) / ("array", dtype, shape, bytes) /
    (type name, items or value)."""
    stubs = {}

    class Unpickler(pickle.Unpickler):
        def find_class(self, module, name):
            if module.startswith("colosseumrl."):
                return stubs.setdefault((module, name), type(name, (), {"__module__": module}))
            return super().find_class(module, name)

    def tree(x):
        if isinstance(x, np.ndarray):
            return ("array", x.dtype.str, x.shape, x.tobytes())
        if type(x).__module__.startswith("colosseumrl."):
            return ("obj", type(x).__module__, type(x).__name__, {k: tree(v) for k, v in vars(x).items()})
        if isinstance(x, (list, tuple)):
            return (type(x).__name__, [tree(v) for v in x])
        if isinstance(x, dict):
            return (type(x).__name__, {k: tree(v) for k, v in x.items()})
        return (type(x).__name__, x)

    return tree(Unpickler(io.BytesIO(bytes(raw))).load())


# attributes the reference's objects carry that the adapters' states leave out: AI.all_valid_moves is the AI's scratch
# cache of its last enumeration (ai.py:39; refilled on use, SURVEY.md section 5), Board.player_color the colour of the
# last placement (written by Board.update_board before it is read); the reference ran its valid_actions / next_state on
# streams without them (test_untouched_reference_consumes_our_stream)
_REFERENCE_ONLY = {("colosseumrl.envs.blokus.ai", "AI"): {"all_valid_moves"},
                   ("colosseumrl.envs.blokus.board", "Board"): {"player_color"}}


def _same_as_reference(ours, theirs, where="state"):
    """Our decoded tree equals the reference's: same containers, class paths, dtypes, shapes and values; an object of
    ours carries the reference's attributes (less _REFERENCE_ONLY) with equal values."""
    assert ours[0] == theirs[0], (where, ours[0], theirs[0])
    if ours[0] == "obj":
        assert ours[1:3] == theirs[1:3], where
        extra = set(theirs[3]) - set(ours[3])
        assert set(ours[3]) <= set(theirs[3]) and extra <= _REFERENCE_ONLY.get(ours[1:3], set()), (where, extra)
        for k in ours[3]:
            _same_as_reference(ours[3][k], theirs[3][k], "%s.%s" % (where, k))
    elif ours[0] in ("list", "tuple"):
        assert len(ours[1]) == len(theirs[1]), where
        for i, (a, b) in enumerate(zip(ours[1], theirs[1])):
            _same_as_reference(a, b, "%s[%d]" % (where, i))
    else:
        assert ours == theirs, where


def test_our_streams_decode_like_the_references_own():
    """serialize_state against the bytes the untouched reference's serialize_state wrote for the same states
    (tests/golden/wire_*.dill, oracle/make_golden_wire.py): our stream is protocol 2 without dill's helpers, theirs
    protocol 4 with them, so they are compared as decoded trees -- the class paths the reference's dill.loads resolves,
    every attribute, dtype, shape and value -- rather than opcode by opcode."""
    from colosseumrl_b200 import wire
    from colosseumrl_b200.single import BlokusEnvironment
    _, state = _golden_state(19)                        # the state after step 20 of game 0: the Blokus stream's state
    theirs = open(os.path.join(GOLDEN, "wire_blokus_step20.dill"), "rb").read()
    _same_as_reference(_decoded(BlokusEnvironment.serialize_state(state)), _decoded(theirs))
    # Tic Tac Toe / Tron: the adapters' state layouts ((int8 board, winner); four int64 arrays) with the reference's values
    board, winner = wire.loads(open(os.path.join(GOLDEN, "wire_ttt2_step4.dill"), "rb").read())
    theirs = open(os.path.join(GOLDEN, "wire_ttt2_step4.dill"), "rb").read()
    _same_as_reference(_decoded(wire.dumps((np.array(board.tolist(), np.int8), winner))), _decoded(theirs))
    theirs = open(os.path.join(GOLDEN, "wire_tron_step5.dill"), "rb").read()
    tron = tuple(np.array(a.tolist(), np.int64) for a in wire.loads(theirs))
    _same_as_reference(_decoded(wire.dumps(tron)), _decoded(theirs))


def test_adapters_cover_the_reference_base_environment():
    """Every single-environment adapter defines each member of the reference's BaseEnvironment surface
    (tests/golden/reference_base_environment.json) as the same kind of member -- property, static (callable on the
    class) or method -- taking the reference's parameters in the reference's order, defaults where it has them, and
    nothing more without a default: every call the reference's callers make is a call the adapter takes."""
    import inspect
    import json
    import colosseumrl_b200.single as s
    ref = json.load(open(os.path.join(GOLDEN, "reference_base_environment.json")))["members"]
    assert s.ENVIRONMENT_CLASSES
    for cls in s.ENVIRONMENT_CLASSES.values():
        for name, spec in ref.items():
            raw = inspect.getattr_static(cls, name, None)
            assert raw is not None, (cls, name)
            if spec["kind"] == "property":
                assert isinstance(raw, property), (cls, name)
                continue
            if spec["kind"] == "static":
                assert isinstance(raw, (staticmethod, classmethod)), (cls, name)
            else:
                assert inspect.isfunction(raw), (cls, name)
            params = list(inspect.signature(getattr(cls, name)).parameters.values())
            if spec["kind"] == "method":
                params = params[1:]                                  # self
            want = spec["params"]
            assert [p.name for p in params[:len(want)]] == [n for n, _ in want], (cls, name, params)
            for p, (_, has_default) in zip(params, want):
                assert p.default is not p.empty or not has_default, (cls, name, p)
            assert all(p.default is not p.empty for p in params[len(want):]), (cls, name, params)


@pytest.mark.reference
@pytest.mark.skipif(not ref_shim.available(), reason="needs /root/reference (build container only)")
def test_untouched_reference_consumes_our_stream():
    """The reference's own `deserialize_state` (dill.loads) on our bytes gives REAL Board / AI objects, and the
    reference's `valid_actions` / `next_state` on them reproduce its recorded game (ClientEnvironment.py:176-198, :327-328)."""
    from colosseumrl_b200.single import BlokusEnvironment
    R = ref_shim.load()
    env = R["BlokusEnvironment"]()
    for step in (0, 7, 19, 41):
        g, state = _golden_state(step)
        theirs = env.deserialize_state(BlokusEnvironment.serialize_state(state))
        assert type(theirs[0]) is R["blokus_board"].Board and all(type(p) is R["blokus_ai"].AI for p in theirs[2])
        i = step + 1                                         # the recorded step that starts from this state
        mover = int(g["mover"][i])
        va = env.valid_actions(theirs, mover)
        exp = g["valid_flat"][g["valid_off"][i]:g["valid_off"][i + 1]]
        assert va == ([orc.blokus_action_to_string(int(a)) for a in exp] or [""])
        new, players, rewards, terminal, winners = env.next_state(theirs, [mover], [orc.blokus_action_to_string(int(g["action"][i]))])
        assert (new[0].board_contents == g["board"][i]).all() and players[0] == g["next_mover"][i]
        assert [p.player_score for p in new[2]] == g["scores"][i].tolist() and terminal == bool(g["terminal"][i])
    # and the other direction: the reference's fresh bytes through our reader, with the real classes importable
    _, expect = _golden_state(19)
    state, players = env.new_state()
    for i in range(20):
        state, players, _, _, _ = env.next_state(state, players, [orc.blokus_action_to_string(int(g["action"][i]))])
    _same_state(BlokusEnvironment.deserialize_state(env.serialize_state(state)), expect)


@pytest.mark.reference
@pytest.mark.skipif(not ref_shim.available(), reason="needs /root/reference (build container only)")
def test_adapters_subclass_the_reference_abc_when_it_is_importable():
    """With the reference package importable, the single-environment adapters ARE `BaseEnvironment` subclasses with no
    abstract member left open (colosseumrl/BaseEnvironment.py:10-283); without it they fall back to plain classes."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = ("import sys; sys.path.insert(0, %r)\n"
            "from oracle import ref_shim; ref_shim.load()\n"
            "from colosseumrl.BaseEnvironment import BaseEnvironment\n"
            "import colosseumrl_b200.single as s\n"
            "for c in s.ENVIRONMENT_CLASSES.values():\n"
            "    assert issubclass(c, BaseEnvironment), c\n"
            "    assert not getattr(c, '__abstractmethods__', None), (c, c.__abstractmethods__)\n"
            "print('ok', len(s.ENVIRONMENT_CLASSES))\n" % root)
    out = subprocess.run([sys.executable, "-c", code], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=300)
    assert out.returncode == 0 and out.stdout.strip() == "ok 5", out.stderr[-1500:]
    from colosseumrl_b200 import single
    assert single.SingleEnvironment.__mro__[1] is object or single.SingleEnvironment.__mro__[1].__name__ == "BaseEnvironment"
