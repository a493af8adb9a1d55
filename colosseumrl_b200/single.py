"""Single-environment, string-action adapters: the reference's `BaseEnvironment` surface (colosseumrl/
BaseEnvironment.py:10-283) on top of the batched engine with B = 1, for callers that drive ONE game with Python
lists and action strings -- the match server (`match_server.py:64,137,144,193,201-203,240`), `ClientEnvironment`
and the RLlib wrappers (`envs/wrappers/rllib.py:37-55`).

States are *reference-layout* objects (the same tuples of numpy arrays / attribute names the reference's games use),
so code that peeks into a state (`state[0]` is the Tron board, `state[0].board_contents` the Blokus board, ...) keeps
working, `next_state` is functional like the reference's, and `serialize_state` writes the reference's own wire
format (wire.py: the stream names the reference's class paths, so an untouched reference client can load it).
Every call packs the state into the engine's bit-packed layout, runs the same CUDA kernels the batched classes use
and unpacks the result: there is no CPU implementation of the dynamics here, and no GPU means `CrlError`.

Differences from the reference, all deliberate:
  * Tic Tac Toe `valid_actions` returns clean "(r, c)" strings; the reference's own strings are unparsable under
    numpy >= 2 (SURVEY.md Appendix A-X1).
  * a Blokus action string that is not in the mover's valid list is applied as a pass (the reference applies it
    blindly, BlokusEnvironment.py:419-422); `is_valid_action` tells them apart beforehand, as the server does.
"""
from typing import Dict, List

import numpy as np
import torch

from . import blokus as _blokus
from . import wire
from .blokus import BatchedBlokusEnvironment
from .tictactoe import BatchedTicTacToe2PlayerEnv, BatchedTicTacToe3PlayerEnv, BatchedTicTacToe4PlayerEnv
from .tron import BatchedTronGridEnvironment


def _reference_base():
    """The reference's own ABC (colosseumrl/BaseEnvironment.py:10) when that package is importable -- the adapters are
    then real `BaseEnvironment` subclasses, as `server_app` / `RllibWrapper` type-annotate them -- else `object` (the
    engine does not depend on the reference being installed)."""
    try:
        from colosseumrl.BaseEnvironment import BaseEnvironment
        return BaseEnvironment
    except Exception:
        return object


class SingleEnvironment(_reference_base()):
    """Common part of the adapters (BaseEnvironment.py:10-283)."""
    _batched_class = None

    _batched_kwargs = {}

    def __init__(self, config: str = "", device="cuda:0"):
        self._config = config
        self._b = self._batched_class(config, batch=1, device=device, **self._batched_kwargs)
        self._b.collect_stats = False

    @property
    def min_players(self) -> int:
        return self._b.min_players

    @property
    def max_players(self) -> int:
        return self._b.max_players

    @property
    def observation_shape(self) -> Dict[str, tuple]:
        return self._b.observation_shape

    @classmethod
    def observation_names(cls) -> List[str]:
        """Static in the reference (callable on the class): the batched class's names."""
        return cls._batched_class.observation_names()

    def compute_ranking(self, state, players: List[int], winners: List[int]) -> Dict[int, int]:
        """Default ranking (BaseEnvironment.py:173-195): winners 0, everybody else 1."""
        winners = set(int(w) for w in winners)
        return {int(p): (0 if int(p) in winners else 1) for p in players}

    @staticmethod
    def serializable() -> bool:
        return True

    @staticmethod
    def serialize_state(state) -> bytes:
        """The reference's wire format (`dill.dumps(state)`, BlokusEnvironment.py:305-320): a Blokus state names the
        reference's own class paths, so an untouched `ClientEnvironment.full_state` rebuilds it (wire.py)."""
        return wire.dumps(state)

    @staticmethod
    def deserialize_state(serialized_state: bytes):
        """Reads the reference's own serialized states as well as ours (wire.py)."""
        return wire.loads(serialized_state)

    @staticmethod
    def _np(t: torch.Tensor) -> np.ndarray:
        return t.cpu().numpy()


# ------------------------------------------------------------------------------------------------ Tron
class TronGridEnvironment(SingleEnvironment):
    """envs/tron/TronGridEnvironment.py:61-508.  state = (board int64 [N,N], heads, directions, deaths int64 [P])."""
    _batched_class = BatchedTronGridEnvironment
    STRING_TO_ACTION = BatchedTronGridEnvironment.STRING_TO_ACTION

    def __init__(self, config: str = "", device="cuda:0"):
        super().__init__(config, device)
        self.N, self.num_players = self._b.N, self._b.num_players
        self.player_array = np.arange(self.num_players)
        self.move_array = ["forward", "right", "left"]
        self._moves = np.zeros(self.num_players, np.int64)      # persists across calls like the reference's (:118)

    @classmethod
    def create(cls, board_size: int = 19, num_players: int = 4, observation_window: int = -1,
               remove_on_death: bool = False, device="cuda:0") -> "TronGridEnvironment":
        """TronGridEnvironment.create (:69-90): build the environment from options instead of a config string."""
        from .tron import create_tron_config
        return cls(create_tron_config(board_size, num_players, observation_window, remove_on_death), device=device)

    def new_state(self, num_players: int = None, ring_offset: int = 1, spawn_offset=2):
        st, _ = self._b.new_state(num_players, ring_offset, spawn_offset)
        return self._unpack(st), self.player_array

    def generate_start_positions(self, ring_offset: int = 1, spawn_offset: int = 0):
        return self._b.generate_start_positions(ring_offset, spawn_offset)

    def _pack(self, state):
        board, heads, directions, deaths = state
        return self._b.state_from_arrays(np.asarray(board, np.int8)[None], np.asarray(heads, np.int32)[None],
                                         np.asarray(directions, np.int32)[None], np.asarray(deaths, np.int32)[None])

    def _unpack(self, st):
        o = self._b.state_to_observation(st, -1)
        return (self._np(o["board"][0]).astype(np.int64), self._np(o["heads"][0]).astype(np.int64),
                self._np(o["directions"][0]).astype(np.int64), self._np(o["deaths"][0]).astype(np.int64))

    def next_state(self, state, players: List[int], actions: List[str]):
        for player, action in zip(players, actions):
            self._moves[player] = self.STRING_TO_ACTION[action]  # unknown string: KeyError, as in the reference (:298)
        act = torch.zeros((1, self._b.action_stride), dtype=torch.int8)
        act[0, :self.num_players] = torch.from_numpy(self._moves.astype(np.int8))
        new = self._b.step_(self._pack(state), act)
        r = self._np(new.result[0])
        P = self.num_players
        rewards = r[:P].view(np.int8).astype(np.int64)
        alive, term = (r[9], r[8]) if self._b.wide else (r[5], r[4])          # 16-byte record beyond N <= 19, P <= 4
        new_players = np.array([p for p in range(P) if alive >> p & 1], dtype=np.int64)
        terminal = bool(term)
        winners = new_players if terminal else None
        return self._unpack(new), new_players, rewards, terminal, winners

    def valid_actions(self, state, player: int) -> List[str]:
        return self.move_array

    def is_valid_action(self, state, player: int, action: str) -> bool:
        return True

    def compute_ranking(self, state, players=None, winners=None) -> Dict[int, int]:
        """TronGridEnvironment.compute_ranking (:483-508), through crl_tron_ranking."""
        rk = self._np(self._b.compute_ranking(self._pack(state))[0])
        return {p: int(rk[p]) for p in range(self.num_players)}

    def state_to_observation(self, state, player: int) -> Dict[str, np.ndarray]:
        o = self._b.state_to_observation(self._pack(state), player)
        return {k: self._np(v[0]).astype(np.int64) for k, v in o.items()}

    def next_cell(self, x, y, direction, action):
        """Helper used by the reference's example agents (TronGridEnvironment.py): the cell a move leads to."""
        d = (direction + self.STRING_TO_ACTION[action] + 4) % 4
        return x + (d == 1) - (d == 3), y + (d == 2) - (d == 0)


# ------------------------------------------------------------------------------------------------ Blokus
class Board:
    """Look-alike of envs/blokus/board.py:Board: `board_contents` int64 [20, 20], 0 empty, 1..4 colour."""
    def __init__(self, contents=None):
        self.board_contents = np.zeros((20, 20), np.int64) if contents is None else np.array(contents, np.int64)


class AI:
    """Look-alike of envs/blokus/ai.py:AI: colour, remaining piece names (PIECE_TYPES order), score."""
    def __init__(self, color, pieces=None, score=0):
        self.player_score = int(score)
        self.player_color = color
        self.current_pieces = list(_blokus.PIECE_NAMES) if pieces is None else list(pieces)


# on the wire the two look-alikes carry the reference's class paths (wire.py)
wire.register_lookalike("Board", Board)
wire.register_lookalike("AI", AI)


class BlokusEnvironment(SingleEnvironment):
    """envs/blokus/BlokusEnvironment.py:170-768.  state = (Board, round_count, [AI x 4])."""
    _batched_class = BatchedBlokusEnvironment
    _batched_kwargs = {"capacity": 8192}        # longest valid-action list seen in random play: 1 753 (SURVEY section 6)

    @staticmethod
    def all_piece_types() -> List[str]:
        return list(_blokus.PIECE_NAMES)

    @staticmethod
    def all_orientations() -> List[str]:
        return list(_blokus.ORIENTATIONS)

    def new_state(self, num_players: int = 4):
        assert num_players is None or num_players == 4
        return (Board(), 0, [AI(c) for c in (1, 2, 3, 4)]), [0]

    def _pack(self, state, mover: int):
        board, round_count, players = state
        inv = np.zeros((1, 4, 21), np.uint8)
        for q, pl in enumerate(players):
            for name in pl.current_pieces:
                inv[0, q, _blokus.PIECE_NAMES.index(name)] = 1
        score = np.array([[pl.player_score for pl in players]], np.int32)
        return self._b.state_from_arrays(board.board_contents.astype(np.int8)[None], inv, score,
                                         np.array([round_count], np.int32), np.array([mover], np.int32))

    def _unpack(self, st):
        o = self._b.state_to_observation(st, -1)
        board = Board(self._np(o["board"][0]))
        pieces, score = self._np(o["pieces"][0]), self._np(o["score"][0])
        players = [AI(q + 1, [n for i, n in enumerate(_blokus.PIECE_NAMES) if pieces[q, i]], score[q]) for q in range(4)]
        return board, players

    def current_rewards(self, state) -> List[float]:
        return [float(pl.player_score) for pl in state[2]]

    def next_state(self, state, players: List[int], actions: List[str]):
        mover, action = int(players[0]), actions[0]
        aid = _blokus.string_to_action(action)
        new = self._b.step_(self._pack(state, mover), torch.tensor([aid], dtype=torch.int32))
        r = self._np(new.result[0])
        board, pls = self._unpack(new)
        terminal = bool(r[1] & 1)
        winners = [q for q in range(4) if r[2] >> q & 1] if terminal else None
        round_count = state[1] + (1 if mover == 3 else 0)
        return (board, round_count, pls), [int(r[4])], [int(np.int8(r[0]))], terminal, winners

    def valid_actions(self, state, player: int) -> List[str]:
        counts, ids = self._b.valid_actions(self._pack(state, player), player)
        n = int(counts[0])
        if n == 0:
            return [""]
        if n > ids.shape[1]:
            raise RuntimeError("valid-action list longer than the adapter's capacity (%d > %d)" % (n, ids.shape[1]))
        return [_blokus.action_to_string(int(a)) for a in self._np(ids[0, :n])]

    def valid_actions_dict(self, state, player: int) -> Dict[str, Dict[tuple, List[str]]]:
        """valid_actions_dict (:630-665) = Board.get_all_valid_moves (board.py:170-193): {piece: {(x, y): ["orientk", ...]}}
        with the reference's insertion order (pieces in inventory order, anchors row-major, orientation, shift).
        `valid_actions` is this dictionary flattened (:490-496), so it is rebuilt from the ordered id list."""
        out: Dict[str, Dict[tuple, List[str]]] = {}
        for a in self.valid_actions(state, player):
            if a == "":
                continue
            piece, index, orientation = a.split(";")
            x, y = (int(v) for v in index.strip("()").split(","))
            out.setdefault(piece, {}).setdefault((x, y), []).append(orientation)
        return out

    def player_perspective_valid_actions(self, state, player: int) -> List[str]:
        """BlokusEnvironment.py:502-551: valid actions in the frame of the player's rotated observation."""
        return [self.convert_real_action_to_player_perspective_action(a, player) for a in self.valid_actions(state, player)]

    @staticmethod
    def convert_real_action_to_player_perspective_action(action: str, player: int) -> str:
        """:553-588"""
        return _blokus.action_to_string(_blokus.real_action_to_player_perspective(_blokus.string_to_action(action), player))

    @staticmethod
    def convert_player_perspective_action_to_real_action(player_action: str, player: int) -> str:
        """:591-628"""
        return _blokus.action_to_string(_blokus.player_perspective_action_to_real(_blokus.string_to_action(player_action), player))

    def is_valid_action(self, state, player: int, action: str) -> bool:
        if len(action) == 0:                   # '' is not a valid action here either (BlokusEnvironment.py:702,
            return False                       # tictactoe_2p_env.py:372); match_server special-cases it itself
        try:
            aid = _blokus.string_to_action(action)
        except (ValueError, KeyError, IndexError):
            return False
        return bool(self._b.is_valid_action(self._pack(state, player), player, torch.tensor([aid], dtype=torch.int32))[0])

    def state_to_observation(self, state, player: int) -> Dict[str, np.ndarray]:
        o = self._b.state_to_observation(self._pack(state, player), player)
        return {"board": self._np(o["board"][0]).astype(np.int64), "pieces": self._np(o["pieces"][0]),
                "score": self._np(o["score"][0]).astype(np.int64), "player": np.array([player])}


# ------------------------------------------------------------------------------------------------ Tic Tac Toe
class _TicTacToe(SingleEnvironment):
    """envs/tictactoe/tictactoe_{2,3,4}p_env.py.  state = (board int8 [shape] with -1 empty, winner | None)."""
    _shape = (3, 3)

    def new_state(self, num_players: int = None):
        assert num_players is None or num_players == self.max_players
        return (np.full(self._shape, -1, np.int8), None), [0]

    def current_rewards(self, state) -> List[float]:
        """current_rewards (tictactoe_2p_env.py:219-238): +1 winner / -1 everybody else once there is a winner, else 0."""
        winner = state[1]
        return [0 if winner is None else (1 if p == winner else -1) for p in range(self.max_players)]

    def _pack(self, state, mover: int):
        board, winner = state
        return self._b.state_from_arrays(np.asarray(board, np.int8).reshape(1, -1),
                                         np.array([-1 if winner is None else winner], np.int8), np.array([mover], np.int8))

    def _index(self, action: str) -> int:
        """"(r, c)" / "(i, j, k)" -> C-order flat cell index; '' -> -1 (pass)."""
        if len(action) == 0:
            return -1
        idx = tuple(int(x) for x in action.strip("()").split(","))
        if len(idx) != len(self._shape) or any(not 0 <= i < d for i, d in zip(idx, self._shape)):
            raise ValueError("bad Tic Tac Toe action %r" % (action,))
        return int(np.ravel_multi_index(idx, self._shape))

    # The step kernel already produces everything the NEXT calls need (the packed state and its valid-action mask), so
    # the adapter remembers them for the state object it returns: `valid_actions(state)` on it costs no GPU work and
    # `next_state(state, ...)` no re-pack -- one host round trip per game step (H2D action, step kernel, one D2H) instead
    # of four.  The memo is checked by CONTENT (board bytes, winner, mover), so a caller that edits a state still gets
    # the right answer (it just pays for the pack again).
    _memo = None

    def _lookup(self, state, mover: int):
        m = self._memo
        if m is not None and m[2] == mover and m[1] == state[1] and m[0] == np.asarray(state[0], np.int8).tobytes():
            return m
        return None

    def _packed(self, state, mover: int):
        m = self._lookup(state, mover)
        return m[3] if m is not None else self._pack(state, mover)

    def next_state(self, state, players: List[int], actions: List[str]):
        mover, n = int(players[0]), self.max_players
        new = self._b.step_(self._packed(state, mover), torch.tensor([self._index(actions[0])], dtype=torch.int8))
        # ONE device -> host read: packed state (16 B) | result record (4 B) | valid-after mask (4 B)
        raw = torch.cat([new.packed.view(torch.uint8).reshape(-1), new.result.reshape(-1),
                         new.valid.view(torch.uint8).reshape(-1)]).cpu().numpy()
        words, r, mask = raw[:16].view(np.uint32), raw[16:20], int(raw[20:24].view(np.uint32)[0])
        nmover, w1 = int(words[0] >> 27) & 3, int(words[0] >> 29)
        board = np.full(int(np.prod(self._shape)), -1, np.int8)
        for p in range(n):                         # mover-relative layout (csrc/ttt.cuh): word j = player (mover + j) % n
            cells = int(words[(p - nmover) % n]) & 0x07ffffff
            while cells:
                c = (cells & -cells).bit_length() - 1
                board[c] = p
                cells &= cells - 1
        w = None if w1 == 0 else w1 - 1
        out = (board.reshape(self._shape), w)
        self._memo = (board.tobytes(), w, nmover, new, mask)
        terminal = bool(r[1] & 1)
        return out, [(mover + 1) % n], [int(np.int8(r[0]))], terminal, ([w] if w is not None else None)

    def valid_actions(self, state, player: int) -> List[str]:
        m = self._lookup(state, int(player))
        mask = m[4] if m is not None else int(self._b.valid_actions(self._pack(state, player))[0])
        cells = [c for c in range(int(np.prod(self._shape))) if mask >> c & 1]
        if not cells:
            return [""]
        return [str(tuple(int(i) for i in np.unravel_index(c, self._shape))) for c in cells]

    def is_valid_action(self, state, player: int, action: str) -> bool:
        if len(action) == 0:                   # '' is not a valid action here either (BlokusEnvironment.py:702,
            return False                       # tictactoe_2p_env.py:372); match_server special-cases it itself
        try:
            c = self._index(action)
        except ValueError:
            return False
        return bool(int(self._b.valid_actions(self._pack(state, player))[0]) >> c & 1)

    def state_to_observation(self, state, player: int) -> Dict[str, np.ndarray]:
        o = self._b.state_to_observation(self._pack(state, player), player)
        return {"board": self._np(o["board"][0]).reshape(self._shape)}


class TicTacToe2PlayerEnv(_TicTacToe):
    _batched_class = BatchedTicTacToe2PlayerEnv
    _shape = (3, 3)


class TicTacToe3PlayerEnv(_TicTacToe):
    _batched_class = BatchedTicTacToe3PlayerEnv
    _shape = (3, 5)


class TicTacToe4PlayerEnv(_TicTacToe):
    _batched_class = BatchedTicTacToe4PlayerEnv
    _shape = (3, 3, 3)


# name -> class, the names of colosseumrl/config.py:37-44
ENVIRONMENT_CLASSES = {"blokus": BlokusEnvironment, "tron": TronGridEnvironment, "tictactoe": TicTacToe2PlayerEnv,
                       "tictactoe_3p": TicTacToe3PlayerEnv, "tictactoe_4p": TicTacToe4PlayerEnv}


def get_environment(environment: str):
    return ENVIRONMENT_CLASSES[environment]
