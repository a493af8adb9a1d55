"""BatchedBlokusEnvironment: drop-in batched counterpart of BlokusEnvironment
(colosseumrl/envs/blokus/BlokusEnvironment.py), backed by csrc/blokus.cuh."""
from dataclasses import dataclass
from typing import Dict, List, Optional, Tuple

import torch

from .base import BatchedBaseEnvironment
from . import _lib

PIECE_NAMES = ["monomino1", "domino1", "trominoe1", "trominoe2", "tetrominoes1", "tetrominoes2", "tetrominoes3",
               "tetrominoes4", "tetrominoes5"] + ["pentominoe%d" % i for i in range(1, 13)]   # board.py:24-44
ORIENTATIONS = ["north", "northeast", "east", "southeast", "south", "southwest", "west", "northwest"]  # board.py:47


def action_to_string(action_id: int) -> str:
    """Engine action id -> the reference's action string (BlokusEnvironment.py:55-80); -1 -> ''."""
    if action_id < 0:
        return ""
    k, o, cell, piece = action_id % 5, (action_id // 5) % 8, (action_id // 40) % 400, action_id // 16000
    return "{};{};{}".format(PIECE_NAMES[piece], (cell % 20, cell // 20), ORIENTATIONS[o] + str(k))


def string_to_action(action_str: str) -> int:
    """The reference's action string (BlokusEnvironment.py:83-106) -> engine action id; '' -> -1."""
    if action_str == "":
        return -1
    piece, index, orientation = action_str.split(";")
    x, y = (int(v) for v in index.replace("(", "").replace(")", "").split(","))
    return ((PIECE_NAMES.index(piece) * 400 + y * 20 + x) * 8 + ORIENTATIONS.index(orientation[:-1])) * 5 + int(orientation[-1])


def _rotate_action_ids(ids, player, inverse: bool):
    """Action ids between the board frame and a player's rotated observation frame (np.rot90(k=-player),
    BlokusEnvironment.py:31-32): index -> M[player] @ (index - 9.5) + 9.5, orientation +- 2 * player, shift unchanged
    (:553-628; matrices board.py:52-73).  Works on ints and on integer tensors / arrays; -1 (pass) stays -1."""
    k, o, cell, piece = ids % 5, (ids // 5) % 8, (ids // 40) % 400, ids // 16000
    x, y = cell % 20, cell // 20
    r = (-player if inverse else player) % 4
    if r == 1:
        x, y = 19 - y, x
    elif r == 2:
        x, y = 19 - x, 19 - y
    elif r == 3:
        x, y = y, 19 - x
    o = (o + (-2 * player if inverse else 2 * player)) % 8
    out = ((piece * 400 + y * 20 + x) * 8 + o) * 5 + k
    if isinstance(ids, int):
        return out if ids >= 0 else -1
    return out * (ids >= 0) - (ids < 0) * 1


def real_action_to_player_perspective(ids, player: int):
    """convert_real_action_to_player_perspective_action (BlokusEnvironment.py:553-588) on action ids."""
    return _rotate_action_ids(ids, int(player), False)


def player_perspective_action_to_real(ids, player: int):
    """convert_player_perspective_action_to_real_action (:591-628) on action ids."""
    return _rotate_action_ids(ids, int(player), True)


# ---- placements (include/colosseum_b200_placement.h) -----------------------------------------------------------------
# A placement is p = s * 400 + y * 20 + x: oriented shape s (0..90, the engine's shape order: by size, then piece, then
# first appearance in ORIENTATIONS order) with the top-left corner of its bounding box at (x, y); -1 is a pass.  It is
# legal for a player iff the player holds the piece of s, every cell is on the board and allowed, and a cell is one of
# the player's anchors (round 0: the corner) -- exactly the placements of the ids in valid_actions' list.  In a
# player's perspective frame (the frame of state_to_observation(state, player)) a placement is the rotated cell set.
NUM_SHAPES = 91
NUM_PLACEMENTS = NUM_SHAPES * 400
ILLEGAL_ACTION = 21 * 16000             # what an illegal placement converts to: flagged and applied as a pass by a step


def shape_tables() -> Dict[str, "np.ndarray"]:
    """The library's shape tables (crl_blokus_shape_table), read once: "piece" [91], "cells" [91, 5, 2] ((dx, dy), -1
    past the shape's size), "rotation" [91, 4] (the image in player q's frame) and "action_shape" [21, 40, 3]
    ((shape, dx, dy) per piece and orientation * 5 + shift; -1 for shifts past the piece's size)."""
    global _SHAPE_TABLES
    if _SHAPE_TABLES is None:
        import numpy as np
        t = {"piece": np.zeros(91, np.int32), "cells": np.zeros((91, 5, 2), np.int32),
             "rotation": np.zeros((91, 4), np.int32), "action_shape": np.zeros((21, 40, 3), np.int32)}
        n = _lib.load().crl_blokus_shape_table(*(t[k].ctypes.data for k in ("piece", "cells", "rotation", "action_shape")))
        assert n == NUM_SHAPES
        # id -> placement of the id's own frame, over all 336 000 ids
        a = t["action_shape"]
        ids = np.arange(ILLEGAL_ACTION)
        ok, cell, piece = ids % 40, (ids // 40) % 400, ids // 16000
        s, dx, dy = a[piece, ok, 0], a[piece, ok, 1], a[piece, ok, 2]
        x, y = cell % 20 - dx, cell // 20 - dy
        t["id_placement"] = np.where((s >= 0) & (x >= 0) & (y >= 0), s * 400 + y * 20 + x, -1).astype(np.int32)
        _SHAPE_TABLES = t
    return _SHAPE_TABLES


_SHAPE_TABLES = None


def action_to_placement(ids, player: Optional[int] = None):
    """Action id -> placement, on ints, numpy arrays or integer tensors; -1 (pass) stays -1.  With `player`, the
    placement in that player's perspective frame: action_to_placement(id, r) == action_to_placement(
    real_action_to_player_perspective(id, r)).  Ids that no list can hold (a shift past the piece's size, a corner off
    the board) give -1 as well."""
    if player is not None:
        ids = real_action_to_player_perspective(ids, player)
    lut = shape_tables()["id_placement"]
    if isinstance(ids, int):
        return int(lut[ids]) if 0 <= ids < ILLEGAL_ACTION else -1
    if isinstance(ids, torch.Tensor):
        t = torch.as_tensor(lut, device=ids.device)
        inside = (ids >= 0) & (ids < ILLEGAL_ACTION)
        return torch.where(inside, t[ids.clamp(0, ILLEGAL_ACTION - 1).long()], torch.full_like(t[:1], -1)).to(ids.dtype)
    import numpy as np
    ids = np.asarray(ids)
    inside = (ids >= 0) & (ids < ILLEGAL_ACTION)
    return np.where(inside, lut[np.clip(ids, 0, ILLEGAL_ACTION - 1)], -1).astype(ids.dtype)


def placement_mask(words: torch.Tensor) -> torch.Tensor:
    """valid_placements' words int32 [B, 91, 20] -> bool [B, 36 400], entry p = s * 400 + y * 20 + x set iff placement
    p is legal: ready for logits.masked_fill(~mask, float("-inf"))."""
    bits = torch.arange(20, dtype=torch.int32, device=words.device)
    return ((words.unsqueeze(-1) >> bits) & 1).bool().reshape(words.shape[0], NUM_PLACEMENTS)


@dataclass
class BlokusBatchState:
    packed: torch.Tensor                        # int32 [B, 22, 4]: 352 bytes per game
    result: Optional[torch.Tensor] = None       # uint8 [B, 8] of the step that produced this state


class BatchedBlokusEnvironment(BatchedBaseEnvironment):
    def __init__(self, config: str = "", batch: int = 1, device="cuda:0", seed: int = 0, auto_reset: bool = False,
                 first_env_id: int = 0, capacity: int = 4096):
        super().__init__(config, batch, device, seed, auto_reset, first_env_id)
        self.capacity = int(capacity)      # slots per game in the valid-action list (longest list seen in 16 384 random
                                           # games x 70 steps: 2 104; counts > capacity signals a truncated list)

    @property
    def min_players(self) -> int:
        return 4

    @property
    def max_players(self) -> int:
        return 4

    @property
    def observation_shape(self) -> Dict[str, tuple]:
        return {"board": (20, 20), "pieces": (4, 21), "score": (4,), "player": (1,)}

    @staticmethod
    def observation_names() -> List[str]:
        return ["board", "pieces", "score", "player"]

    @staticmethod
    def all_piece_types() -> List[str]:
        return PIECE_NAMES

    @staticmethod
    def all_orientations() -> List[str]:
        return ORIENTATIONS

    def _alloc(self):
        return torch.empty((self.batch, 22, 4), dtype=torch.int32, device=self.device)

    def new_state(self, num_players: int = 4, out: Optional[BlokusBatchState] = None):
        assert num_players in (None, 4)
        packed = out.packed if out is not None else self._alloc()
        self._check(self._lib.crl_blokus_reset(packed.data_ptr(), None, self.batch, self._stream))
        return BlokusBatchState(packed), torch.ones((self.batch,), dtype=torch.uint8, device=self.device)

    def reset_where(self, state: BlokusBatchState, mask: torch.Tensor) -> BlokusBatchState:
        """new_state for the games with mask != 0 (in place)."""
        mask = self._dev(mask, torch.uint8)
        self._check(self._lib.crl_blokus_reset(state.packed.data_ptr(), mask.data_ptr(), self.batch, self._stream))
        state.result = None
        return state

    def valid_actions(self, state: BlokusBatchState, player: int = -1,
                      out: Optional[Tuple[torch.Tensor, torch.Tensor]] = None, count_stats: bool = True):
        """valid_actions (:453-500): (counts int32 [B], ids int32 [B, capacity]) in the reference's order;
        counts == 0 <=> [''].  player = -1: each game's current mover."""
        if out is None:
            out = (torch.empty((self.batch,), dtype=torch.int32, device=self.device),
                   torch.empty((self.batch, self.capacity), dtype=torch.int32, device=self.device))
        counts, ids = out
        self._check(self._lib.crl_blokus_legal(state.packed.data_ptr(), int(player), counts.data_ptr(), ids.data_ptr(),
                                               ids.shape[1], self._stats_ptr if count_stats else None, self.batch,
                                               self.flags, self._stream))
        return counts, ids

    def valid_placements(self, state: BlokusBatchState, player: int = -1, perspective: bool = False,
                         out: Optional[Tuple[torch.Tensor, torch.Tensor]] = None):
        """Legal placements of `player` (-1: each game's mover) as (counts int32 [B], words int32 [B, 91, 20]): bit x of
        words[g, s, y] is set iff placement s * 400 + y * 20 + x is legal (placement_mask unpacks it).  perspective:
        placements in the player's rotated frame (that of state_to_observation(state, player)).  One
        crl_blokus_placement_mask launch; no action list is built."""
        if out is None:
            out = (torch.empty((self.batch,), dtype=torch.int32, device=self.device),
                   torch.empty((self.batch, NUM_SHAPES, 20), dtype=torch.int32, device=self.device))
        counts, words = out
        self._check(self._lib.crl_blokus_placement_mask(state.packed.data_ptr(), int(player), int(bool(perspective)),
                                                        words.data_ptr(), counts.data_ptr(), self.batch, self.flags,
                                                        self._stream))
        return counts, words

    def placements_to_actions(self, state: BlokusBatchState, placements, player: int = -1,
                              perspective: bool = False) -> torch.Tensor:
        """Placements (int32 [B], -1 = pass; perspective: in the player's rotated frame) -> action ids int32 [B] in the
        board frame: the first id of the player's valid list with that placement, -1 for -1, ILLEGAL_ACTION for an
        illegal or out-of-range placement (a step flags it and applies a pass)."""
        placements = self._dev(placements, torch.int32)
        actions = torch.empty((self.batch,), dtype=torch.int32, device=self.device)
        self._check(self._lib.crl_blokus_placement_to_action(state.packed.data_ptr(), int(player), int(bool(perspective)),
                                                             placements.data_ptr(), actions.data_ptr(), self.batch,
                                                             self.flags, self._stream))
        return actions

    def is_valid_action(self, state: BlokusBatchState, player: int, action) -> torch.Tensor:
        """is_valid_action (:667-719): uint8 [B], 1 iff action[g] is in `player`'s valid list (-1 / '' is not).
        One crl_blokus_is_valid launch: the id is tested against the allowed / anchor boards, no list is built."""
        action = self._dev(action, torch.int32)
        valid = torch.empty((self.batch,), dtype=torch.uint8, device=self.device)
        self._check(self._lib.crl_blokus_is_valid(state.packed.data_ptr(), -1 if player is None else int(player),
                                                  action.data_ptr(), valid.data_ptr(), self.batch, self.flags,
                                                  self._stream))
        return valid

    def player_perspective_valid_actions(self, state: BlokusBatchState, player: int):
        """player_perspective_valid_actions (:502-551): the valid list of `player`, same order, every id rotated into
        that player's observation frame.  (counts, ids) like valid_actions."""
        counts, ids = self.valid_actions(state, player, count_stats=False)
        return counts, real_action_to_player_perspective(ids, player)

    def next_state(self, state: BlokusBatchState, players, actions, out: Optional[BlokusBatchState] = None):
        """next_state (:357-451).  actions: int32 [B] action ids (-1 = pass).
        Returns (new_state, new_players mask, reward int8 [B] (mover's), terminal uint8 [B], winners mask uint8 [B])."""
        new = self.step_(state, actions, out)
        r = new.result
        # views of the record only (bytes 5 / 6 are the players mask and the terminal flag as plain bytes): no launches
        return new, r[:, 5], r[:, 0].view(torch.int8), r[:, 6], r[:, 2]

    def step_(self, state: BlokusBatchState, actions, out: Optional[BlokusBatchState] = None) -> BlokusBatchState:
        """The bare crl_blokus_step launch (out may be `state` itself: in place).  Outputs are in new.result."""
        actions = self._dev(actions, torch.int32)
        new = out if out is not None else BlokusBatchState(self._alloc())
        if new.result is None:
            new.result = self._new_result((self.batch, 8))
        self._check(self._lib.crl_blokus_step(state.packed.data_ptr(), new.packed.data_ptr(), actions.data_ptr(),
                                              new.result.data_ptr(), self._stats_ptr, self.batch, self.flags,
                                              self._stream))
        return new

    def host_stepper(self, state: BlokusBatchState, stream=None) -> "BlokusHostStepper":
        """Two graph launches per game step for a policy that runs on the host (see BlokusHostStepper)."""
        return BlokusHostStepper(self, state, stream=stream)

    def is_terminal(self, state: BlokusBatchState) -> torch.Tensor:
        return ((state.packed[:, 21, 1] >> 16) & 1).to(torch.uint8)

    def current_rewards(self, state: BlokusBatchState) -> torch.Tensor:
        """Scores per player (BlokusEnvironment.py:340-355): int32 [B, 4]."""
        s = state.packed[:, 21, 0]
        return torch.stack([(s >> (8 * p)) & 0xff for p in range(4)], dim=1)

    def state_to_observation(self, state: BlokusBatchState, player: int) -> Dict[str, torch.Tensor]:
        """state_to_observation (:721-768).  player = -1: absolute unpack; -2: every game from its mover's perspective."""
        B = self.batch
        board = torch.empty((B, 20, 20), dtype=torch.int8, device=self.device)
        pieces = torch.empty((B, 4, 21), dtype=torch.uint8, device=self.device)
        score = torch.empty((B, 4), dtype=torch.int32, device=self.device)
        meta = torch.empty((B, 4), dtype=torch.int32, device=self.device)
        self._check(self._lib.crl_blokus_observe(state.packed.data_ptr(), int(player), board.data_ptr(), pieces.data_ptr(),
                                                 score.data_ptr(), meta.data_ptr(), B, self._stream))
        obs = {"board": board, "pieces": pieces, "score": score,
               "player": meta[:, 1:2].clone() if player == -2 else
               torch.full((B, 1), int(player), dtype=torch.int32, device=self.device)}
        if player == -1:
            obs.update(round=meta[:, 0], mover=meta[:, 1], terminal=meta[:, 2], episode_steps=meta[:, 3])
        return obs

    def state_from_arrays(self, board, pieces, score, round_count, mover) -> BlokusBatchState:
        st = BlokusBatchState(self._alloc())
        meta = torch.zeros((self.batch, 4), dtype=torch.int32, device=self.device)
        meta[:, 0] = self._dev(round_count, torch.int32)
        meta[:, 1] = self._dev(mover, torch.int32)
        b, p, s = self._dev(board, torch.int8), self._dev(pieces, torch.uint8), self._dev(score, torch.int32)
        self._check(self._lib.crl_blokus_pack(st.packed.data_ptr(), b.data_ptr(), p.data_ptr(), s.data_ptr(),
                                              meta.data_ptr(), self.batch, self._stream))
        return st

    def rollout(self, state: BlokusBatchState, step0: int, K: int) -> BlokusBatchState:
        """K uniform-random-policy steps (steps step0 .. step0 + K - 1 of this env's seed and env ids) in one launch,
        state updated in place; the last step's record goes to state.result and the statistics to `stats`.  Finished
        games are always restarted, whatever `auto_reset` says.  Equal to K x valid_actions -> random_actions -> step_
        with auto-reset whenever every list fits `capacity`: the pick is drawn over the full list, which is never
        stored."""
        if state.result is None:
            state.result = self._new_result((self.batch, 8))
        self._check(self._lib.crl_blokus_rollout(state.packed.data_ptr(), state.result.data_ptr(), self._stats_ptr,
                                                 self.seed, self.first_env_id, int(step0), int(K), self.batch,
                                                 self._stream))
        return state

    def advance(self, state: BlokusBatchState, actions, seat: int, step: int) -> torch.Tensor:
        """One learner move against uniform random opponents, in place (crl_blokus_advance; the rule is stated in
        include/colosseum_b200_learner.h): the learner at `seat` plays `actions` (int32 [B] ids, -1 = pass; None: it
        does not move), then the other seats play until `seat` is to move again, restarting finished games.  Returns
        the record uint8 [B, 8]: int8 learner reward (its index in the stable ascending sort of the final scores) |
        flags (1 a game finished, 2 illegal, 4 placed, 8 the learner did not move) | winners mask | opponent moves |
        the finished game's scores of seats 0..3."""
        a = None if actions is None else self._dev(actions, torch.int32)
        rec = self._new_result((self.batch, 8))
        self._check(self._lib.crl_blokus_advance(state.packed.data_ptr(), None if a is None else a.data_ptr(), int(seat),
                                                 rec.data_ptr(), self._stats_ptr, self.seed, self.first_env_id, int(step),
                                                 self.batch, self._stream))
        state.result = None
        return rec

    def random_actions(self, valid, step: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        counts, ids = valid
        out = out if out is not None else torch.empty((self.batch,), dtype=torch.int32, device=self.device)
        self._check(self._lib.crl_blokus_policy_random(counts.data_ptr(), ids.data_ptr(), ids.shape[1], out.data_ptr(),
                                                       self.seed, self.first_env_id, int(step), self.batch, self._stream))
        return out


class BlokusHostStepper:
    """A Blokus batch driven by a policy that runs on the HOST, in two CUDA-graph launches per game step:

      A  `launch_legal()`:  crl_blokus_legal (the movers' ordered valid lists stay on the device) -> D2H of the list
                            LENGTHS into `counts_np` (pinned int32 [B])
      B  `launch_step()`:   H2D of `choice_np` (pinned int32 [B]: index into each game's valid list, negative = pass)
                            -> crl_blokus_pick -> crl_blokus_step (in place on `state`) -> D2H of the result records
                            into `result_np` (pinned uint8 [B, 8])

        stepper = env.host_stepper(state)
        counts = stepper.legal()                     # launch A + wait
        stepper.choice_np[...] = my_policy(counts)   # e.g. a random index < counts
        records = stepper.step()                     # launch B + wait
    The kilobytes of action ids per game never cross PCIe; an actor serving several batches pipelines them
    (`launch_legal` / `wait_legal` / `launch_step` / `wait_step`), one stream per stepper.  `ids_device` is the
    device-side list for policies that want to look at the ids themselves."""

    def __init__(self, env, state, stream=None):
        from . import _cudart
        self.env, self.state = env, state
        B, dev = env.batch, env.device
        with torch.cuda.device(dev):
            s = stream if stream is not None else torch.cuda.current_stream(dev)
            self.counts = torch.zeros((B,), dtype=torch.int32).pin_memory()
            self.choice = torch.zeros((B,), dtype=torch.int32).pin_memory()
            self.result = torch.zeros((B, 8), dtype=torch.uint8).pin_memory()
            self.counts_np, self.choice_np, self.result_np = self.counts.numpy(), self.choice.numpy(), self.result.numpy()
            self._counts_dev = torch.zeros((B,), dtype=torch.int32, device=dev)
            self.ids_device = torch.zeros((B, env.capacity), dtype=torch.int32, device=dev)
            self._choice_dev = torch.zeros((B,), dtype=torch.int32, device=dev)
            self._action_dev = torch.zeros((B,), dtype=torch.int32, device=dev)
            self._result_dev = torch.zeros((B, 8), dtype=torch.uint8, device=dev)

            def phase_a():
                env.valid_actions(state, -1, out=(self._counts_dev, self.ids_device))
                self.counts.copy_(self._counts_dev, non_blocking=True)

            def phase_b():
                self._choice_dev.copy_(self.choice, non_blocking=True)
                env._check(env._lib.crl_blokus_pick(self._counts_dev.data_ptr(), self.ids_device.data_ptr(), env.capacity,
                                                    self._choice_dev.data_ptr(), self._action_dev.data_ptr(), B, env._stream))
                env._check(env._lib.crl_blokus_step(state.packed.data_ptr(), state.packed.data_ptr(), self._action_dev.data_ptr(),
                                                    self._result_dev.data_ptr(), env._stats_ptr, B, env.flags, env._stream))
                state.result = None
                self.result.copy_(self._result_dev, non_blocking=True)

            with torch.cuda.stream(s):
                phase_a()                                        # warm the launch paths (the state is not stepped:
            torch.cuda.synchronize(dev)                          # phase B is only captured, never run eagerly)
            self._graphs = []
            for fn in (phase_a, phase_b):
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    fn()
                self._graphs.append(g)
            raw = _lib.load()
            self._launch_fn, self._wait_fn = raw.crl_host_graph_launch, raw.crl_host_event_wait
            self._exec = [g.raw_cuda_graph_exec() for g in self._graphs]
            self._done = [_cudart.new_event(), _cudart.new_event()]
            self._stream_handle = s.cuda_stream
            for e in self._exec:
                _cudart.check(_cudart.rt().cudaGraphUpload(e, self._stream_handle), "cudaGraphUpload")

    def _launch(self, i):
        rc = self._launch_fn(self._exec[i], self._stream_handle, self._done[i])
        if rc == _lib.ERR_ARG:                                   # wrong current device: retry under a guard
            with torch.cuda.device(self.env.device):
                rc = self._launch_fn(self._exec[i], self._stream_handle, self._done[i])
        if rc:
            raise RuntimeError("BlokusHostStepper launch failed: %s" % _lib.load().crl_last_error().decode())

    def _wait(self, i):
        if self._wait_fn(self._done[i]):
            raise RuntimeError("BlokusHostStepper wait failed: %s" % _lib.load().crl_last_error().decode())

    def launch_legal(self):
        self._launch(0)

    def wait_legal(self):
        self._wait(0)
        return self.counts_np

    def launch_step(self):
        self._launch(1)

    def wait_step(self):
        self._wait(1)
        return self.result_np

    def legal(self):
        self.launch_legal()
        return self.wait_legal()

    def step(self):
        self.launch_step()
        return self.wait_step()
