"""Batched generalised Tic Tac Toe: drop-in batched counterparts of TicTacToe{2,3,4}PlayerEnv
(colosseumrl/envs/tictactoe/tictactoe_{2,3,4}p_env.py), backed by csrc/ttt.cuh."""
from dataclasses import dataclass
from typing import Dict, List, Optional

import torch

from .base import BatchedBaseEnvironment
from . import _lib

BOARD_SHAPE = {2: (3, 3), 3: (3, 5), 4: (3, 3, 3)}


@dataclass
class TTTBatchState:
    packed: torch.Tensor                       # int32 [B, 4]: one 16-byte vector per environment
    result: Optional[torch.Tensor] = None      # uint8 [B, 4] of the step that produced this state
    valid: Optional[torch.Tensor] = None       # int32 [B] empty-cell mask (valid actions of the next mover)


class _BatchedTicTacToe(BatchedBaseEnvironment):
    N_PLAYERS = 0

    @property
    def min_players(self) -> int:
        return self.N_PLAYERS

    @property
    def max_players(self) -> int:
        return self.N_PLAYERS

    @property
    def observation_shape(self) -> Dict[str, tuple]:
        return {"board": BOARD_SHAPE[self.N_PLAYERS]}

    @staticmethod
    def observation_names() -> List[str]:
        return ["board"]

    @property
    def cells(self) -> int:
        s = BOARD_SHAPE[self.N_PLAYERS]
        return s[0] * s[1] * (s[2] if len(s) > 2 else 1)

    def new_state(self, num_players: int = None, out: Optional[TTTBatchState] = None):
        assert num_players is None or num_players == self.N_PLAYERS
        packed = out.packed if out is not None else torch.empty((self.batch, 4), dtype=torch.int32, device=self.device)
        self._check(self._lib.crl_ttt_reset(packed.data_ptr(), None, self.batch, self.N_PLAYERS, self._stream))
        players = torch.ones((self.batch,), dtype=torch.uint8, device=self.device)      # player 0 moves first
        return TTTBatchState(packed), players

    def reset_where(self, state: TTTBatchState, mask: torch.Tensor) -> TTTBatchState:
        """new_state for the environments with mask != 0 (in place)."""
        mask = self._dev(mask, torch.uint8)
        self._check(self._lib.crl_ttt_reset(state.packed.data_ptr(), mask.data_ptr(), self.batch, self.N_PLAYERS, self._stream))
        state.valid = None                     # the cached empty-cell masks no longer describe the reset boards
        return state

    def next_state(self, state: TTTBatchState, players, actions, out: Optional[TTTBatchState] = None):
        """next_state (2p :240-315).  actions: int8 [B], C-order flat cell index, negative = '' (pass).
        Returns (new_state, new_players mask, reward int8 [B] (the mover's), terminal uint8 [B], winners mask uint8 [B])."""
        new = self.step_(state, actions, out)
        r = new.result
        mover = (new.packed[:, 0] >> 27) & 3
        return new, (1 << mover).to(torch.uint8), r[:, 0].view(torch.int8), r[:, 1] & 1, r[:, 2]

    def current_rewards(self, state: TTTBatchState) -> torch.Tensor:
        """current_rewards (tictactoe_2p_env.py:219-238): int8 [B, n], +1 winner / -1 the others once a game has a
        winner, 0 before."""
        w1 = (state.packed[:, 0] >> 29) & 7                                        # winner + 1, 0 = None
        seat = torch.arange(self.N_PLAYERS, device=self.device, dtype=torch.int32)[None]
        return torch.where(w1[:, None] == 0, 0, torch.where(seat + 1 == w1[:, None], 1, -1)).to(torch.int8)

    def step_(self, state: TTTBatchState, actions, out: Optional[TTTBatchState] = None) -> TTTBatchState:
        """The bare crl_ttt_step launch (out may be `state` itself: in place).  Outputs are in new.result / new.valid."""
        actions = self._dev(actions, torch.int8)
        new = out if out is not None else TTTBatchState(torch.empty_like(state.packed))
        if new.result is None:
            new.result = self._new_result((self.batch, 4))
        if new.valid is None:
            new.valid = torch.empty((self.batch,), dtype=torch.int32, device=self.device)
        self._check(self._lib.crl_ttt_step(state.packed.data_ptr(), new.packed.data_ptr(), actions.data_ptr(),
                                           new.result.data_ptr(), new.valid.data_ptr(), self._stats_ptr,
                                           self.batch, self.N_PLAYERS, self.flags, self._stream))
        return new

    def host_stepper(self, state: TTTBatchState, stream=None, compact: bool = False):
        """Graph-fused H2D actions -> step -> D2H result for host-side policies (see base.HostStepper).
        compact=True: the step writes the 1-byte record (CRL_FLAG_COMPACT_RESULT: flags | (winner + 1) << 3 | mover << 6),
        a quarter of the PCIe read-back; `decode_compact` rebuilds next_state's return values from it on the host.
        NOTE: the warm-up inside applies one step of cell-0 actions to `state`."""
        from .base import HostStepper
        if not compact:
            return HostStepper(self, state, (self.batch,), torch.int8, stream=stream)
        rec = torch.empty((self.batch, 1), dtype=torch.uint8, device=self.device)
        flags = self.flags | _lib.FLAG_COMPACT_RESULT

        def step(dev_actions):
            self._check(self._lib.crl_ttt_step(state.packed.data_ptr(), state.packed.data_ptr(), dev_actions.data_ptr(),
                                               rec.data_ptr(), None, self._stats_ptr, self.batch, self.N_PLAYERS, flags,
                                               self._stream))
            state.result = state.valid = None       # the records of an earlier step no longer describe `state`
            return rec
        return HostStepper(self, state, (self.batch,), torch.int8, stream=stream, step=step)

    def decode_compact(self, rec):
        """next_state's return values from 1-byte records (numpy uint8 [B, 1], e.g. HostStepper.wait()):
        (new_players mask [B], reward int8 [B] (the mover's), terminal [B], winners mask [B]).
        reward = +1 if the mover is the winner, -1 if somebody else is, else 0 (tictactoe_2p_env.py:302-308)."""
        import numpy as np
        r = np.asarray(rec).reshape(-1)
        terminal, w1, mover = r & 1, (r >> 3) & 7, r >> 6
        nxt = (mover + 1) % self.N_PLAYERS
        reward = np.where(w1 == 0, 0, np.where(w1 == mover + 1, 1, -1)).astype(np.int8)
        winners = np.where(w1 == 0, 0, 1 << np.maximum(w1.astype(np.int32) - 1, 0)).astype(np.uint8)
        return (1 << nxt).astype(np.uint8), reward, terminal.astype(np.uint8), winners

    def valid_actions(self, state: TTTBatchState, player=None) -> torch.Tensor:
        """valid_actions (2p :317-348) as a bit mask: int32 [B], bit c = cell c (C order) is empty; 0 <=> ['']."""
        if state.valid is not None:
            return state.valid
        mask = torch.empty((self.batch,), dtype=torch.int32, device=self.device)
        self._check(self._lib.crl_ttt_valid_actions(state.packed.data_ptr(), mask.data_ptr(), self.batch,
                                                    self.N_PLAYERS, self._stream))
        return mask

    def is_valid_action(self, state: TTTBatchState, player, action) -> torch.Tensor:
        action = self._dev(action, torch.int8).to(torch.int32)
        mask = self.valid_actions(state)
        return ((action >= 0) & (((mask >> action.clamp(min=0)) & 1) == 1) & (action < self.cells)).to(torch.uint8)

    def is_terminal(self, state: TTTBatchState) -> torch.Tensor:
        p = state.packed
        full = (p[:, 0] | p[:, 1] | p[:, 2] | p[:, 3]) & ((1 << self.cells) - 1)
        return ((((p[:, 0] >> 29) & 7) != 0) | (full == (1 << self.cells) - 1)).to(torch.uint8)

    def state_to_observation(self, state: TTTBatchState, player: int) -> Dict[str, torch.Tensor]:
        board = torch.empty((self.batch,) + BOARD_SHAPE[self.N_PLAYERS], dtype=torch.int8, device=self.device)
        self._check(self._lib.crl_ttt_observe(state.packed.data_ptr(), int(player), board.data_ptr(), None, None,
                                              self.batch, self.N_PLAYERS, self._stream))
        return {"board": board}

    def state_arrays(self, state: TTTBatchState):
        """(board int8 [B, ...], winner int8 [B] (-1 None), mover int8 [B])."""
        board = torch.empty((self.batch,) + BOARD_SHAPE[self.N_PLAYERS], dtype=torch.int8, device=self.device)
        winner = torch.empty((self.batch,), dtype=torch.int8, device=self.device)
        mover = torch.empty_like(winner)
        self._check(self._lib.crl_ttt_observe(state.packed.data_ptr(), -1, board.data_ptr(), winner.data_ptr(),
                                              mover.data_ptr(), self.batch, self.N_PLAYERS, self._stream))
        return board, winner, mover

    def state_from_arrays(self, board, winner, mover) -> TTTBatchState:
        st = TTTBatchState(torch.empty((self.batch, 4), dtype=torch.int32, device=self.device))
        b, w, m = self._dev(board, torch.int8), self._dev(winner, torch.int8), self._dev(mover, torch.int8)
        self._check(self._lib.crl_ttt_pack(st.packed.data_ptr(), b.data_ptr(), w.data_ptr(), m.data_ptr(), self.batch,
                                           self.N_PLAYERS, self._stream))
        return st

    def random_actions(self, state: TTTBatchState, step: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        out = out if out is not None else torch.empty((self.batch,), dtype=torch.int8, device=self.device)
        self._check(self._lib.crl_ttt_policy_random(state.packed.data_ptr(), out.data_ptr(), self.seed, self.first_env_id,
                                                    int(step), self.batch, self.N_PLAYERS, self.flags, self._stream))
        return out

    def rollout(self, state: TTTBatchState, step0: int, K: int) -> TTTBatchState:
        if state.result is None:
            state.result = self._new_result((self.batch, 4))
        state.valid = None
        self._check(self._lib.crl_ttt_rollout(state.packed.data_ptr(), state.result.data_ptr(), self._stats_ptr,
                                              self.seed, self.first_env_id, int(step0), int(K), self.batch,
                                              self.N_PLAYERS, self._stream))
        return state

    def advance(self, state: TTTBatchState, actions, seat: int, step: int) -> torch.Tensor:
        """One learner move against uniform random opponents, in place (crl_ttt_advance; the rule is stated in
        include/colosseum_b200_learner.h): the learner at `seat` plays `actions` (int8 [B] cells; None: it does not
        move), then the other seats play until `seat` is to move again, restarting finished games.  Returns the record
        uint8 [B, 4]: int8 learner reward | flags (1 a game finished, 2 illegal, 4 placed, 8 the learner did not move) |
        winners mask of the finished game | opponent moves.  state.valid becomes the learner's valid actions."""
        a = None if actions is None else self._dev(actions, torch.int8)
        if state.valid is None:
            state.valid = torch.empty((self.batch,), dtype=torch.int32, device=self.device)
        rec = self._new_result((self.batch, 4))
        self._check(self._lib.crl_ttt_advance(state.packed.data_ptr(), None if a is None else a.data_ptr(), int(seat),
                                              rec.data_ptr(), state.valid.data_ptr(), self._stats_ptr, self.seed,
                                              self.first_env_id, int(step), self.batch, self.N_PLAYERS, self._stream))
        state.result = None                    # the record of an earlier step no longer describes `state`
        return rec


class BatchedTicTacToe2PlayerEnv(_BatchedTicTacToe):
    N_PLAYERS = 2


class BatchedTicTacToe3PlayerEnv(_BatchedTicTacToe):
    N_PLAYERS = 3


class BatchedTicTacToe4PlayerEnv(_BatchedTicTacToe):
    N_PLAYERS = 4
