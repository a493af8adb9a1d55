"""BatchedTronGridEnvironment: drop-in batched counterpart of the reference's TronGridEnvironment
(colosseumrl/envs/tron/TronGridEnvironment.py:61-508), backed by csrc/tron.cuh."""
from dataclasses import dataclass
from typing import Dict, List, Optional

import torch

from .base import BatchedBaseEnvironment
from . import _lib


def create_tron_config(*args) -> str:
    """Options -> config string "N;P;window;remove_on_death" (TronGridEnvironment.py:12-25)."""
    return ";".join(str(a) for a in args)


def parse_tron_config(config: str):
    """Same config string as the reference: "N;P;window;remove_on_death" (TronGridEnvironment.py:28-58)."""
    if len(config) == 0:
        return 19, 4, -1, False

    def parse(inp):
        try:
            return int(inp)
        except ValueError:
            return inp.lower() == "true"

    options = list(map(parse, config.split(";")))
    defaults = [None, 4, -1, False]
    while len(options) < 4:
        options.append(defaults[len(options)])
    return options


@dataclass
class TronBatchState:
    packed: torch.Tensor                    # int32 [13, B, 4]: SoA of 16-byte vectors, 208 B per environment: 9 owner-code
                                            # bit-plane vectors, 3 reserved (zero), the header at 12
    #                                         (shapes beyond N <= 19, P <= 4: int32 [W, B], csrc/tron_wide.cuh)
    result: Optional[torch.Tensor] = None   # uint8 [B, 8] (wide shapes: [B, 16]) written by the step that produced this state


class BatchedTronGridEnvironment(BatchedBaseEnvironment):
    # action codes == TronGridEnvironment.STRING_TO_ACTION (:62-67)
    STRING_TO_ACTION = {"": 0, "forward": 0, "right": 1, "left": -1}
    ACTIONS = ["forward", "right", "left"]

    def __init__(self, config: str = "", batch: int = 1, device="cuda:0", seed: int = 0, auto_reset: bool = False,
                 first_env_id: int = 0):
        super().__init__(config, batch, device, seed, auto_reset, first_env_id)
        self.N, self.num_players, self.observation_window, self.remove_on_death = parse_tron_config(config)
        if self._lib.crl_tron_state_bytes(self.N, self.num_players, self.batch) < 0:
            raise _lib.CrlError(self._lib.crl_last_error().decode())
        # buffer geometry of this shape: 4 actions / 8 result bytes per environment on the tuned path (N <= 19, P <= 4),
        # 8 / 16 on the wide path (include/colosseum_b200.h)
        self.action_stride = self._lib.crl_tron_action_stride(self.N, self.num_players)
        self.result_bytes = self._lib.crl_tron_result_bytes(self.N, self.num_players)
        self.wide = self.action_stride != 4
        # the spawns of the last new_state(): auto-reset inside the step restarts finished games from the same ones
        self._ring_offset, self._spawn_offsets = 1, None          # None = the reference's defaults (1, 2)

    @classmethod
    def create(cls, board_size: int = 19, num_players: int = 4, observation_window: int = -1,
               remove_on_death: bool = False, **kwargs) -> "BatchedTronGridEnvironment":
        """TronGridEnvironment.create (:69-90); kwargs: batch, device, seed, auto_reset, first_env_id."""
        return cls(create_tron_config(board_size, num_players, observation_window, remove_on_death), **kwargs)

    def __repr__(self):
        return ("BatchedTronGridEnvironment(size=%dx%d, players=%d, batch=%d, fully_observable=%s, remove_on_death=%s)"
                % (self.N, self.N, self.num_players, self.batch, self.observation_window < 0, self.remove_on_death))

    @property
    def min_players(self) -> int:
        return self.num_players

    @property
    def max_players(self) -> int:
        return self.num_players

    @staticmethod
    def observation_names() -> List[str]:
        return ["board", "heads", "directions", "deaths"]

    @property
    def observation_shape(self) -> Dict[str, tuple]:
        return {"board": (self.N, self.N), "heads": (self.num_players,), "directions": (self.num_players,),
                "deaths": (self.num_players,)}

    def _alloc(self):
        if self.wide:
            words = self._lib.crl_tron_state_bytes(self.N, self.num_players, 1) // 4
            return torch.empty((words, self.batch), dtype=torch.int32, device=self.device)
        return torch.empty((13, self.batch, 4), dtype=torch.int32, device=self.device)

    def _spawn_array(self, spawn_offset):
        """spawn_offset as new_state takes it -> one int per player: an int is used for every player; a (lo, hi) tuple
        draws np.random.randint(lo, hi) once PER PLAYER like the reference (:222-224); a list gives them explicitly."""
        import ctypes as C
        import numpy as np
        P = self.num_players
        if isinstance(spawn_offset, (int, np.integer)):
            offs = [int(spawn_offset)] * P
        elif isinstance(spawn_offset, tuple) and len(spawn_offset) == 2:
            offs = [int(np.random.randint(*spawn_offset)) for _ in range(P)]
        else:
            offs = [int(o) for o in spawn_offset]
            if len(offs) != P:
                raise ValueError("spawn_offset list must have one entry per player")
        return (C.c_int32 * P)(*offs)

    def new_state(self, num_players: int = None, ring_offset: int = 1, spawn_offset=2,
                  out: Optional[TronBatchState] = None):
        """TronGridEnvironment.new_state (:228-263) for every environment of the batch.  ring_offset / spawn_offset as
        in the reference (generate_start_positions :183-226): an int shifts every player's spawn, a (lo, hi) tuple
        draws one offset PER PLAYER (np.random.randint(lo, hi), :222-224; the draw is taken on the host and shared by
        the batch), a list of P ints sets them explicitly.  The environment remembers the spawns: auto-reset restarts
        finished games from them."""
        assert num_players is None or num_players == self.num_players, \
            "Do not change the number of players from the game configuration."
        so = self._spawn_array(spawn_offset)
        packed = out.packed if out is not None else self._alloc()
        self._check(self._lib.crl_tron_reset_spawns(packed.data_ptr(), None, self.batch, self.N, self.num_players,
                                                    int(ring_offset), so, self._stream))
        default = int(ring_offset) == 1 and all(o == 2 for o in so)
        self._ring_offset, self._spawn_offsets = int(ring_offset), (None if default else so)
        players = torch.full((self.batch,), (1 << self.num_players) - 1, dtype=torch.uint8, device=self.device)
        return TronBatchState(packed), players

    def generate_start_positions(self, ring_offset: int = 1, spawn_offset=0):
        """generate_start_positions (:183-226): (heads = y * N + x, directions) as int64 numpy arrays."""
        import ctypes as C
        import numpy as np
        h, d = (C.c_int32 * 8)(), (C.c_int32 * 8)()
        self._check(self._lib.crl_tron_start_positions_spawns(self.N, self.num_players, int(ring_offset),
                                                              self._spawn_array(spawn_offset), h, d))
        return (np.array(h[:self.num_players], np.int64), np.array(d[:self.num_players], np.int64))

    def reset_where(self, state: TronBatchState, mask: torch.Tensor):
        mask = self._dev(mask, torch.uint8)
        if self._spawn_offsets is None:
            self._check(self._lib.crl_tron_reset(state.packed.data_ptr(), mask.data_ptr(), self.batch, self.N,
                                                 self.num_players, self._stream))
        else:
            self._check(self._lib.crl_tron_reset_spawns(state.packed.data_ptr(), mask.data_ptr(), self.batch, self.N,
                                                        self.num_players, self._ring_offset, self._spawn_offsets,
                                                        self._stream))
        state.result = None                     # the record of the step before the reset no longer describes `state`
        return state

    def _step_call(self, src, dst, actions_ptr, result_ptr, flags):
        """crl_tron_step, or crl_tron_step_spawns when new_state() was given non-default spawns (auto-reset uses them)."""
        if self._spawn_offsets is None:
            return self._lib.crl_tron_step(src, dst, actions_ptr, result_ptr, self._stats_ptr, self.batch, self.N,
                                           self.num_players, flags, self._stream)
        return self._lib.crl_tron_step_spawns(src, dst, actions_ptr, result_ptr, self._stats_ptr, self.batch, self.N,
                                              self.num_players, flags, self._ring_offset, self._spawn_offsets,
                                              self._stream)

    def next_state(self, state: TronBatchState, players, actions, out: Optional[TronBatchState] = None):
        """TronGridEnvironment.next_state (:265-323).  actions: int8 [B, 4] ([B, 8] for shapes beyond N <= 19, P <= 4:
        `self.action_stride`) (0 forward, 1 right, -1 left; entries of dead / absent players ignored).  `players` is accepted for signature parity and ignored (dense action tensor).
        Returns (new_state, new_players mask, rewards int8 [B, P], terminal uint8 [B], winners mask uint8 [B])."""
        new = self.step_(state, actions, out)
        r = new.result
        if self.wide:                           # 16-byte record: reward[8] | terminal | alive | winners | 0 | ranking u32
            return new, r[:, 9], r[:, :self.num_players].view(torch.int8), r[:, 8], r[:, 10]
        return new, r[:, 5], r[:, :self.num_players].view(torch.int8), r[:, 4], r[:, 6]

    def step_(self, state: TronBatchState, actions, out: Optional[TronBatchState] = None) -> TronBatchState:
        """The bare crl_tron_step launch (out may be `state` itself: in place).  Outputs are in new.result."""
        actions = self._dev(actions, torch.int8)
        if actions.shape != (self.batch, self.action_stride):
            raise ValueError("actions must have shape [B, %d]" % self.action_stride)
        new = out if out is not None else TronBatchState(self._alloc())
        if new.result is None:
            new.result = self._new_result((self.batch, self.result_bytes))
        self._check(self._step_call(state.packed.data_ptr(), new.packed.data_ptr(), actions.data_ptr(),
                                    new.result.data_ptr(), self.flags))
        return new

    def host_stepper(self, state: TronBatchState, stream=None, compact=False, packed_actions: bool = False,
                     zero_copy: bool = False):
        """Graph-fused H2D actions -> step -> D2H result for host-side policies (see base.HostStepper).
        compact=True: the step writes the 4-byte record (CRL_FLAG_COMPACT_RESULT: terminal | alive | winners | ranking),
        which halves the PCIe read-back; compact=2: the 2-byte record (CRL_FLAG_COMPACT2_RESULT: alive | terminal << 4,
        ranking), a quarter -- the read-back is the slowest leg of a host-side actor's step.  `decode_compact`
        rebuilds the reference's return values from either on the host.
        packed_actions=True: the pinned action buffer is uint8 [B], 2 bits per player (`pack_actions`), a quarter of
        the PCIe upload.  zero_copy=True (with compact=2 and packed_actions): the step kernel reads the pinned action
        buffer and writes the pinned record buffer directly over PCIe -- one kernel node per step instead of memcpy +
        kernel + memcpy (base.HostStepper).  NOTE: the warm-up inside applies one step of all-forward actions to `state`."""
        from .base import HostStepper
        if self.wide and (compact or packed_actions):
            raise ValueError("compact records / packed actions exist for N <= 19, P <= 4 only")
        if not compact and not packed_actions:
            return HostStepper(self, state, (self.batch, self.action_stride), torch.int8, stream=stream)
        width = 2 if compact == 2 else (4 if compact else 8)
        flags = self.flags | {8: 0, 4: _lib.FLAG_COMPACT_RESULT, 2: _lib.FLAG_COMPACT2_RESULT}[width] | \
            (_lib.FLAG_PACKED_ACTIONS if packed_actions else 0)
        if zero_copy:
            if not (compact == 2 and packed_actions):
                raise ValueError("zero_copy needs compact=2 and packed_actions=True (narrow, coalesced PCIe accesses)")

            def zstep(host_actions, host_result):
                self._check(self._step_call(state.packed.data_ptr(), state.packed.data_ptr(), host_actions.data_ptr(),
                                            host_result.data_ptr(), flags))
                state.result = None
            return HostStepper(self, state, (self.batch,), torch.uint8, stream=stream, zero_copy_step=zstep,
                               result_shape=(self.batch, 2))
        rec = torch.empty((self.batch, width), dtype=torch.uint8, device=self.device)

        def step(dev_actions):
            self._check(self._step_call(state.packed.data_ptr(), state.packed.data_ptr(), dev_actions.data_ptr(),
                                        rec.data_ptr(), flags))
            state.result = None                 # the full record of an earlier step no longer describes `state`
            return rec
        if packed_actions:
            return HostStepper(self, state, (self.batch,), torch.uint8, stream=stream, step=step)
        return HostStepper(self, state, (self.batch, 4), torch.int8, stream=stream, step=step)

    @staticmethod
    def pack_actions(actions):
        """int8 [B, 4] actions (0 forward, 1 right, -1 left) -> uint8 [B], player p in bits 2p..2p+1 (numpy, host side)."""
        import numpy as np
        a = np.asarray(actions).astype(np.uint8) & 3
        return (a[:, 0] | a[:, 1] << 2 | a[:, 2] << 4 | a[:, 3] << 6).astype(np.uint8)

    def decode_compact(self, rec):
        """The reference's next_state return values from compact records (numpy uint8 [B, 4], e.g. HostStepper.wait()):
        (new_players mask [B], rewards int8 [B, P], terminal [B], winners mask [B], ranking [B, P]).
        rewards = -2 * (deaths > 0) + 1, winners of a terminal step + 9 (TronGridEnvironment.py:313-320)."""
        import numpy as np
        rec = np.asarray(rec)
        if rec.shape[1] == 2:                   # 2-byte record: winners of a terminal step = its alive players (:316-319)
            alive, terminal, rk = rec[:, 0] & 15, (rec[:, 0] >> 4) & 1, rec[:, 1]
            winners = alive * terminal
        else:
            terminal, alive, winners, rk = rec[:, 0], rec[:, 1], rec[:, 2], rec[:, 3]
        p = np.arange(self.num_players, dtype=np.uint8)[None, :]
        a = (alive[:, None] >> p) & 1
        w = ((winners[:, None] >> p) & 1) * (terminal[:, None] & 1)
        rewards = (2 * a.astype(np.int8) - 1 + 9 * w.astype(np.int8)).astype(np.int8)
        return alive, rewards, terminal, winners, ((rk[:, None] >> (2 * p)) & 3).astype(np.uint8)

    def valid_actions(self, state, player):
        """Always ['forward', 'right', 'left'] (:325-341): uint8 [B, 3] of ones."""
        return torch.ones((self.batch, 3), dtype=torch.uint8, device=self.device)

    def is_valid_action(self, state, player, action):
        return torch.ones((self.batch,), dtype=torch.uint8, device=self.device)

    def is_terminal(self, state: TronBatchState) -> torch.Tensor:
        if state.result is not None:
            return state.result[:, 8 if self.wide else 4]
        if self.wide:
            return (state.packed[-1] & 1).to(torch.uint8)
        return ((state.packed[12, :, 2] >> 27) & 1).to(torch.uint8)

    def compute_ranking(self, state: TronBatchState, players=None, winners=None) -> torch.Tensor:
        """TronGridEnvironment.compute_ranking (:483-508), fused into the step: uint8 [B, P]."""
        bits = 3 if self.wide else 2            # wide shapes: uint32 per environment, 3 bits per player
        if state.result is not None:
            rk = state.result[:, 12:16].contiguous().view(torch.int32)[:, 0] if self.wide else state.result[:, 7].to(torch.int32)
        else:                                   # a state that was not produced by a step (imported / fresh)
            rkb = torch.empty((self.batch,), dtype=torch.int32 if self.wide else torch.uint8, device=self.device)
            self._check(self._lib.crl_tron_ranking(state.packed.data_ptr(), rkb.data_ptr(), self.batch, self.N,
                                                   self.num_players, self._stream))
            rk = rkb.to(torch.int32)
        shifts = bits * torch.arange(self.num_players, device=self.device)
        return ((rk[:, None] >> shifts[None]) & ((1 << bits) - 1)).to(torch.uint8)

    def state_to_observation(self, state: TronBatchState, player: int) -> Dict[str, torch.Tensor]:
        """TronGridEnvironment.state_to_observation (:363-405); player = -1 gives the absolute (unrotated) state,
        player = -3 the views of ALL players in one pass: board [B, P, N, N], vectors [B, P, P]."""
        B, N, P = self.batch, self.N, self.num_players
        views = (P,) if player == -3 else ()
        board = torch.empty((B,) + views + (N, N), dtype=torch.int8, device=self.device)
        heads, dirs, deaths = (torch.empty((B,) + views + (P,), dtype=torch.int32, device=self.device) for _ in range(3))
        self._check(self._lib.crl_tron_observe(state.packed.data_ptr(), int(player), board.data_ptr(), heads.data_ptr(),
                                               dirs.data_ptr(), deaths.data_ptr(), None, B, N, P, self._stream))
        return {"board": board, "heads": heads, "directions": dirs, "deaths": deaths}

    def state_from_arrays(self, board, heads, directions, deaths) -> TronBatchState:
        """Import reference-layout arrays (board [B,N,N], heads = y*N+x, directions, deaths [B,P])."""
        st = TronBatchState(self._alloc())
        b, h = self._dev(board, torch.int8), self._dev(heads, torch.int32)
        d, de = self._dev(directions, torch.int32), self._dev(deaths, torch.int32)
        self._check(self._lib.crl_tron_pack(st.packed.data_ptr(), b.data_ptr(), h.data_ptr(), d.data_ptr(),
                                            de.data_ptr(), self.batch, self.N, self.num_players, self._stream))
        return st

    # -- random policy / fused rollouts (benchmark + self-play helpers) -------------------------------
    def random_actions(self, step: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        out = out if out is not None else torch.empty((self.batch, self.action_stride), dtype=torch.int8, device=self.device)
        fn = self._lib.crl_tron_policy_random_wide if self.wide else self._lib.crl_tron_policy_random
        self._check(fn(out.data_ptr(), self.seed, self.first_env_id, int(step), self.batch, self._stream))
        return out

    def _seat_mask(self, seats) -> int:
        """None = every seat; an int is a bit mask (bit p = seat p); otherwise an iterable of seat indices."""
        if seats is None:
            return (1 << self.num_players) - 1
        if isinstance(seats, int):
            return seats
        mask = 0
        for p in seats:
            mask |= 1 << int(p)
        return mask

    def avoid_actions(self, state: TronBatchState, step: int, seats=None, noise: float = 0.0,
                      out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """The avoid policy (include/colosseum_b200_tron_policy.h: forward if free, else a Philox coin picks the side
        tried first) for `seats` (None = all) on the device, decided on `state` before the step.  noise: the probability
        of a uniform random move instead.  Into `out` (int8 [B, action_stride]; new and zeroed if None): the other
        seats' entries are left as they are, so a learner's actions can be written there first.  The spawns of the last
        new_state() and this environment's auto_reset are used: with auto_reset, a finished game is decided on the
        fresh game the step will restart."""
        out = out if out is not None else torch.zeros((self.batch, self.action_stride), dtype=torch.int8,
                                                      device=self.device)
        if out.shape != (self.batch, self.action_stride) or out.dtype != torch.int8 or not out.is_contiguous():
            raise ValueError("out must be a contiguous int8 tensor of shape [B, %d]" % self.action_stride)
        self._check(self._lib.crl_tron_policy_avoid(
            state.packed.data_ptr(), out.data_ptr(), self._seat_mask(seats), int(round(noise * 65536)), self.seed,
            self.first_env_id, int(step), self.batch, self.N, self.num_players, self.flags & _lib.FLAG_AUTO_RESET,
            self._ring_offset, self._spawn_offsets, self._stream))
        return out

    def rollout(self, state: TronBatchState, step0: int, K: int, avoid_seats=0, noise: float = 0.0) -> TronBatchState:
        """K steps with auto-reset in one launch (state updated in place): every seat on the random policy, or with
        avoid_seats (a bit mask or a list of seats) those seats on the avoid policy (`avoid_actions`, with `noise`).  The
        random-only form restarts finished games from new_state's default spawns; the avoid form from the spawns of the
        last new_state()."""
        if state.result is None:
            state.result = self._new_result((self.batch, self.result_bytes))
        mask = self._seat_mask(avoid_seats)
        if mask == 0 and noise == 0.0:
            self._check(self._lib.crl_tron_rollout(state.packed.data_ptr(), state.result.data_ptr(), self._stats_ptr,
                                                   self.seed, self.first_env_id, int(step0), int(K), self.batch, self.N,
                                                   self.num_players, self._stream))
            return state
        self._check(self._lib.crl_tron_rollout_avoid(
            state.packed.data_ptr(), state.result.data_ptr(), self._stats_ptr, self.seed, self.first_env_id, int(step0),
            int(K), self.batch, self.N, self.num_players, mask, int(round(noise * 65536)), self._ring_offset,
            self._spawn_offsets, self._stream))
        return state
