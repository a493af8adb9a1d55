"""Vectorised reset / step wrapper: the batched analogue of the reference's RLlib adapter
(colosseumrl/envs/wrappers/rllib.py:8-55, envs/tron/rllib.py:13-66), which drives ONE game per Python object through
new_state -> state_to_observation and next_state -> state_to_observation -> reward / done dicts.  Here one object
steps B games per call and the per-agent dicts become tensors:

    venv = VectorEnv(BatchedTronGridEnvironment("", batch=4096, auto_reset=True))
    obs = venv.reset()                       # {"board": [B, P, N, N], "heads": [B, P, P], ...}
    obs, rewards, dones, info = venv.step(actions)     # rewards [B, P], dones uint8 [B]

Simultaneous-move games (Tron) are observed from every seat; turn-based games (Blokus, Tic Tac Toe) from the seat of
each game's next mover (`info["mover"]`).  `dones` marks the step that ended an episode.  With auto_reset=True a
finished game is restarted INSIDE that step() call (gym's vector-env convention): the observation, `info["mover"]` and
`valid_actions()` returned next all describe the fresh game the next action will be applied to, never the finished
board; `step(..., final_observation=True)` additionally returns the finished games' last observation in
`info["final_observation"]`.
"""
from typing import Dict

import torch


class VectorEnv:
    def __init__(self, env):
        self.env = env
        self.state = None
        self.simultaneous = hasattr(env, "remove_on_death")          # Tron: all live players act every step

    @property
    def num_envs(self) -> int:
        return self.env.batch

    @property
    def num_players(self) -> int:
        return self.env.max_players

    def _observe(self) -> Dict[str, torch.Tensor]:
        if self.simultaneous:
            return self.env.state_to_observation(self.state, -3)      # CRL_PLAYER_ALL: every seat in one launch
        return self.env.state_to_observation(self.state, -2)          # CRL_PLAYER_MOVER

    def reset(self) -> Dict[str, torch.Tensor]:
        self.state, _ = self.env.new_state()
        return self._observe()

    def valid_actions(self):
        """Valid actions of every game's acting player(s), in the batched environment's own format."""
        return self.env.valid_actions(self.state, -1)

    def step(self, actions, final_observation: bool = False):
        """actions: the batched environment's action tensor (Tron int8 [B, 4]; Blokus int32 [B] ids; TTT int8 [B])."""
        new, players, rewards, terminal, winners = self.env.next_state(self.state, None, actions, out=self.state)
        self.state = new
        info = {"players": players, "winners": winners}
        if self.env.auto_reset:
            if final_observation:
                info["final_observation"] = self._observe()
            # restart the finished games now, so that what the agent sees next is what its next action applies to
            self.env.reset_where(self.state, terminal)
            fresh = terminal != 0
            first = (1 << self.num_players) - 1 if self.simultaneous else 1          # new_state's acting players
            players = torch.where(fresh, torch.full_like(players, first), players)
            info["players"] = players
        if not self.simultaneous:                                     # players = 1 << next mover
            info["mover"] = (players >> 1) - (players >> 3)           # 1, 2, 4, 8 -> 0, 1, 2, 3
        return self._observe(), rewards, terminal, info


class SingleAgentVectorEnv:
    """One learner against avoid-policy opponents on the device: the batched analogue of the reference's single-player
    Tron trainer (TronRaySinglePlayerEnvironment, envs/tron/rllib.py:119-150, whose opponents are SimpleAvoidAgent,
    :69-96).  Every other seat plays the avoid policy of BatchedTronGridEnvironment.avoid_actions, so a step is two
    launches (policy, step) plus the observation, and no game leaves the device:

        venv = SingleAgentVectorEnv(BatchedTronGridEnvironment("", batch=4096), seat=0, noise=0.0)
        obs = venv.reset()                           # the learner's view: {"board": [B, N, N], "heads": [B, P], ...}
        obs, reward, done, info = venv.step(actions)  # actions int8 [B]; reward int8 [B]; done uint8 [B]

    End of an episode (this engine's choice: the reference's exact single-player semantics are not available to check
    against): `done` is set when the game is terminal OR the learner has died, since the learner's episode is over as
    soon as it can no longer act.  Such games are restarted inside that step() call, as VectorEnv does with auto_reset,
    so the observation returned is already the fresh game.  The opponents' Philox step is a counter kept here (reset()
    sets it to 0); restarted games use the spawns of the environment's last new_state()."""

    def __init__(self, env, seat: int = 0, noise: float = 0.0):
        if not hasattr(env, "avoid_actions"):
            raise TypeError("SingleAgentVectorEnv needs a Tron environment (BatchedTronGridEnvironment)")
        if not 0 <= seat < env.num_players:
            raise ValueError("seat must be in [0, %d)" % env.num_players)
        self.env, self.seat, self.noise = env, int(seat), float(noise)
        self.opponents = [p for p in range(env.num_players) if p != self.seat]
        self.state, self.t = None, 0
        self._actions = torch.zeros((env.batch, env.action_stride), dtype=torch.int8, device=env.device)

    @property
    def num_envs(self) -> int:
        return self.env.batch

    def _observe(self) -> Dict[str, torch.Tensor]:
        return self.env.state_to_observation(self.state, self.seat)

    def reset(self) -> Dict[str, torch.Tensor]:
        self.state, _ = self.env.new_state()
        self.t = 0
        return self._observe()

    def step(self, actions):
        """actions: int8 [B], the learner's.  Returns (the learner's observation, its reward int8 [B], done uint8 [B],
        info = {"players": alive mask, "winners": winners mask, "terminal": uint8 [B]} of the step just taken)."""
        self._actions[:, self.seat] = self.env._dev(actions, torch.int8)
        self.env.avoid_actions(self.state, self.t, seats=self.opponents, noise=self.noise, out=self._actions)
        self.t += 1
        new, players, rewards, terminal, winners = self.env.next_state(self.state, None, self._actions, out=self.state)
        self.state = new
        reward = rewards[:, self.seat].clone()
        learner_dead = ((players >> self.seat) & 1) == 0
        done = (terminal.bool() | learner_dead).to(torch.uint8)
        info = {"players": players.clone(), "winners": winners.clone(), "terminal": terminal.clone()}
        self.env.reset_where(self.state, done)
        return self._observe(), reward, done, info


class SingleAgentTurnVectorEnv:
    """One learner seat against uniform random opponents on the device, for the turn-based games (Tic Tac Toe, Blokus).
    Each step is ONE advance launch (the learner's move, then every opponent move up to the learner's next turn, with
    finished games restarted) plus the observation:

        venv = SingleAgentTurnVectorEnv(BatchedBlokusEnvironment(batch=1024), seat=1, perspective=True)
        obs = venv.reset()                           # the seat's view (Blokus: rotated for the seat)
        counts, ids = venv.valid_actions()           # Blokus: the seat's lists (perspective: in the rotated frame)
        obs, reward, done, info = venv.step(actions)  # reward int8 [B]; done uint8 [B]

    With action_space="placement" (Blokus only) the learner acts on the fixed space of 36 400 placements
    (colosseumrl_b200.blokus: p = shape * 400 + y * 20 + x) instead of the ragged id lists:

        venv = SingleAgentTurnVectorEnv(BatchedBlokusEnvironment(batch=1024), seat=1, perspective=True,
                                        action_space="placement")
        counts, mask = venv.valid_actions()          # bool [B, 36 400], in the seat's frame
        logits = logits.masked_fill(~mask, float("-inf"))
        obs, reward, done, info = venv.step(placements)   # int32 [B]; an illegal placement: info["illegal"], a pass

    The rule is this engine's definition (include/colosseum_b200_learner.h).  Every returned game is the learner's
    turn; `done` marks the step in which a game finished, and that game has already been restarted (and played up to
    the learner's turn), so the observation describes the game the next action applies to.  reward: Tic Tac Toe +1 /
    -1 / 0 for a win / loss / draw of the learner, Blokus its index in the stable ascending sort of the final scores;
    0 while a game goes on.  info: "winners" (mask of the finished game), "opponent_moves", "illegal" and, for Blokus,
    "scores" (uint8 [B, 4], the finished game's).  The opponents' Philox step is a counter kept here (reset() sets it to
    0, and reset() itself is step 0)."""

    def __init__(self, env, seat: int = 0, perspective: bool = False, action_space: str = "id"):
        if not hasattr(env, "advance"):
            raise TypeError("SingleAgentTurnVectorEnv needs a Tic Tac Toe or Blokus environment")
        if not 0 <= seat < env.max_players:
            raise ValueError("seat must be in [0, %d)" % env.max_players)
        self.blokus = hasattr(env, "player_perspective_valid_actions")
        if perspective and not self.blokus:
            raise ValueError("perspective=True exists for Blokus only")
        if action_space not in ("id", "placement"):
            raise ValueError('action_space must be "id" or "placement"')
        if action_space == "placement" and not self.blokus:
            raise ValueError('action_space="placement" exists for Blokus only')
        self.env, self.seat, self.perspective = env, int(seat), bool(perspective)
        self.action_space = action_space
        self.state, self.t = None, 0

    @property
    def num_envs(self) -> int:
        return self.env.batch

    def _observe(self) -> Dict[str, torch.Tensor]:
        return self.env.state_to_observation(self.state, self.seat)

    def reset(self) -> Dict[str, torch.Tensor]:
        self.state, _ = self.env.new_state()
        self.env.advance(self.state, None, self.seat, 0)
        self.t = 1
        return self._observe()

    def valid_actions(self):
        """Tic Tac Toe: the empty-cell mask int32 [B]; Blokus: (counts, ids) of the seat (perspective=True: rotated), or
        with action_space="placement" (counts, bool mask [B, 36 400]) of its legal placements.  Fresh tensors: the next
        step() does not change them."""
        if self.action_space == "placement":
            from .blokus import placement_mask
            counts, words = self.env.valid_placements(self.state, self.seat, self.perspective)
            return counts, placement_mask(words)
        if not self.blokus:
            return self.env.valid_actions(self.state).clone()     # (the cached mask is rewritten by the next advance)
        if self.perspective:
            return self.env.player_perspective_valid_actions(self.state, self.seat)
        return self.env.valid_actions(self.state, self.seat, count_stats=False)

    def step(self, actions):
        """actions: the learner's, int8 [B] cells (Tic Tac Toe) or int32 [B] ids (Blokus; perspective=True: in the
        seat's rotated frame), or int32 [B] placements with action_space="placement" (one conversion launch to the
        canonical ids; an illegal placement is reported in info["illegal"] and played as a pass).  Returns
        (observation, reward int8 [B], done uint8 [B], info)."""
        if self.action_space == "placement":
            actions = self.env.placements_to_actions(self.state, actions, self.seat, self.perspective)
        elif self.perspective:
            from .blokus import player_perspective_action_to_real
            actions = player_perspective_action_to_real(self.env._dev(actions, torch.int32), self.seat)
        rec = self.env.advance(self.state, actions, self.seat, self.t)
        self.t += 1
        info = {"winners": rec[:, 2], "opponent_moves": rec[:, 3], "illegal": (rec[:, 1] >> 1) & 1}
        if self.blokus:
            info["scores"] = rec[:, 4:8]
        return self._observe(), rec[:, 0].view(torch.int8), rec[:, 1] & 1, info
