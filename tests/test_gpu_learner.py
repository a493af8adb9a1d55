"""GPU parity tests (B200): the single-learner advance of Tic Tac Toe and Blokus and SingleAgentTurnVectorEnv through
libcolosseum_b200.so, bit-exact against the C oracle tests/oracle_learner.c."""
import numpy as np
import pytest

import backends
import cases_learner as cases
from oracle import oracle as orc

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def be():
    return backends.Cuda()


@pytest.mark.parametrize("n", [2, 3, 4])
def test_ttt_calls(be, n):
    for seat in range(n):
        cases.case_ttt_calls(be, n, seat, B=5000, calls=30, seed=3 + seat)


def test_ttt_4p_full_size(be):
    # 1,048,576 environments x 48 calls, the seat that plays the most opponent moves
    ob, recs = cases.case_ttt_calls(be, 4, 3, B=1 << 20, calls=48, seed=0, env0=0, check_every=6)
    assert (recs[..., 3] == 6).any()


@pytest.mark.parametrize("n", [2, 3, 4])
def test_ttt_handbuilt(be, n):
    cases.case_ttt_handbuilt(be, n)


@pytest.mark.parametrize("n", [2, 3, 4])
def test_ttt_null_mode(be, n):
    cases.case_ttt_null_mode(be, n, B=3000)


@pytest.mark.parametrize("seat", [0, 1, 2, 3])
def test_blokus_calls(be, seat):
    cases.case_blokus_calls(be, seat, B=1024, calls=200, check_every=10)


def test_blokus_calls_4096(be):
    cases.case_blokus_calls(be, 3, B=4096, calls=70, seed=8, check_every=10)


def test_blokus_handbuilt(be):
    cases.case_blokus_handbuilt(be)


def test_blokus_null_mode(be):
    cases.case_blokus_null_mode(be, B=300)


def test_sharding(be):
    cases.case_sharding(be, "ttt", n=4, B=100000, calls=20)
    cases.case_sharding(be, "ttt", n=2, B=5000, calls=20, seat=0)
    cases.case_sharding(be, "blokus", B=300, calls=40, seat=2)


def test_contract_product_library(be):
    assert cases.case_contract(be.lib, emulator=False) >= 3


def test_python_surface_ttt():
    import torch
    from colosseumrl_b200.tictactoe import BatchedTicTacToe3PlayerEnv
    from colosseumrl_b200.vector import SingleAgentTurnVectorEnv

    B, seat, seed, env0 = 512, 2, 17, 90
    venv = SingleAgentTurnVectorEnv(BatchedTicTacToe3PlayerEnv(batch=B, seed=seed, first_env_id=env0), seat=seat)
    obs = venv.reset()
    ob = cases.TTTOracle(3, B)
    ob.advance(None, seat, seed, env0, 0)
    rng = np.random.RandomState(4)
    done_total = 0
    for t in range(1, 201):
        exp_obs = np.stack([orc.ttt_observation(3, (ob.board[e].reshape(3, 5), -1), seat) for e in range(B)])
        assert (obs["board"].cpu().numpy() == exp_obs).all(), t
        kept = venv.valid_actions()
        mask = kept.cpu().numpy().view(np.uint32)
        assert (mask == ((ob.board == -1).astype(np.uint64) << np.arange(15, dtype=np.uint64)).sum(1)).all()
        act = cases.ttt_learner_actions(rng, ob.board)
        obs, reward, done, info = venv.step(torch.tensor(act))
        assert (kept.cpu().numpy().view(np.uint32) == mask).all()          # a mask kept across a step does not change
        rec = ob.advance(act, seat, seed, env0, t)
        assert (reward.cpu().numpy() == rec[:, 0].view(np.int8)).all() and (done.cpu().numpy() == (rec[:, 1] & 1)).all()
        assert (info["winners"].cpu().numpy() == rec[:, 2]).all() and (info["opponent_moves"].cpu().numpy() == rec[:, 3]).all()
        assert (info["illegal"].cpu().numpy() == (rec[:, 1] >> 1 & 1)).all()
        done_total += int((rec[:, 1] & 1).sum())
    assert done_total > B


def test_python_surface_blokus():
    import torch
    from colosseumrl_b200.blokus import BatchedBlokusEnvironment, player_perspective_action_to_real, real_action_to_player_perspective
    from colosseumrl_b200.vector import SingleAgentTurnVectorEnv

    B, seat, seed, env0 = 64, 1, 23, 500
    venv = SingleAgentTurnVectorEnv(BatchedBlokusEnvironment(batch=B, seed=seed, first_env_id=env0), seat=seat, perspective=True)
    obs = venv.reset()
    ob = cases.BlokusOracle(B)
    ob.advance(None, seat, seed, env0, 0)
    rng = np.random.RandomState(6)
    done_total = 0
    for t in range(1, 201):
        counts, ids = (x.cpu().numpy() for x in venv.valid_actions())
        for e in range(0, B, 3):
            state = (ob.board[e], ob.round_count[e], ob.inventory[e], ob.scores[e])
            o = orc.blokus_observation(state, seat)
            assert (obs["board"][e].cpu().numpy() == o["board"]).all() and (obs["score"][e].cpu().numpy() == o["score"]).all()
            valid = orc.blokus_valid_moves(state, seat)
            assert counts[e] == len(valid) and (ids[e, :counts[e]] == real_action_to_player_perspective(valid, seat)).all(), (t, e)
        act = cases.blokus_learner_actions(rng, counts, ids)            # in the seat's rotated frame
        obs, reward, done, info = venv.step(torch.tensor(act))
        rec = ob.advance(player_perspective_action_to_real(act.astype(np.int64), seat).astype(np.int32), seat, seed, env0, t)
        assert (reward.cpu().numpy() == rec[:, 0].view(np.int8)).all() and (done.cpu().numpy() == (rec[:, 1] & 1)).all()
        assert (info["scores"].cpu().numpy() == rec[:, 4:8]).all() and (info["winners"].cpu().numpy() == rec[:, 2]).all()
        done_total += int((rec[:, 1] & 1).sum())
    assert done_total > 0
