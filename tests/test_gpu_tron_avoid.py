"""GPU parity tests (B200): the Tron avoid policy, its fused mixed-policy rollout and the single-learner vector env
through libcolosseum_b200.so, bit-exact against the C oracle (tests/oracle_tron_avoid.c)."""
import numpy as np
import pytest

import backends
import cases_tron_avoid as cases
from oracle import oracle as orc

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def be():
    return backends.Cuda()


def test_rule_handbuilt(be):
    cases.case_rule_handbuilt(be)
    cases.case_rule_handbuilt(be, N=19, P=2, n=400, seed=23)
    cases.case_rule_handbuilt(be, N=11, P=6, n=600, seed=22)           # the wide layout
    cases.case_rule_handbuilt(be, N=25, P=8, n=300, seed=24)


def test_policy_golden(be):
    cases.case_policy_golden(be)


def test_rollout_vs_oracle_small(be):
    cases.case_rollout_vs_oracle(be, N=19, P=4, B=130, K=30, mask=0b0010)
    cases.case_rollout_vs_oracle(be, N=7, P=3, B=400, K=60, mask=0b111, seed=5, spawns=[3, 0, -1])
    cases.case_rollout_vs_oracle(be, N=8, P=2, B=1000, K=40, mask=0b01, noise_q16=6554, seed=2)
    cases.case_rollout_vs_oracle(be, N=9, P=4, B=300, K=50, mask=0b1011, noise_q16=32768, seed=6, ring_offset=2,
                                 spawns=[1, 4, 0, 2])


@pytest.mark.parametrize("mask", [0, 0b0001, 0b1110, 0b1111])
def test_rollout_vs_oracle_full_size(be, mask):
    # BASELINE.json configs[1]: 65,536 environments x 64 steps, 19x19, 4 players
    cases.case_rollout_vs_oracle(be, N=19, P=4, B=65536, K=64, mask=mask, seed=0, env0=0)


def test_wide_rollout_vs_oracle(be):
    cases.case_rollout_vs_oracle(be, N=21, P=4, B=300, K=60, mask=0b0001, seed=7)
    cases.case_rollout_vs_oracle(be, N=11, P=6, B=500, K=40, mask=0b111110, seed=8, spawns=[2, 0, 1, 3, -1, 2])
    cases.case_rollout_vs_oracle(be, N=25, P=8, B=2000, K=50, mask=0b10101010, noise_q16=3277, seed=6, env0=77)
    cases.case_rollout_vs_oracle(be, N=64, P=8, B=70, K=90, mask=0xFF, seed=9)
    cases.case_rollout_vs_oracle(be, N=64, P=8, B=70, K=90, mask=0x7F, noise_q16=65536, seed=10)


def test_mask_zero_is_random_rollout(be):
    cases.case_mask_zero_is_random_rollout(be, N=19, P=4, B=65536, K=64)
    cases.case_mask_zero_is_random_rollout(be, N=11, P=6, B=500, K=40)


def test_contract_product_library(be):
    assert cases.case_contract(be.lib, emulator=False) > 10


def test_sanity_counts(be):
    """seats 1..3 on the avoid policy, seat 0 random, 19x19: the GPU reproduces the oracle's exact counts, and they meet
    the bounds (avoid seats win far more often, episodes last longer than under random play)"""
    s = cases.SANITY
    ob, rnd = cases.sanity_counts()
    assert ob.stats[:8].tolist() == cases.SANITY_ORACLE
    st = cases.device_reset(be, s["N"], s["P"], s["B"])
    stats = be.zeros((cases.STAT_ROWS, 32), np.int64)
    cases.rollout_avoid(be, st, s["seed"], s["env0"], 0, s["K"], s["N"], s["P"], 0b1110, 0, stats=stats)
    got = be.download(stats).sum(0)
    assert (got == ob.stats).all(), (got, ob.stats)
    cases.check_sanity_bounds(got, rnd.stats)


def _absolute(env, state):
    obs = env.state_to_observation(state, -1)
    return tuple(obs[k].cpu().numpy().astype(np.int64) for k in ("board", "heads", "directions", "deaths"))


def test_python_surface():
    import torch
    from colosseumrl_b200.tron import BatchedTronGridEnvironment, create_tron_config
    from colosseumrl_b200.vector import SingleAgentVectorEnv

    # avoid_actions: a played-in state, non-default spawns, auto-reset of the finished games
    B, N, P, seed, env0, spawns = 256, 11, 4, 13, 100, [3, 0, 1, -1]
    env = BatchedTronGridEnvironment(create_tron_config(N, P), batch=B, seed=seed, auto_reset=True, first_env_id=env0)
    state, _ = env.new_state(spawn_offset=spawns)
    for t in range(12):
        state, *_ = env.next_state(state, None, env.random_actions(t))
    board, heads, dirs, deaths = _absolute(env, state)
    assert (env.is_terminal(state).cpu().numpy() != 0).any()
    prior = np.full((B, 4), cases.SENTINEL, np.int8)
    got = env.avoid_actions(state, 12, seats=[1, 3], noise=0.25, out=torch.tensor(prior, device=env.device))
    exp, _ = cases.expected_policy(board, heads, dirs, deaths, prior, 0b1010, 16384, seed, env0, 12, cases.AUTO_RESET, 1, spawns)
    assert (got.cpu().numpy() == exp).all()
    got = env.avoid_actions(state, 13)                                    # all seats, a fresh zeroed buffer
    exp, _ = cases.expected_policy(board, heads, dirs, deaths, np.zeros((B, 4), np.int8), 0b1111, 0, seed, env0, 13,
                                   cases.AUTO_RESET, 1, spawns)
    assert (got.cpu().numpy() == exp).all()

    # rollout(avoid_seats=...) with the remembered spawns
    env.reset_stats()
    state, _ = env.new_state(spawn_offset=spawns)
    env.rollout(state, 0, 70, avoid_seats=0b0110, noise=0.1)
    ob = cases.AvoidBatch(B, N, P)
    ob.rollout_avoid(seed, env0, 0, 70, 0b0110, 6554, 1, spawns, fresh=True)
    board, heads, dirs, deaths = _absolute(env, state)
    assert (board == ob.board).all() and (heads == ob.heads).all() and (deaths == ob.deaths).all()
    assert (env.stats.cpu().numpy() == ob.stats).all()

    # SingleAgentVectorEnv against the oracle driven the same way, over a few hundred steps
    B, N, P, seat, noise_q16, env0, seed = 48, 9, 4, 2, 3277, 7, 31
    venv = SingleAgentVectorEnv(BatchedTronGridEnvironment(create_tron_config(N, P), batch=B, seed=seed,
                                                           first_env_id=env0), seat=seat, noise=noise_q16 / 65536)
    obs = venv.reset()
    states = [orc.tron_new_state(N, P) for _ in range(B)]
    rng = np.random.RandomState(5)
    opponents = sum(1 << p for p in range(P) if p != seat)
    ends, deaths_only = 0, 0
    for t in range(300):
        for e in range(0, B, 7):
            o = orc.tron_observation(states[e], seat)
            assert (obs["board"][e].cpu().numpy() == o["board"]).all() and (obs["heads"][e].cpu().numpy() == o["heads"]).all()
        la = rng.randint(-1, 2, size=B).astype(np.int8)
        obs, reward, done, info = venv.step(torch.tensor(la))
        reward, done = reward.cpu().numpy(), done.cpu().numpy()
        for e in range(B):
            act = np.zeros(P, np.int64)
            act[seat] = la[e]
            act = cases.orc_avoid(states[e], act, opponents, noise_q16, seed, env0 + e, t)
            new, alive, rewards, terminal, _ = orc.tron_next_state(states[e], act)
            learner_dead = not (alive >> seat) & 1
            assert reward[e] == rewards[seat] and bool(done[e]) == (terminal or learner_dead), (t, e)
            ends += int(terminal)
            deaths_only += int(learner_dead and not terminal)
            states[e] = orc.tron_new_state(N, P) if (terminal or learner_dead) else new
    assert ends > 0 and deaths_only > 0, (ends, deaths_only)
