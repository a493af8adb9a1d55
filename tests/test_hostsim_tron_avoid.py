"""CPU unit tests: the Tron avoid policy and its fused rollout (csrc/tron.cuh, csrc/tron_wide.cuh) executed on the SIMT
emulator against the C oracle and a numpy restatement of the rule; the host-side contract of both entry points.  (The
same cases run on the real GPU in test_gpu_tron_avoid.py.)"""
import pytest

import backends
import cases_tron_avoid as cases


@pytest.fixture(scope="module")
def be():
    return backends.HostSim()


def test_rule_handbuilt(be):
    cases.case_rule_handbuilt(be)                                     # the tuned layout
    cases.case_rule_handbuilt(be, N=11, P=6, n=300, seed=22)          # the wide layout


def test_policy_golden(be):
    cases.case_policy_golden(be)


def test_rollout_vs_oracle(be):
    cases.case_rollout_vs_oracle(be, N=19, P=4, B=130, K=30, mask=0b0010)
    cases.case_rollout_vs_oracle(be, N=19, P=4, B=70, K=40, mask=0b1110, noise_q16=6554, seed=4)
    cases.case_rollout_vs_oracle(be, N=7, P=3, B=65, K=40, mask=0b111, seed=5, spawns=[3, 0, -1])
    cases.case_rollout_vs_oracle(be, N=9, P=4, B=40, K=50, mask=0b1011, noise_q16=32768, seed=6, ring_offset=2,
                                 spawns=[1, 4, 0, 2])


def test_wide_rollout_vs_oracle(be):
    cases.case_rollout_vs_oracle(be, N=21, P=4, B=40, K=40, mask=0b0001, seed=7)
    cases.case_rollout_vs_oracle(be, N=11, P=6, B=40, K=30, mask=0b111110, seed=8, spawns=[2, 0, 1, 3, -1, 2])
    cases.case_rollout_vs_oracle(be, N=64, P=8, B=8, K=40, mask=0xFF, noise_q16=3277, seed=9)


def test_mask_zero_is_random_rollout(be):
    cases.case_mask_zero_is_random_rollout(be, N=19, P=4, B=70, K=30)
    cases.case_mask_zero_is_random_rollout(be, N=11, P=6, B=40, K=30)


def test_contract_emulator(be):
    assert cases.case_contract(be.lib, emulator=True) > 60


def test_contract_product_library():
    import torch
    from colosseumrl_b200 import _lib
    if torch.cuda.is_available():
        pytest.skip("GPU present: the emulator rows cover the shared argument checks")
    assert cases.case_contract(_lib.load(), emulator=False) > 10


def test_sanity_on_the_oracle():
    """the oracle's own run of the meaning check: the bounds hold, and the counts are the ones the bounds were set from"""
    ob, rnd = cases.sanity_counts()
    cases.check_sanity_bounds(ob.stats, rnd.stats)
    assert ob.stats[:8].tolist() == cases.SANITY_ORACLE
