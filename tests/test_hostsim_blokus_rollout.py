"""CPU unit tests: the fused Blokus rollout (blokus_rollout_kernel, crl_blokus_rollout) on the SIMT emulator vs the
oracle and the three-launch legal -> policy -> step sequence; host-side argument checks of the product library."""
import pytest

import backends
import cases_blokus_rollout as cases


@pytest.fixture(scope="module")
def be():
    return backends.HostSim()


def test_fused_vs_oracle(be):
    cases.case_fused_vs_oracle(be, B=4, K=72)                 # crosses an episode end


def test_fused_vs_chain(be):
    cases.case_fused_vs_chain(be, B=3, K=40, k1=13)


def test_arbitrary_positions(be):
    placed, missed = cases.case_positions(be, B=384, stride=14, strict=False)
    assert placed > 100


def test_sharding(be):
    cases.case_sharding(be, B=6, K=30)


def test_argument_checks_emulator(be):
    cases.case_argument_checks(be.lib)


def test_argument_checks_product_library():
    from colosseumrl_b200 import _lib
    cases.case_argument_checks(_lib.load())
