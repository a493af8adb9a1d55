"""GPU parity tests (B200): the Blokus placement masks, placement -> action conversion and the placement action space of
SingleAgentTurnVectorEnv through libcolosseum_b200.so, bit-exact against the C oracle's lists and crl_blokus_legal."""
import pytest

import backends
import cases_blokus_placement as cases

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def be():
    return backends.Cuda()


def test_golden_masks(be):
    cases.case_golden_masks(be)


def test_conversion(be):
    cases.case_conversion(be)


def test_step_equivalence(be):
    cases.case_step_equivalence(be)


def test_edges(be):
    cases.case_edges(be)


def test_full_size(be):
    cases.case_full_size(be, B=16384)


def test_contract_product_library(be):
    assert cases.case_contract(be.lib, emulator=False) >= 3


def test_python_surface():
    cases.case_python_surface()
