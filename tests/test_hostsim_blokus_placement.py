"""CPU unit tests: the Blokus placement masks and placement -> action conversion (csrc/blokus.cuh) executed on the SIMT
emulator against the C oracle's lists; the shape table, the Python helpers and the host-side contract of the three entry
points.  (The same cases run on the real GPU, on every position and at full size, in test_gpu_blokus_placement.py.)"""
import pytest

import backends
import cases_blokus_placement as cases


@pytest.fixture(scope="module")
def be():
    return backends.HostSim()


def test_golden_masks(be):
    cases.case_golden_masks(be, stride=5)


def test_conversion(be):
    cases.case_conversion(be, stride=7, per_position=6)


def test_step_equivalence(be):
    cases.case_step_equivalence(be, stride=9, ids_per_position=8)


def test_edges(be):
    cases.case_edges(be)


def test_shape_table(be):
    cases.case_shape_table(be.lib)


def test_python_helpers():
    cases.case_python_helpers()


def test_contract_emulator(be):
    assert cases.case_contract(be.lib, emulator=True) > 30


def test_contract_product_library():
    import torch
    from colosseumrl_b200 import _lib
    if torch.cuda.is_available():
        pytest.skip("GPU present: the emulator rows cover the shared argument checks")
    assert cases.case_contract(_lib.load(), emulator=False) >= 3
