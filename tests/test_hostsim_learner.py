"""CPU unit tests: the single-learner advance of Tic Tac Toe and Blokus (csrc/ttt.cuh, csrc/blokus.cuh) executed on the
SIMT emulator against the C oracle tests/oracle_learner.c; the host-side contract of both entry points.  (The same
cases run on the real GPU, at larger sizes, in test_gpu_learner.py.)"""
import pytest

import backends
import cases_learner as cases


@pytest.fixture(scope="module")
def be():
    return backends.HostSim()


@pytest.mark.parametrize("n", [2, 3, 4])
def test_ttt_calls(be, n):
    for seat in range(n):
        cases.case_ttt_calls(be, n, seat, B=70, calls=16, seed=3 + seat)


@pytest.mark.parametrize("n", [2, 3, 4])
def test_ttt_handbuilt(be, n):
    cases.case_ttt_handbuilt(be, n)


@pytest.mark.parametrize("n", [2, 3, 4])
def test_ttt_null_mode(be, n):
    cases.case_ttt_null_mode(be, n, B=70)


@pytest.mark.parametrize("seat", [0, 1, 2, 3])
def test_blokus_calls(be, seat):
    cases.case_blokus_calls(be, seat, B=6, calls=80)


def test_blokus_handbuilt(be):
    cases.case_blokus_handbuilt(be, stride=6, calls=2)


def test_blokus_null_mode(be):
    cases.case_blokus_null_mode(be, B=3)


def test_sharding(be):
    cases.case_sharding(be, "ttt", n=4, B=70, calls=10)
    cases.case_sharding(be, "ttt", n=3, B=40, calls=10, seat=2)
    cases.case_sharding(be, "blokus", B=4, calls=30, seat=2)


def test_contract_emulator(be):
    assert cases.case_contract(be.lib, emulator=True) > 40


def test_contract_product_library():
    import torch
    from colosseumrl_b200 import _lib
    if torch.cuda.is_available():
        pytest.skip("GPU present: the emulator rows cover the shared argument checks")
    assert cases.case_contract(_lib.load(), emulator=False) >= 3
