"""CPU unit tests: the host-side contract of every C-ABI entry point (cases_api_contract.py) -- refusals, their codes,
messages and order, accepted no-ops, host-only return values -- on the SIMT emulator build of crl_api.cu and, for the
rows that pass no device memory, on the product library."""
import pytest

import backends
import cases_api_contract as cases


@pytest.fixture(scope="module")
def be():
    return backends.HostSim()


def test_contract_emulator(be):
    assert cases.case_contract(be.lib, emulator=True) > 400


def test_host_values_emulator(be):
    cases.case_host_values(be.lib)


def test_contract_product_library():
    import torch
    from colosseumrl_b200 import _lib
    if torch.cuda.is_available():
        pytest.skip("GPU present: the emulator rows cover the shared argument checks")
    assert cases.case_contract(_lib.load(), emulator=False) > 100


def test_host_values_product_library():
    from colosseumrl_b200 import _lib
    cases.case_host_values(_lib.load())
