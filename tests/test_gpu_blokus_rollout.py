"""GPU parity tests (B200): the fused Blokus rollout (crl_blokus_rollout) vs the oracle and the three-launch
legal -> policy -> step sequence."""
import pytest

import backends
import cases_blokus_rollout as cases

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def be():
    return backends.Cuda()


def test_fused_vs_oracle(be):
    cases.case_fused_vs_oracle(be, B=1024, K=150, seed=0, env0=0)


def test_fused_vs_oracle_full_size(be):
    # 16 384 games x 70 steps: one full episode and the restart
    cases.case_fused_vs_oracle(be, B=16384, K=70, seed=2, env0=0)


def test_fused_vs_chain(be):
    cases.case_fused_vs_chain(be, B=512, K=90, seed=9, env0=77, k1=31)


def test_arbitrary_positions(be):
    # every first / middle / last draw of all 672 positions placed; the per-piece targets almost all
    placed, missed = cases.case_positions(be, B=1 << 17, strict=True)
    assert missed <= placed // 100, (placed, missed)


def test_sharding(be):
    cases.case_sharding(be, B=4096, K=80)


def test_python_surface():
    cases.case_python_surface()
