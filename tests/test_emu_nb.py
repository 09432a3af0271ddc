"""CPU: the bf16 per-tile kernel (mmn_nb.cuh) on the host emulator — fragment bookkeeping, staging, stash and masks end to
end against the oracle's bf16 restatement (tests/nb_cases.py).  The real mma.sync / ldmatrix / movmatrix instructions are
exercised by tests/test_gpu_nb.py."""
import pytest

from nb_cases import CASES, run_case
import bf16_feature_cases as features


@pytest.mark.parametrize("name", sorted(CASES))
def test_nb_case(emu, name):
    run_case(name, "cpu", emu)


def test_nb_batch_missing_mode(emu):
    run_case("ragged_dims_mnar", "cpu", emu, missing_mode="batch")


@pytest.mark.parametrize("B", [1, 37, 129])
def test_nb_tiny_and_ragged_batches(emu, B):
    run_case("dropout_mnar", "cpu", emu, B=B)


@pytest.mark.parametrize("name", sorted(features.CASES))
def test_nb_feature_case(emu, name):
    """non-ReLU activations, 1- to 8-class decoders, mixed module kinds, permuted / partial sequences (tests/bf16_feature_cases.py)"""
    features.run_feature_case(name, "cpu", emu, features.ENGINE_NB)
