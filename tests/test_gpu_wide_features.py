"""GPU: the layer-wise regime (precision="bf16", mmn_wide*.cuh) on the model features tests/test_gpu_wide.py never builds --
sigmoid / tanh / identity activations in every position, decoder heads of 1, 3 and 4 classes, decoders off the K-concatenated
data-gradient path, permuted and partial encoding sequences, a skipped batch-mode step -- against the oracle's bf16 restatement
and the fp32 oracle (tests/bf16_feature_cases.py: the cases, the coverage table and the measured margins).

The cases the tile kernel also takes run here under MMN_ENGINE=wide; their small, ragged shapes put every GEMM tile on the
generic edge epilogue.  "lean_epilogue" (state and hidden widths 256, 256 rows) puts every tile on the interior epi_lean path."""
import pytest

from multimodn_b200 import _lib
import bf16_feature_cases as features

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def force_layerwise_regime(monkeypatch):
    """narrow models under precision="bf16" default to the per-tile kernel (tests/test_gpu_nb.py); this file is about the
    layer-wise tcgen05 regime, which MMN_ENGINE=wide selects for any model"""
    monkeypatch.setenv("MMN_ENGINE", "wide")


@pytest.mark.parametrize("name", sorted(features.CASES) + sorted(features.WIDE_ONLY_CASES))
def test_wide_feature_case(name):
    features.run_feature_case(name, "cuda", _lib.get_lib(), features.ENGINE_WIDE)
