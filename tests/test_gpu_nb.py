"""GPU: the bf16 per-tile kernel (mmn_nb.cuh: precision="bf16" on narrow models; mma.sync.m16n8k16 + ldmatrix + movmatrix,
activations chained through registers) against the oracle's bf16 restatement and the fp32 oracle (tests/nb_cases.py), plus
the full BASELINE config-2 shape at B = 65 536 through size-independent properties."""
import numpy as np
import pytest
import torch
from torch.nn import CrossEntropyLoss

from oracle import multimodn_oracle as O
from oracle.spec_io import random_spec, synthetic_batch
from multimodn_b200 import MultiModNHistory, FusedAdam, _lib
from helpers import flat_grads, assert_close
from model_utils import model_from_spec, GradTap, tapped_flat
from nb_cases import CASES, run_case, ENGINE_NB
import bf16_feature_cases as features

pytestmark = pytest.mark.gpu
DEV = "cuda"


@pytest.mark.parametrize("name", sorted(CASES))
def test_nb_case(name):
    run_case(name, DEV, _lib.get_lib())


@pytest.mark.parametrize("name", sorted(features.CASES))
def test_nb_feature_case(name):
    """non-ReLU activations, 1- to 8-class decoders, mixed module kinds, permuted / partial sequences (tests/bf16_feature_cases.py)"""
    features.run_feature_case(name, DEV, _lib.get_lib(), ENGINE_NB)


def test_nb_batch_missing_mode():
    run_case("ragged_dims_mnar", DEV, _lib.get_lib(), missing_mode="batch")


@pytest.mark.parametrize("B", [1, 37, 129, 5000])
def test_nb_tiny_ragged_and_multi_tile_batches(B):
    run_case("dropout_mnar", DEV, _lib.get_lib(), B=B)


def test_nb_c2_full_dims_against_the_bf16_oracle():
    """BASELINE config 2's exact layer sizes (6 / 99 / 1024 features, state 64, hidden 32), 2048 rows with MNAR rows and
    dropout: gradients per tensor against the bf16 restatement"""
    S, feats = 64, [6, 99, 1024]
    rng = np.random.default_rng(42)
    spec = random_spec(rng, S, feats, enc_kind="mimic", enc_hidden=(32, 32), dropout=0.2, n_decoders=2, dec_hidden=(32, 32))
    data, y = synthetic_batch(rng, feats, 2, 2048, mnar=True)
    model = model_from_spec(spec, 1.0, 0.3, DEV, "row", precision="bf16")
    rt = model.runtime()
    assert _lib.get_lib().dll.mmn_plan_engine(rt.plan) == ENGINE_NB
    rt.dropout_base_seed, rt.step_counter = 5, 0
    seed = (5 * 0x9E3779B1 + 1 * 0x85EBCA77) & 0xFFFFFFFF
    tap = GradTap(model.parameters())
    hist = MultiModNHistory(["a", "b"])
    loader = [([torch.from_numpy(x).to(DEV) for x in data], torch.from_numpy(y).to(DEV))]
    model.train_epoch(loader, tap, CrossEntropyLoss(), hist)
    got, _ = tapped_flat(model, tap)
    ospec = dict(O.cast_spec(spec, np.float32), precision="bf16")
    fwd, _, grads, _ = O.train_step(ospec, data, y, 1.0, 0.003, dropout_seed=seed)
    assert_close(got, flat_grads(grads), rtol=2e-3, what="C2-shaped grads vs the bf16 restatement")
    assert_close(hist.loss["train"][0], fwd["ce"], rtol=1e-4, what="loss")
    f32, _, _, _ = O.train_step(O.cast_spec(spec, np.float32), data, y, 1.0, 0.003, dropout_seed=seed)
    assert_close(hist.loss["train"][0], f32["ce"], rtol=1e-2, what="loss vs the fp32 oracle (north star: 1e-2 in bf16)")


def test_nb_full_batch_properties():
    """B = 65 536 on the config-2 shape: shard additivity of gradients / metrics (the data-parallel contract, dropout keyed by
    the global row), a 512-row oracle sample of the states, and bit-exact pass-through of rows whose modalities are all
    missing"""
    S, feats, B = 64, [6, 99, 1024], 65536
    rng = np.random.default_rng(9)
    spec = random_spec(rng, S, feats, enc_kind="mimic", enc_hidden=(32, 32), dropout=0.2, n_decoders=2, dec_hidden=(32, 32))
    g = torch.Generator(device=DEV).manual_seed(3)
    y = (torch.rand((B, 2), generator=g, device=DEV) < 0.3).to(torch.int64)
    xs = []
    for f in feats:
        x = torch.randn((B, f), generator=g, device=DEV)
        x[torch.rand((B,), generator=g, device=DEV) < 0.3] = float("nan")
        xs.append(x)
    model = model_from_spec(spec, 1.0, 0.3, DEV, "row", precision="bf16")
    rt = model.runtime()
    assert _lib.get_lib().dll.mmn_plan_engine(rt.plan) == ENGINE_NB
    seq = [(i, i) for i in range(len(feats))]

    def run(shards):
        acc_g, acc_m = torch.zeros_like(rt.gflat), rt.new_metrics()
        n = B // shards
        for r in range(shards):
            rt.step_counter = 0
            mb, keep, rows = rt.prepare_batch([t[r * n:(r + 1) * n] for t in xs], y[r * n:(r + 1) * n], seq, "row", (shards, r, None))
            rt.train_step(mb, rows, 1.0, 0.003, True, acc_m)
            acc_g += rt.gflat
        return acc_g.cpu().numpy(), acc_m.cpu().numpy()

    g1, m1 = run(1)
    g4, m4 = run(4)
    n_p = rt.packed.n_params
    scale = np.abs(g1[:n_p]).max()
    assert np.abs(g4[:n_p] - g1[:n_p]).max() / scale <= 1e-4, "sharded gradients must add up to the full-batch gradients"
    assert (g4[n_p:] == g1[n_p:]).all()
    assert_close(m4, m1, rtol=1e-5, what="sharded metrics == full-batch metrics")
    loader = [(xs, y)]
    states = torch.stack(model.get_states(loader)).cpu().numpy()
    idx = np.random.default_rng(0).choice(B, 512, replace=False)
    data_s = [x[idx].cpu().numpy() for x in xs]
    ospec = dict(O.cast_spec(spec, np.float32), precision="bf16")
    ofwd = O.forward(ospec, data_s, y[idx].cpu().numpy(), None, "row")
    assert_close(states[idx], ofwd["final_state"], rtol=8e-3, what="states of a 512-row sample vs the bf16 restatement")
    absent = torch.stack([torch.isnan(x).any(1) for x in xs]).all(0).cpu().numpy()
    assert absent.any()
    s0 = torch.tensor(spec["init_state"], dtype=torch.float32).to(torch.bfloat16).float().numpy().reshape(-1)
    assert (states[absent] == s0[None, :]).all()
    pred = model.predict(xs)
    opred = O.forward(ospec, data_s, None, None, "row")["predictions"]
    assert (pred[:, :, idx] != opred).mean() <= 0.005


def test_nb_training_follows_the_fp32_trajectory():
    S, feats = 64, [48, 80]
    rng = np.random.default_rng(5)
    spec = random_spec(rng, S, feats, enc_kind="mimic", enc_hidden=(32, 32), dropout=0.0, n_decoders=2, dec_hidden=(32,), n_classes=2)
    data, y = synthetic_batch(rng, feats, 2, 1024, mnar=True)
    losses = {}
    for prec in ("fp32", "bf16"):
        model = model_from_spec(spec, 1.0, 0.3, DEV, "row", precision=prec)
        opt = FusedAdam(model, lr=1e-2)
        hist = MultiModNHistory(["a", "b"])
        loader = [([torch.from_numpy(x).to(DEV) for x in data], torch.from_numpy(y).to(DEV))]
        for _ in range(8):
            model.train_epoch(loader, opt, CrossEntropyLoss(), hist)
        losses[prec] = np.array([m[-1].sum() for m in hist.loss["train"]])
    assert losses["bf16"][-1] < losses["bf16"][0]
    np.testing.assert_allclose(losses["bf16"], losses["fp32"], rtol=2e-2)
