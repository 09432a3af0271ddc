"""Model features the other bf16 cases (tests/nb_cases.py, tests/test_gpu_wide.py) never build, run through both bf16 engines:
the tile kernel (mmn_nb.cuh; on the host emulator by tests/test_emu_nb.py and on the GPU by tests/test_gpu_nb.py) and the
layer-wise regime (mmn_wide*.cuh, tests/test_gpu_wide_features.py).  Those cases all use random_spec's defaults: ReLU encoders
and decoder hidden layers, a sigmoid output and the identity encoding sequence.  Here the kind and activation are chosen per
encoder, the activations per decoder, and every case walks a non-identity sequence.

Coverage, by construction ("lean_epilogue" runs on the wide regime only, every other case on both engines):

  feature                                       case (encoder eN / decoder dN)
  encoder act sigmoid: mimic / mlp              perm_sigmoid e0, lean_epilogue e0 / perm_sigmoid e1, batch_skip e1
  encoder act tanh: mimic / mlp                 perm_sigmoid e2, batch_skip e0, lean_epilogue e1 / partial_classdec e0
  encoder act identity: mimic / mlp             dropout_single_decoder (every encoder) / partial_classdec e2
  decoder hidden act tanh                       perm_sigmoid d0, batch_skip d1, lean_epilogue d1
  decoder hidden act sigmoid                    perm_sigmoid d1, dropout_single_decoder, lean_epilogue d0
  decoder hidden act identity                   partial_classdec d1, batch_skip d0
  decoder output act identity                   perm_sigmoid d0, batch_skip d0, lean_epilogue d0
  decoder output act relu                       perm_sigmoid d1
  decoder output act tanh                       partial_classdec d0, dropout_single_decoder, lean_epilogue d1
  decoder output act sigmoid                    partial_classdec d1, batch_skip d1
  wide decoder head C = 1                       partial_classdec d1
  wide decoder head C = 2                       dropout_single_decoder, batch_skip d0, lean_epilogue d0
  wide decoder head C = 3                       perm_sigmoid d0 (16-byte rows), batch_skip d1 (hidden 20: the unaligned variant)
  wide decoder head C = 4                       perm_sigmoid d1
  tile-kernel C = 8                             partial_classdec d0 (a ClassDecoder)
  wide data gradient, K-concatenated            perm_sigmoid, lean_epilogue
  wide data gradient, per decoder               partial_classdec (a ClassDecoder beside an MLPDecoder),
                                                dropout_single_decoder (D = 1), batch_skip (first hidden width 12)
  wide GEMM epilogue, lean (interior tiles)     lean_epilogue (S = hidden = 256, B = 256; sigmoid / tanh)
  wide GEMM epilogue, generic (edge tiles)      every other case (S = 24 / 40, ragged hidden widths)
  permuted sequence                             perm_sigmoid [2, 0, 1], lean_epilogue [1, 0]
  partial sequence                              partial_classdec [2, 0] (encoder 1 keeps .grad None)
  permuted sequence with dropout                dropout_single_decoder [1, 2, 0], p = 0.3 (the mask is keyed by encoder id)
  batch mode, one whole step skipped            batch_skip [1, 2, 0] (the step of encoder 2 = E - 1)

Every encoder of a case has the same feature width, so that data[pos] fits whichever encoder the sequence puts at `pos`.  State
widths 24 and 40 are not multiples of 16: the tile kernel runs them zero-padded to 64 columns, where a sigmoid would put
sigma(0) = 1/2 if the padding were not cleared.

Yardsticks, as in nb_cases.run_case: the oracle's bf16 restatement (gradients 2e-3 per tensor, losses 1e-4, state change 2e-3,
states and the outputs MultiModN.test() collects 8e-3, predictions <= 0.5 % flips) and the fp32 oracle (1e-2, gradient direction
cos >= 0.99, <= 3 % flips).  The largest measured error of each bound, as a fraction of the bound, over every case on the
tile kernel (one B200 at its 1000 W limit, and the host emulator) and the wide regime (the same B200):

  bound                                  bf16 restatement                      fp32 oracle
  gradients (2e-3 per tensor)            0.07  (wide, lean_epilogue)            --
  gradient direction (1 - cos)           0.001 of 1e-4 (emulator, batch_skip)   0.002 of 1e-2 (batch_skip)
  train / val loss (1e-4 / 1e-2)         0.011 (wide, lean_epilogue)            0.05  (perm_sigmoid)
  state change (2e-3 / 1e-2)             0.001 (emulator, dropout_single_dec.)  0.14  (dropout_single_decoder)
  states (8e-3 / 1e-2)                   0.32  (emulator, batch_skip)           0.45  (batch_skip)
  outputs test() collects (8e-3 / 1e-2)  0.08  (wide, lean_epilogue)            0.70  (perm_sigmoid)
  prediction flips (0.5 % / 3 %)         0 flips                                0.07  (perm_sigmoid)
The fp32 column measures bf16 itself: both engines are as far from the fp32 oracle as the restatement is.
"""
import numpy as np
import torch
from torch.nn import CrossEntropyLoss

from oracle import multimodn_oracle as O
from oracle.spec_io import _linear_init
from multimodn_b200 import MultiModNHistory
from helpers import flat_grads, assert_close
from model_utils import model_from_spec, GradTap, tapped_flat, batches

HIST = ("loss", "accuracy", "sensitivity", "specificity", "balanced_accuracy")
ENGINE_NB, ENGINE_WIDE = 4, 3

# name: S, F (features per encoder), encoders [(kind, hidden, act, dropout)], decoders [(hidden, n_classes, hidden_act, out_act)],
# encoding sequence, missing mode, P(row missing) per data position, B
CASES = {
    "perm_sigmoid": dict(
        S=24, F=12, seq=[2, 0, 1], mode="row", missing=[0.2, 0.2, 0.2], B=300,
        encoders=[("mimic", (20,), "sigmoid", 0.0), ("mlp", (20,), "sigmoid", 0.0), ("mimic", (16,), "tanh", 0.0)],
        decoders=[((16,), 3, "tanh", "identity"), ((24,), 4, "sigmoid", "relu")]),
    "partial_classdec": dict(
        S=40, F=10, seq=[2, 0], mode="row", missing=[0.2, 0.2, 0.2], B=300,
        encoders=[("mlp", (24,), "tanh", 0.0), ("mimic", (20,), "sigmoid", 0.0), ("mlp", (33,), "identity", 0.0)],
        decoders=[((), 8, "identity", "tanh"), ((16,), 1, "identity", "sigmoid")]),
    "dropout_single_decoder": dict(
        S=24, F=9, seq=[1, 2, 0], mode="row", missing=[0.15, 0.15, 0.15], B=300,
        encoders=[("mimic", (32, 16), "identity", 0.3)] * 3,
        decoders=[((40, 12), 2, "sigmoid", "tanh")]),
    "batch_skip": dict(
        S=24, F=16, seq=[1, 2, 0], mode="batch", missing=[0.0, 0.02, 0.0], B=256,
        encoders=[("mimic", (24,), "tanh", 0.0), ("mlp", (20,), "sigmoid", 0.0), ("mimic", (28,), "identity", 0.0)],
        decoders=[((12,), 2, "identity", "identity"), ((20,), 3, "tanh", "sigmoid")]),
}
# the layer-wise regime only (wider than the tile kernel takes): every GEMM tile interior and 16-byte aligned
WIDE_ONLY_CASES = {
    "lean_epilogue": dict(
        S=256, F=256, seq=[1, 0], mode="row", missing=[0.1, 0.1], B=256,
        encoders=[("mimic", (256,), "sigmoid", 0.0), ("mimic", (256,), "tanh", 0.0)],
        decoders=[((256,), 2, "sigmoid", "identity"), ((256,), 3, "tanh", "tanh")]),
}


def case_spec(c, rng):
    S, F = c["S"], c["F"]
    spec = dict(state_size=S, init_state=rng.standard_normal(S).astype(np.float32), encoders=[], decoders=[])
    for kind, hidden, act, p in c["encoders"]:
        dims = ([F + S] if kind == "mimic" else [F]) + list(hidden) + [S]
        layers = [_linear_init(rng, o, i + (S if kind == "mlp" and j == len(dims) - 2 else 0))
                  for j, (i, o) in enumerate(zip(dims, dims[1:]))]
        spec["encoders"].append(dict(kind=kind, n_features=F, act=act, dropout=p, layers=layers))
    for hidden, C, hact, oact in c["decoders"]:
        dims = [S] + list(hidden) + [C]
        spec["decoders"].append(dict(n_classes=C, hidden_act=hact, out_act=oact,
                                     layers=[_linear_init(rng, o, i) for i, o in zip(dims, dims[1:])]))
    return spec


def case_data(c, rng):
    B = c["B"]
    data = []
    for p in c["missing"]:
        x = rng.standard_normal((B, c["F"])).astype(np.float32)
        x[rng.random(B) < p] = np.nan
        data.append(x)
    y = np.stack([rng.integers(0, C, B) for _, C, _, _ in c["decoders"]], axis=1).astype(np.int64)
    return data, y


def last_outputs(model, data, y, seq, device):
    """the (rows, sum C) decoder outputs MultiModN.test() collects (at the step of encoder E - 1), read from the same forward
    call test() makes"""
    rt = model.runtime()
    pairs = model.get_encoder_iterable(seq, shuffle_mode=False, train=False)
    mb, keep, n = rt.prepare_batch([torch.from_numpy(x).to(device) for x in data], torch.from_numpy(y).to(device), pairs,
                                   model.missing_mode, None)
    out = torch.zeros((n, rt.sumC), dtype=torch.float32, device=rt.device)
    rt.forward(mb, n, metrics=rt.new_metrics(), last_outputs=out)
    del keep
    return out.cpu().numpy()


def run_feature_case(name, device, lib, engine):
    """one train step + predict / get_states / test / the collected outputs against both yardsticks; returns the measured
    error of every bound as a fraction of the bound"""
    c = {**CASES, **WIDE_ONLY_CASES}[name]
    rng = np.random.default_rng(sum(map(ord, name)))
    spec = case_spec(c, rng)
    data, y = case_data(c, rng)
    seq, mode = c["seq"], c["mode"]
    E, D = len(c["encoders"]), len(c["decoders"])
    err, scp = 0.8, 0.6
    model = model_from_spec(spec, err, scp, device, mode, precision="bf16")
    rt = model.runtime()
    assert lib.dll.mmn_plan_engine(rt.plan) == engine, f"{name}: the model should run on engine {engine}"
    tap = GradTap(model.parameters())
    hist = MultiModNHistory([str(i) for i in range(D)])
    loader = batches(data, y, c["B"], seq=seq, device=device)
    rt.dropout_base_seed, rt.step_counter = 77, 0
    seed = (77 * 0x9E3779B1 + 1 * 0x85EBCA77) & 0xFFFFFFFF
    model.train_epoch(loader, tap, CrossEntropyLoss(), hist)
    got, touched = tapped_flat(model, tap)
    assert np.isfinite(got).all()
    if len(seq) < E or mode == "batch":     # an encoder outside the sequence, or a whole step skipped: no gradient at all
        assert not touched.all(), f"{name}: the case should leave an encoder with .grad None"
    pred = model.predict([torch.from_numpy(x) for x in data], encoder_sequence=seq)
    states = torch.stack(model.get_states(loader)).cpu().numpy()
    model.test(loader, CrossEntropyLoss(), hist, tag="val")
    outs = last_outputs(model, data, y, seq, device)

    margins = {}

    def note(key, value):
        margins[key] = float(value)

    s32 = O.cast_spec(spec, np.float32)
    for yard, ospec in (("bf16", dict(s32, precision="bf16")), ("fp32", s32)):
        tight = yard == "bf16"
        fwd, _, grads, otouched = O.train_step(ospec, data, y, err, 0.01 * scp, encoder_sequence=seq, missing_mode=mode,
                                                  dropout_seed=seed)
        assert (touched == otouched).all(), f"{name}: encoders given a gradient {touched} vs the oracle's {otouched}"
        want = flat_grads(grads)
        if tight:
            note("bf16 grads", assert_close(got, want, rtol=2e-3, what=f"{name}: grads vs {yard} oracle"))
        w64 = np.asarray(want, dtype=np.float64)
        cos = float(got @ w64 / (np.linalg.norm(got) * np.linalg.norm(w64)))
        bound = 0.9999 if tight else 0.99
        assert cos >= bound, f"{name}: gradient direction vs {yard} oracle: cos = {cos}"
        note(f"{yard} 1 - cos", (1 - cos) / (1 - bound))
        acc = O.EpochAccumulator(E, D)
        acc.add(fwd)
        fin = acc.finalize()
        note(f"{yard} loss", assert_close(hist.loss["train"][0], fin["loss"], rtol=1e-4 if tight else 1e-2,
                                          what=f"{name}: train loss vs {yard} oracle"))
        note(f"{yard} state change", assert_close(hist.state_change_loss[0], fin["state_change"], rtol=2e-3 if tight else 1e-2,
                                                  what=f"{name}: state change vs {yard} oracle"))
        for n in HIST[1:]:          # counters: a near-tie arg-max may flip
            np.testing.assert_allclose(np.nan_to_num(getattr(hist, n)["train"][0]), np.nan_to_num(fin[n]),
                                       atol=0.01 if tight else 0.03, err_msg=f"{name}: {n} vs {yard} oracle")
        ofwd = O.forward(ospec, data, y, seq, mode)
        flips = (pred != ofwd["predictions"]).mean()
        assert flips <= (0.005 if tight else 0.03), f"{name}: {flips:.2%} of the predictions differ from the {yard} oracle's"
        note(f"{yard} prediction flips", flips / (0.005 if tight else 0.03))
        note(f"{yard} states", assert_close(states, ofwd["final_state"], rtol=8e-3 if tight else 1e-2,
                                            what=f"{name}: states vs {yard} oracle"))
        # test() collects the outputs of the step of encoder E - 1; a sequence without that encoder leaves them zero
        want_out = np.concatenate(ofwd["outputs"][E], axis=1) if E - 1 in seq else np.zeros_like(outs)
        note(f"{yard} collected outputs", assert_close(outs, want_out, rtol=8e-3 if tight else 1e-2,
                                                       what=f"{name}: test() outputs vs {yard} oracle"))
        vacc = O.EpochAccumulator(E, D)
        vacc.add(ofwd)
        note(f"{yard} val loss", assert_close(hist.loss["val"][0], vacc.finalize()["loss"], rtol=1e-4 if tight else 1e-2,
                                              what=f"{name}: val loss vs {yard} oracle"))
    return margins
