"""Shared test helpers: golden-fixture loading and tolerant comparisons."""
import os

import numpy as np

from oracle.spec_io import spec_from_arrays

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

RTOL_FP32 = 1e-5      # BASELINE.json north_star: 1e-5 relative in fp32


def load_golden(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False)
    return {k: z[k] for k in z.files}


def golden_data(fx, prefix="x"):
    out = []
    while f"{prefix}{len(out)}" in fx:
        out.append(fx[f"{prefix}{len(out)}"])
    return out


def golden_spec(fx, prefix="spec0"):
    return spec_from_arrays(fx, prefix)


def golden_grads(fx, spec, prefix="grad0"):
    g = dict(init_state=fx[f"{prefix}_init"], encoders=[], decoders=[])
    for e, enc in enumerate(spec["encoders"]):
        g["encoders"].append([(fx[f"{prefix}_e{e}_W{j}"], fx[f"{prefix}_e{e}_b{j}"]) for j in range(len(enc["layers"]))])
    for d, dec in enumerate(spec["decoders"]):
        g["decoders"].append([(fx[f"{prefix}_d{d}_W{j}"], fx[f"{prefix}_d{d}_b{j}"]) for j in range(len(dec["layers"]))])
    return g


class SegArray(np.ndarray):
    """flat vector that remembers where each parameter tensor starts: ``assert_close`` then normalises every tensor by its
    OWN magnitude (a bias or init-state gradient 1000x smaller than the largest weight gradient is checked as tightly as
    the rest) instead of by the magnitude of the whole concatenation."""
    segments = None


def _seg(parts, names):
    flat = np.concatenate([np.asarray(p).ravel() for p in parts]).view(SegArray)
    segs, at = [], 0
    for n, p in zip(names, parts):
        k = int(np.asarray(p).size)
        segs.append((n, at, at + k))
        at += k
    flat.segments = segs
    return flat


def flat_grads(g):
    parts, names = [np.asarray(g["init_state"])], ["init_state"]
    for gname, group in (("enc", g["encoders"]), ("dec", g["decoders"])):
        for i, layers in enumerate(group):
            for j, (W, b) in enumerate(layers):
                parts += [np.asarray(W), np.asarray(b)]
                names += [f"{gname}{i}.W{j}", f"{gname}{i}.b{j}"]
    return _seg(parts, names)


def flat_params(spec):
    parts, names = [np.asarray(spec["init_state"])], ["init_state"]
    for gname, group in (("enc", spec["encoders"]), ("dec", spec["decoders"])):
        for i, m in enumerate(group):
            for j, (W, b) in enumerate(m["layers"]):
                parts += [W, b]
                names += [f"{gname}{i}.W{j}", f"{gname}{i}.b{j}"]
    return _seg(parts, names)


# a tensor whose expected values are all (nearly) zero is compared against this fraction of the largest tensor's magnitude
ZERO_TENSOR_FLOOR = 1e-6
# Per-tensor bound = PER_TENSOR_SLACK x rtol of the tensor's OWN magnitude, on top of the norm-wise bound rtol over the whole
# vector.  Two fp32 evaluations of the same sum in different orders (kernel tiles + atomics vs numpy) differ by a few 1e-5 of
# a small tensor whose entries cancel (measured: 1.5e-5 on a 16 x 8 decoder weight gradient over 1189 rows); a tensor that
# is actually wrong is off by O(1) of its own magnitude, which is what this check is for.
PER_TENSOR_SLACK = 4.0


def assert_close(actual, expected, rtol=RTOL_FP32, atol_scale=1.0, what=""):
    """relative to the magnitude of the expected ARRAY (norm-wise): the right yardstick for fp32 sums whose individual
    elements may cancel to ~0.  When ``expected`` (or ``actual``) comes from flat_grads / flat_params the comparison runs
    per parameter tensor, each normalised by its own max |expected|.
    Returns the measured error as a fraction of its bound (the larger of the norm-wise and the per-tensor ratio), so that a
    caller can report the margin it passed with."""
    segments = getattr(expected, "segments", None) or getattr(actual, "segments", None)
    actual = np.asarray(actual, dtype=np.float64)
    expected = np.asarray(expected, dtype=np.float64)
    assert actual.shape == expected.shape, (what, actual.shape, expected.shape)
    nan_a, nan_e = np.isnan(actual), np.isnan(expected)
    assert (nan_a == nan_e).all(), f"{what}: NaN pattern differs"
    if nan_e.all():
        return 0.0
    gscale = max(np.abs(expected[~nan_e]).max(), 1e-30)
    err = np.abs(actual[~nan_e] - expected[~nan_e]).max() / gscale
    assert err <= rtol * atol_scale, f"{what}: max err / max|expected| = {err:.3e} > {rtol * atol_scale:.1e}"
    if segments is None or actual.ndim != 1:
        return err / (rtol * atol_scale)
    worst = (0.0, "")
    for name, lo, hi in segments:
        a, e = actual[lo:hi], expected[lo:hi]
        ok = ~np.isnan(e)
        if not ok.any():
            continue
        scale = max(np.abs(e[ok]).max(), ZERO_TENSOR_FLOOR * gscale)
        err = np.abs(a[ok] - e[ok]).max() / scale
        if err > worst[0]:
            worst = (err, name)
    bound = rtol * atol_scale * PER_TENSOR_SLACK
    assert worst[0] <= bound, f"{what}: tensor {worst[1]}: max err / max|expected tensor| = {worst[0]:.3e} > {bound:.1e}"
    return max(err / (rtol * atol_scale), worst[0] / bound)
