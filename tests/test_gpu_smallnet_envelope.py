"""The fused small-network kernels (csrc/smallnet.cu) over the range smallnet_eligible() sends to them: 1 to 4 layers, each 1
to 32 wide, any n_in, through all four routes -- given features (kernel A FUSED 0), the generic front end (FUSED 1), the
staged front end (FUSED 2), and the feature kernel followed by FUSED 0 when the front end does not fit in shared memory.

CASES is a table of networks, batches and inputs chosen for the launch geometry they produce: every kernel B cluster size
from 1 to 8, a one-sample last K-split, the small CTA staging in several passes, one or two small groups with more small
parameters than threads, n_small at kernel A's capacity (4 x 32), widths and class counts of 1 and 32.  The host-side
geometry is restated below so that a CPU-only test keeps the table honest when someone edits it; every case is then run
on the GPU against the oracle (training step, split step, determinism, forward pass, evaluate_images), and each entry
point's launches are pinned so that a dispatcher change cannot quietly move a case off the kernels it is meant to test."""
import zlib
from collections import namedtuple

import numpy as np
import pytest

import oracle as O
from conftest import assert_close

gpu = pytest.mark.gpu

ETA = 3.0
CONV_NONE, CONV_SAME, POOL_MAX = 0, 1, 3   # RCN_LAYER_* codes

# launch names, as test_gpu_step_launches.py / test_gpu_evaluate.py use them
A_FEATS = "smallnet_fwd_bwd_kernel"                                         # kernel A on given features (FUSED 0)
A_FUSED = "smallnet_fwd_bwd_kernel(fused features)"                         # kernel A, FUSED 1 or 2
B_UPDATE = "smallnet_wgrad_kernel(+SGD update)"
B_PLAIN = "smallnet_wgrad_kernel"
SGD = "sgd_update_kernel"
INFER_STAGED = "smallnet_infer_kernel(fused features)"                      # FUSED 2
INFER_GENERIC = "smallnet_infer_kernel(fused features, generic front end)"  # FUSED 1
FEATS_STAGED = "features_cp_kernel"       # feature kernel for stacks make_cp_plan accepts
FEATS_GENERIC = "features_fused_kernel"   # ... and for the others

Case = namedtuple("Case", "name cfg hw n_in hidden classes B route")


def F(name, n_in, hidden, classes, B):
    return Case(name, None, None, n_in, list(hidden), classes, B, "features")


def I(name, cfg, hw, hidden, classes, B, route):
    return Case(name, list(cfg), hw, None, list(hidden), classes, B, route)


CASES = [
    I("staged-784-4x32-B129", [1, 3], (28, 28), [32, 32, 32], 32, 129, "staged"),
    F("feats-784-30-10-B1025", 784, [30], 10, 1025),
    I("staged-784-30-10-B2048", [1, 3], (28, 28), [30], 10, 2048, "staged"),
    I("unfit-4096-4x32-B300", [1, 3], (64, 64), [32, 32, 32], 32, 300, "unfit"),
    F("feats-65-1-1-B257", 65, [1], 1, 257),
    F("feats-3-32-32-32-1-B321", 3, [32, 32, 32], 1, 321),
    F("feats-2000-8-9-32-32-B385", 2000, [8, 9, 32], 32, 385),
    F("feats-63-31-17-5-32-B193", 63, [31, 17, 5], 32, 193),
    I("generic-conv-none-28x28-B7", [0, 3], (28, 28), [16, 8], 10, 7, "generic"),
    I("generic-conv-conv-8x12-B9", [1, 1], (8, 12), [32], 32, 9, "generic"),
    I("generic-pool-first-32x32-B8", [3, 1, 3, 3], (32, 32), [32, 32, 32], 10, 8, "generic"),
    I("generic-one-row-maps-8x12-B1", [1, 3, 0, 3], (8, 12), [5], 3, 1, "generic"),
    I("generic-30x28-B100", [1, 3], (30, 28), [30], 10, 100, "generic"),
    I("unfit-conv-conv-12x20-B65", [1, 1], (12, 20), [7, 3], 2, 65, "unfit"),
]
IMAGE_CASES = [c for c in CASES if c.cfg is not None]


# ---- smallnet.cu's host-side launch geometry, restated ---------------------------------------------------------------
def plan_stages(cfg, H, W):
    """plan_features (features.cu:17-73): [(kind, same, n_in, h_in, w_in, h_out, w_out)], n_conv, max_elems, L."""
    st, maps, h, w, i, n_conv, max_elems = [], 0, H, W, 0, 0, H * W
    while i < len(cfg):
        if cfg[i] in (CONV_NONE, CONV_SAME):
            same, n_in, h_in, w_in = cfg[i] == CONV_SAME, maps or 1, h, w
            if not same:
                h, w = h - 2, w - 2
            kind, maps, n_conv = 0, maps * 4 or 4, n_conv + 1
            if i + 1 < len(cfg) and cfg[i + 1] == POOL_MAX:   # a directly following pool is fused into the stage
                kind, h, w, i = 1, (h + 1) // 2, (w + 1) // 2, i + 1
            st.append((kind, same, n_in, h_in, w_in, h, w))
            max_elems = max(max_elems, n_in * h_in * w_in)
        elif maps:                                            # pooling an empty feature set is a no-op
            st.append((2, True, maps, h, w, (h + 1) // 2, (w + 1) // 2))
            max_elems = max(max_elems, maps * h * w)
            h, w = (h + 1) // 2, (w + 1) // 2
        i += 1
    return st, n_conv, max_elems, maps * h * w


def cp_plan(st, n_conv, H, W):
    """make_cp_plan (features.cu:199-230) and smallnet_front_select's H*W % 16 (smallnet.cu:1022-1027):
    (stage_bytes, tile_ints), or None when the staged front end does not take the stack."""
    if not 1 <= len(st) <= 8 or n_conv > 10 or W % 4 or (H * W) % 16:
        return None
    off = 0
    for kind, same, n_in, h, w, ho, wo in st:
        if kind != 1 or not same or ho < 2:
            return None
        off += n_in * ((h + 4) & ~1) * (w + 3)                # cp_pitch(h) * cp_cols(w) ints per map
        if n_in * ho * wo >= 1 << 16 or off > 1 << 20:
            return None
    return (H * W + 127) // 128 * 128, off


def geometry(c):
    rows = c.hidden + [c.classes]
    route, n_in = "features", c.n_in
    if c.cfg is not None:
        st, n_conv, max_elems, n_in = plan_stages(c.cfg, *c.hw)
        cp = cp_plan(st, n_conv, *c.hw)
        smem = (16 * 8 * 36 + 32 + 3 * (32 * 32 + 32)) * 8 + 8 * (n_in + 4) * 8   # kernel_a_smem (smallnet.cu:1010-1018)
        smem += 128 + 8 * (cp[0] + 4 * cp[1]) if cp else 8 * 2 * max_elems * 4
        route = "unfit" if smem > 200 * 1024 else "staged" if cp else "generic"   # smallnet_front_fits (:1020)
    s = 1                                                     # smallnet_splits (:986-994)
    while s < 8 and s * 64 < c.B:
        s *= 2
    ksplit = (-(-c.B // s) + 63) // 64 * 64
    S = -(-c.B // ksplit)
    n_small = rows[0] + sum(r * k + r for k, r in zip(rows, rows[1:]))   # n_params - b_off[0] (:1132)
    per_sample = sum(rows[:-1]) + sum(rows)                  # a_0..a_{n-2} | delta_0..delta_{n-1} (:1140-1145)
    chunk = max(1, min(ksplit, 96 * 1024 // 8 // per_sample))
    col_groups = -(-n_in // 64)                              # (:1131)
    small_groups = 2 if n_small > 256 and (col_groups + 2) * S <= 120 else 1   # (:1166)
    return dict(route=route, n_in=n_in, rows=rows, S=S, ksplit=ksplit, last=c.B - (S - 1) * ksplit, n_small=n_small,
                chunk=chunk, multi=min(c.B, ksplit) > chunk, small_groups=small_groups, col_groups=col_groups)


def test_case_table_covers_the_envelope():
    """CPU only: the table reaches every geometry the kernels branch on (see the module docstring)."""
    geo = {c.name: geometry(c) for c in CASES}
    for c in CASES:
        g = geo[c.name]
        assert g["route"] == c.route, (c.name, g["route"])
        assert 1 <= len(g["rows"]) <= 4 and all(1 <= r <= 32 for r in g["rows"]), c.name   # smallnet_eligible
        if c.cfg is not None:
            n, h, w = O.feature_shape(c.cfg, *c.hw)
            assert n * h * w == g["n_in"], (c.name, "plan_stages disagrees with the oracle's feature length")
    gs = list(geo.values())
    assert {g["S"] for g in gs} == set(range(1, 9)), "cluster sizes 1..8"
    assert any(g["S"] > 1 and g["last"] == 1 for g in gs), "a one-sample last K-split"
    assert any(g["multi"] for g in gs), "small CTA staging in several passes"
    assert {g["small_groups"] for g in gs if g["n_small"] > 256} == {1, 2}
    assert any(g["n_small"] == 32 + 3 * (32 * 32 + 32) for g in gs), "n_small == SN_MAX_SMALL"
    assert {len(g["rows"]) for g in gs} >= {2, 3, 4}
    assert {1, 32} <= {r for g in gs for r in g["rows"][:-1]}, "hidden widths 1 and 32"
    assert {1, 32} <= {g["rows"][-1] for g in gs}, "1 and 32 classes"
    assert any(g["n_in"] % 4 for g in gs) and any(g["n_in"] < 64 for g in gs)
    assert {1, 63} <= {g["n_in"] % 64 for g in gs}
    assert {c.route for c in CASES} == {"features", "generic", "staged", "unfit"}
    assert any(c.B in (1, 7, 8, 9) for c in IMAGE_CASES), "kernel A tile edges"
    # a 2x2 map cannot be convolved (kernel.rs:199-201): 1-row maps need a Padding::None stage
    with pytest.raises(O.RefPanic):
        O.feature_shape([1, 3, 1, 3], 4, 4)


# ---- GPU side -------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def api(built_library):
    import mercer_research_b200 as m
    return m


def launched(fn):
    """(kernel launches by name, fn()) -- the library's launch profile around one call."""
    import torch
    from mercer_research_b200 import _lib
    torch.cuda.synchronize()
    _lib.profile_enable(True)
    try:
        out = fn()
        got = {name: v["launches"] for name, v in _lib.profile_report().items()}
    finally:
        _lib.profile_enable(False)
    return got, out


def draw_params(shapes, rng):
    """W ~ N(0, 4 / cols), b ~ N(0, 1/4): the sigmoids stay mostly unsaturated."""
    parts = []
    for r, k in shapes:
        parts += [rng.standard_normal(r * k) * (2.0 / np.sqrt(k)), rng.standard_normal(r) * 0.5]
    return np.concatenate(parts)


def make_case(api, c, params=None):
    """(model, net, params, X, images, labels): standardised features X as the oracle computes them, u8 images for the
    image cases, and labels of which half are the oracle's prediction (so that there are hits to count)."""
    g = geometry(c)
    rng = np.random.default_rng(zlib.crc32(c.name.encode()))
    shapes = list(zip(g["rows"], [g["n_in"]] + g["rows"][:-1]))
    model = api.RCN(c.classes, c.cfg or [], c.hidden, device=0)
    model.load_weights_and_bias_shapes(shapes)
    net = O.Net(shapes)
    images = None
    if c.cfg is None:
        X = np.maximum(rng.standard_normal((c.B, c.n_in)), 0)
    else:
        images = rng.integers(0, 256, size=(c.B,) + c.hw, dtype=np.uint8)
        calib = rng.integers(0, 256, size=(32,) + c.hw, dtype=np.uint8)
        mean, sd = O.gen_scales(O.features_u8(c.cfg, calib))
        model.scale_set = (mean, sd)
        X = O.standardise(O.features_u8(c.cfg, images), mean, sd)
    if params is None:
        params = draw_params(shapes, rng)
    model.set_params(params)
    labels = rng.integers(0, c.classes, size=c.B).astype(np.int64)
    pred = O.argmax_last(net.forward(params, X))
    labels[: c.B // 2] = pred[: c.B // 2]
    return model, net, params, X, images, labels


def onehot(labels, classes):
    return np.eye(classes)[labels]


def step_launches(c, fused):
    a = A_FEATS if c.route in ("features", "unfit") else A_FUSED
    want = {a: 1, B_UPDATE: 1} if fused else {a: 1, B_PLAIN: 1, SGD: 1}
    if c.route == "unfit":
        want[FEATS_STAGED if cp_plan(*plan_stages(c.cfg, *c.hw)[:2], *c.hw) else FEATS_GENERIC] = 1
    return want


def fused_step(model, c, X, images, labels):
    if images is None:
        model.train_batch(X, ETA, labels=labels)
    else:
        model.train_batch_images(images, labels, ETA)


def split_step(model, c, X, images, labels):
    if images is None:
        model.accumulate_gradients(X, labels=labels)
    else:
        model.accumulate_gradients_images(images, labels)
    stats = model.last_batch_stats()
    model.apply_gradients(ETA, c.B)
    return stats


def tap_samples(B, ksplit):
    """Every sample up to 1100; above, positions 0-7 of the first and last tile of 8 and the first and last sample of each
    K-split."""
    if B <= 1100:
        return range(B)
    last_tile = (B - 1) // 8 * 8
    s = set(range(8)) | set(range(last_tile, B))
    for k0 in range(0, B, ksplit):
        s |= {k0, min(B, k0 + ksplit) - 1}
    return sorted(s)


def check_taps(model, net, params, X, Y, samples, what):
    acts = [model.activations(l) for l in range(net.n)]
    dels = [model.deltas(l) for l in range(net.n)]
    for b in samples:
        _, _, a, d = net.backprop(params, X[b], Y[b])
        o = 0
        for l, (r, _) in enumerate(net.shapes):
            assert_close(acts[l][b], a[o:o + r], what=f"{what}: a[{l}][sample {b}]")
            assert_close(dels[l][b], d[o:o + r], what=f"{what}: delta[{l}][sample {b}]")
            o += r


@gpu
@pytest.mark.parametrize("c", CASES, ids=[c.name for c in CASES])
def test_training_step(api, c):
    """Kernel A + kernel B MODE 2 (fused SGD update) against the oracle: gradient sums, parameters, statistics and every
    layer's activations and deltas; then MODE 0 + sgd_update_kernel, a repeat, and one-hot targets, bit for bit."""
    g = geometry(c)
    model, net, params, X, images, labels = make_case(api, c)
    Y = onehot(labels, c.classes)
    want_params, want_grads = net.train_batch(params, X, Y, ETA)
    want_acts = net.forward(params, X)

    got, _ = launched(lambda: fused_step(model, c, X, images, labels))
    assert got == step_launches(c, fused=True), got
    grads, new_params, stats = model.get_gradients(), model.get_params(), model.last_batch_stats()
    assert_close(grads, want_grads, what="sum dW/db")
    assert_close(new_params, want_params, what="post-step parameters")
    cost, hits = stats
    assert hits == O.accuracy(want_acts, labels)
    want_cost = 0.5 * float(np.sum((want_acts - Y) ** 2))
    assert abs(cost - want_cost) <= 1e-9 * max(1.0, want_cost), (cost, want_cost)
    check_taps(model, net, params, X, Y, tap_samples(c.B, g["ksplit"]), c.name)

    model.set_params(params)
    got, split_stats = launched(lambda: split_step(model, c, X, images, labels))
    assert got == step_launches(c, fused=False), got
    assert split_stats == stats
    assert np.array_equal(model.get_gradients(), grads), "split step: gradients differ from the fused step's"
    assert np.array_equal(model.get_params(), new_params), "split step: parameters differ from the fused step's"

    model.set_params(params)
    fused_step(model, c, X, images, labels)
    assert np.array_equal(model.get_gradients(), grads), "repeated step: gradients are not deterministic"
    assert np.array_equal(model.get_params(), new_params)
    assert model.last_batch_stats() == stats

    if images is None:
        model.set_params(params)
        model.train_batch(X, ETA, onehot=Y)
        assert np.array_equal(model.get_gradients(), grads), "one-hot targets: gradients differ from labels'"
        assert np.array_equal(model.get_params(), new_params)


@gpu
@pytest.mark.parametrize("c", CASES, ids=[c.name for c in CASES])
def test_forward(api, c):
    """Kernel A forward only (backward == 0) on the features: outputs, argmax labels and the hit count."""
    model, net, params, X, _, labels = make_case(api, c)
    want = net.forward(params, X)
    got, acts = launched(lambda: model.classify_test(X))
    assert got == {A_FEATS: 1}, got
    assert_close(acts, want, what="classify_test")
    assert np.array_equal(model.classify_features(X), O.argmax_last(want))
    assert model.evaluate(X, labels) == O.accuracy(want, labels)


@gpu
@pytest.mark.parametrize("c", IMAGE_CASES, ids=[c.name for c in IMAGE_CASES])
def test_evaluate_images(api, c):
    """evaluate_images against the oracle, and against the training step's statistics on the same batch and parameters."""
    model, net, params, X, images, labels = make_case(api, c)
    want = net.forward(params, X)
    want_cost = 0.5 * float(np.sum((want - onehot(labels, c.classes)) ** 2))
    got, (acc, cost, lab) = launched(lambda: model.evaluate_images(images, labels, want_labels=True))
    if c.route == "unfit":
        feats = FEATS_STAGED if cp_plan(*plan_stages(c.cfg, *c.hw)[:2], *c.hw) else FEATS_GENERIC
        assert got == {feats: 1, A_FEATS: 1, "batch_stats_kernel": 1, "argmax_last_kernel": 1}, got
    else:
        assert got == {INFER_STAGED if c.route == "staged" else INFER_GENERIC: 1}, got
    assert acc == O.accuracy(want, labels)
    assert abs(cost - want_cost) <= 1e-9 * max(1.0, want_cost), (cost, want_cost)
    assert np.array_equal(lab, O.argmax_last(want))
    model.accumulate_gradients_images(images, labels)
    if c.route == "unfit":   # batch_stats_kernel adds the per-sample costs in another order than kernel A's tiles
        tc, th = model.last_batch_stats()
        assert th == acc and abs(tc - cost) <= 1e-12 * max(1.0, cost)
    else:
        assert model.last_batch_stats() == (cost, acc), "the inference kernel must add the partials as kernel B does"


# ---- ties: saturated outputs are exactly 1.0 -------------------------------------------------------------------------
TIE_CASES = [
    I("tie-784-30-10-B256", [1, 3], (28, 28), [30], 10, 256, "staged"),
    I("tie-784-4x32-B129", [1, 3], (28, 28), [32, 32, 32], 10, 129, "staged"),
]


@gpu
@pytest.mark.parametrize("c", TIE_CASES, ids=[c.name for c in TIE_CASES])
def test_tied_outputs(api, c):
    """Output weights scaled up until several outputs of a sample are exactly 1.0.  Such a sample is never a hit (its max
    set is not the one-hot), even when its label is one of the tied classes; its label is the LAST maximum; the output
    delta is an exact zero where a * (1 - a) == 0."""
    model, net, params, X, images, labels = make_case(api, c)
    # output layer rescaled so that every output's pre-activation is ~ N(0, 60^2) over the batch: above ~37 the sigmoid is
    # exactly 1.0, so about 27 % of the outputs saturate and most samples, but not all, tie
    ws, bs = net.unpack(params)
    n_hidden = sum(r * k + r for r, k in net.shapes[:-1])
    z = O.Net(net.shapes[:-1]).forward(params[:n_hidden], X) @ ws[-1].T + bs[-1]
    s = 60.0 / z.std(axis=0)
    ws[-1], bs[-1] = ws[-1] * s[:, None], (bs[-1] - z.mean(axis=0)) * s
    params = net.pack(ws, bs)
    model.set_params(params)
    want = net.forward(params, X)
    tied = (want == want.max(axis=1, keepdims=True)).sum(axis=1) > 1
    assert tied.sum() >= c.B // 4 and (~tied).sum() >= 8, int(tied.sum())
    pred = O.argmax_last(want)
    labels = np.where(tied | (np.arange(c.B) % 2 == 0), pred, labels)   # tied samples labelled with one of their maxima
    Y = onehot(labels, c.classes)
    want_hits = O.accuracy(want, labels)
    assert want_hits < int(np.sum(pred == labels)), "an argmax == label rule would count the tied samples"
    want_cost = 0.5 * float(np.sum((want - Y) ** 2))

    acc, cost, lab = model.evaluate_images(images, labels, want_labels=True)
    assert np.array_equal(lab, pred)
    assert acc == want_hits
    assert abs(cost - want_cost) <= 1e-9 * max(1.0, want_cost)

    want_params, want_grads = net.train_batch(params, X, Y, ETA)
    model.train_batch_images(images, labels, ETA)
    assert model.last_batch_stats() == (cost, acc)
    out = model.activations(net.n - 1)
    assert np.array_equal(out == 1.0, want == 1.0)
    assert np.all(model.deltas(net.n - 1)[out == 1.0] == 0.0)
    check_taps(model, net, params, X, Y, range(c.B), c.name)
    assert_close(model.get_gradients(), want_grads, what="sum dW/db")
    assert_close(model.get_params(), want_params, what="post-step parameters")


# ---- the streamed host epoch at 4 x 32 --------------------------------------------------------------------------------
@gpu
def test_train_epoch_host_4x32_equals_step_by_step(api):
    """train_epoch_host on pinned u8 images (kernel A with its front end ahead of the wait, the only one-GPU route to it)
    == train_batch_images batch by batch: parameters and per-step (cost, hits) bit for bit, remainder dropped."""
    import torch
    c = CASES[0]
    assert c.name == "staged-784-4x32-B129"
    B, N = c.B, 4 * c.B + 5
    rng = np.random.default_rng(31)
    images = torch.from_numpy(rng.integers(0, 256, size=(N, 28, 28), dtype=np.uint8)).pin_memory()
    labels = torch.from_numpy(rng.integers(0, c.classes, size=N).astype(np.int64)).pin_memory()
    model, _, params, _, _, _ = make_case(api, c)
    stats = []
    for k in range(N // B):
        model.train_batch_images(images.numpy()[k * B:(k + 1) * B], labels.numpy()[k * B:(k + 1) * B], ETA)
        stats.append(model.last_batch_stats())
    want_params = model.get_params()
    model.set_params(params)
    cost, hits = model.train_epoch_host(images.numpy(), labels.numpy(), B, ETA)
    assert len(cost) == N // B
    assert np.array_equal(model.get_params(), want_params)
    assert [(float(a), int(b)) for a, b in zip(cost, hits)] == stats
