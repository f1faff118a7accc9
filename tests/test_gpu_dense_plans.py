"""The f64 dense layers of csrc/dense.cu on every skinny, tile, split and reduction plan, the heads past one grid-stride
pass, and the skinny forward kernel's alignment condition.

Shapes are chosen with a restatement of the host plan (``skinny_layer``, ``launch_gemm_tiles``' tile rule, the split rules of
``launch_dense_backward_weight`` and ``split_plan``, both ``launch_bias_grad`` branches, ``use_tensor_cores``).  Every case is
driven through the public handles (``RCN`` and ``ConvNet``), prints its plan and asserts, with the library's launch
profiler, which kernels ran and how often.  The profiler gives both bias-gradient variants one name: the printed plan is
the record of which variant ran.  Every network has a layer wider than 32 (off the fused small-network kernels) and every
GEMM is off the tcgen05 path by shape; both are asserted.

Bars: own-magnitude 1e-9 (``assert_close``) against the C++ oracle (oracle ``Net``: ``train_batch`` with one thread,
``forward``, ``backprop``) for gradients, post-step parameters and batch costs, and against a numpy f64 restatement for
the activations and deltas of every sample.  Gradient sums over 20 000 samples or more are held componentwise: within 1e-9
of the same sums of |delta| |A|^T (DESIGN.md section 2).  Labels and hits are exact.  Cases that move more than 1 GB have
``large`` in their id."""
from collections import Counter

import numpy as np
import pytest

import oracle as O
from conftest import assert_close

NUM_SMS, KT, MAX_GRID_YZ = 148, 16, 65535
OZ_BM, OZ_BN, OZ_MAX_K = 128, 96, 16384
SK_MAX_ROWS = 16
ETA = 3.0


# -- the host plan, restated ---------------------------------------------------------------------------------------------
def cdiv(a, b):
    return -(-a // b)


def skinny_layer(M, K):
    return 1 <= M <= SK_MAX_ROWS and K >= 512 and K % 128 == 0


def use_tensor_cores(M, N, K):
    if K > OZ_MAX_K:
        return False
    tiles = cdiv(M, OZ_BM) * cdiv(N, OZ_BN)
    return M >= 256 and N >= 256 and K >= 512 and tiles >= NUM_SMS // 2 and M * N * K >= 4.0e9


def split_plan(K, splits):
    splits = max(splits, 1)
    kps = max(cdiv(cdiv(K, splits), KT) * KT, KT)
    return (cdiv(K, kps) if K > 0 else 1), kps


def gemm_tile(M, N, splits=1):
    if M <= 32:
        return (32, 128)
    return (128, 128) if cdiv(M, 128) * cdiv(N, 128) * splits >= NUM_SMS * 7 // 8 else (64, 64)


def bias_plan(M, N):
    """launch_bias_grad: (variant, column splits S)."""
    if M >= 256 and cdiv(M, 256) <= 1023:
        rb = cdiv(M, 256)
        S = max(min(cdiv(4 * NUM_SMS, rb), cdiv(N, 64)), 1)
        nps = cdiv(cdiv(N, S), 16) * 16
        return "wide", max(cdiv(N, nps), 1)
    rb = cdiv(M, 32)
    S = max(min(cdiv(4 * NUM_SMS, rb), cdiv(N, 256)), 1)
    nps = cdiv(cdiv(N, S), 32) * 32
    return "narrow", max(cdiv(N, nps), 1)


def wgrad_plan(M, N, Kb):
    """launch_dense_backward_weight for dW (M x N) = delta (M x Kb) A_prev^T: engine or tile, batch splits, bias plan."""
    bias = bias_plan(M, Kb)
    if skinny_layer(M, N):
        splits = max(min(cdiv(4 * NUM_SMS, cdiv(N, 256)), cdiv(Kb, 64)), 1)
        nps = cdiv(cdiv(Kb, splits), 16) * 16
        return dict(engine="skinny", splits=cdiv(Kb, nps), bias=bias)
    if M <= 32:
        tiles = cdiv(M, 32) * cdiv(N, 128)
    else:
        tiles = cdiv(M, 128) * cdiv(N, 128)
        if tiles < NUM_SMS:
            tiles = cdiv(M, 64) * cdiv(N, 64)
    splits = 1
    if tiles < NUM_SMS:
        splits = min(cdiv(2 * NUM_SMS, tiles), max(Kb // 64, 1), 64)
        big = cdiv(M, 128) * cdiv(N, 128) if M > 32 else 0
        if 0 < big < NUM_SMS:
            s_big = NUM_SMS // big
            if s_big >= 2 and Kb // s_big >= 256 and big * s_big >= NUM_SMS * 7 // 8:
                splits = s_big
    splits = split_plan(Kb, splits)[0]
    return dict(engine=gemm_tile(M, N, splits), splits=splits, bias=bias)


def _aligned(rows, l, B):
    """Layer l reads the feature buffer (l = 0) or act(l - 1, B): sum(rows[:l-1]) * B doubles into the activation buffer."""
    return l == 0 or sum(rows[:l - 1]) * B % 2 == 0


def plan(shapes, B):
    """Per layer: forward engine, backward-data engine (from the layer above), weight-gradient plan."""
    rows = [r for r, _ in shapes]
    out = []
    for l, (r, c) in enumerate(shapes):
        fwd = "skinny" if skinny_layer(r, c) and _aligned(rows, l, B) else gemm_tile(r, B)
        bwd = None
        if l + 1 < len(shapes):
            bwd = "skinny" if skinny_layer(rows[l + 1], r) else gemm_tile(r, B)
        out.append(dict(fwd=fwd, bwd=bwd, wgrad=wgrad_plan(r, c, B)))
    return out


def off_tensor_cores(shapes, B):
    rows = [r for r, _ in shapes]
    for l, (r, c) in enumerate(shapes):
        if use_tensor_cores(r, B, c) or use_tensor_cores(r, c, B):
            return False
        if l + 1 < len(shapes) and use_tensor_cores(r, B, rows[l + 1]):
            return False
    return True


def forward_kernels(shapes, B, logits=False):
    k = Counter()
    for l, p in enumerate(plan(shapes, B)):
        last = l + 1 == len(shapes)
        if p["fwd"] == "skinny":
            k["skinny_forward_kernel(logits)" if logits and last else "skinny_forward_kernel"] += 1
        else:
            k["dense_logits_gemm" if logits and last else "dense_forward_gemm"] += 1
    return k


def train_kernels(shapes, B):
    """What a sigmoid-head train_batch launches on the generic path."""
    k = forward_kernels(shapes, B)
    for p in plan(shapes, B):
        if p["bwd"] == "skinny":
            k["skinny_backward_data_kernel"] += cdiv(cdiv(B, 16), MAX_GRID_YZ)
        elif p["bwd"] is not None:
            k["dense_backward_data_gemm"] += 1
        w = p["wgrad"]
        if w["engine"] == "skinny":
            k["skinny_backward_weight_kernel"] += 1
            k["reduce_splits_kernel"] += 1      # the skinny branch always reduces, also one split
        else:
            k["dense_backward_weight_gemm"] += 1
            k["reduce_splits_kernel"] += w["splits"] > 1
        k["bias_grad_kernel"] += 1
    k["batch_stats_kernel"] += 1
    k["sgd_update_kernel"] += 1
    return +k


def test_plan_restatement_examples():
    """Hand-worked points of the plan, re-derived from dense.cu, so an edit of the restatement cannot drift silently."""
    assert wgrad_plan(10, 640, 333) == dict(engine="skinny", splits=6, bias=("narrow", 2))
    assert wgrad_plan(10, 512, 20000) == dict(engine="skinny", splits=250, bias=("narrow", 79))
    assert wgrad_plan(384, 640, 2048) == dict(engine=(64, 64), splits=5, bias=("wide", 32))
    assert wgrad_plan(256, 1024, 4096) == dict(engine=(128, 128), splits=9, bias=("wide", 64))     # c3's dW0: s_big
    assert wgrad_plan(10, 256, 4096)["engine"] == (32, 128) and wgrad_plan(10, 256, 4096)["splits"] == 64   # the cap
    assert wgrad_plan(1152, 384, 2048)["engine"] == (128, 128) and wgrad_plan(1152, 384, 2048)["splits"] == 5
    assert gemm_tile(1152, 2048) == (128, 128) and gemm_tile(1024, 2048) == (64, 64)
    assert split_plan(1000, 15) == (13, 80) and wgrad_plan(10, 100, 1000)["splits"] == 13
    assert bias_plan(1, 256) == ("narrow", 1) and bias_plan(255, 2000) == ("narrow", 8)
    assert bias_plan(256, 64) == ("wide", 1) and bias_plan(257, 2000) == ("wide", 32)
    assert not skinny_layer(17, 512) and not skinny_layer(16, 384) and not skinny_layer(16, 520) and skinny_layer(1, 1152)
    # the skinny forward reads act(l - 1) as double2: [33, 512] -> 10 at B = 333 starts layer 2 at an odd double
    assert plan([(33, 64), (512, 33), (10, 512)], 333)[2]["fwd"] == (32, 128)
    assert plan([(33, 64), (512, 33), (10, 512)], 334)[2]["fwd"] == "skinny"
    assert not use_tensor_cores(256, 4096, 1024) and use_tensor_cores(2048, 4096, 1024)


# -- helpers ---------------------------------------------------------------------------------------------------------------
def _m():
    import mercer_research_b200 as m
    return m


def _profile(fn):
    """{kernel name: launches} of everything the library launched inside fn."""
    from mercer_research_b200 import _lib
    _lib.profile_enable(True)
    try:
        out = fn()
        rep = _lib.profile_report()
    finally:
        _lib.profile_enable(False)
    return out, Counter({k: v["launches"] for k, v in rep.items()})


def _assert_generic(k):
    assert not any(n.startswith("smallnet") or "tcgen05" in n for n in k), k


def _params(shapes, rng, bias=0.1):
    """W ~ N(0, 1 / fan_in), b ~ N(0, bias^2): unsaturated units, so every delta carries information."""
    parts = []
    for r, c in shapes:
        parts += [rng.standard_normal(r * c) / np.sqrt(c), rng.standard_normal(r) * bias]
    return np.concatenate(parts)


def _sigmoid(z):
    return 1.0 / (1.0 + np.exp(-z))


def _np_step(net, params, X, Y):
    """numpy f64 restatement of one sigmoid-head step: activations, deltas (B, rows) per layer and the componentwise
    gradient bound (sums of |delta| |A|^T in the flat layout)."""
    Ws, bs = net.unpack(params)
    acts, a = [], X
    for W, b in zip(Ws, bs):
        a = _sigmoid(a @ W.T + b)
        acts.append(a)
    deltas = [None] * len(Ws)
    deltas[-1] = (acts[-1] - Y) * acts[-1] * (1 - acts[-1])
    for l in range(len(Ws) - 2, -1, -1):
        deltas[l] = (deltas[l + 1] @ Ws[l + 1]) * acts[l] * (1 - acts[l])
    bound = []
    for l, d in enumerate(deltas):
        a_prev = X if l == 0 else acts[l - 1]
        bound += [(np.abs(d).T @ np.abs(a_prev)).T.ravel(), np.abs(d).sum(0)]
    return acts, deltas, np.concatenate(bound)


def _grads_close(got, want, bound, B, what):
    if B >= 20000:
        bad = np.abs(got - want) > 1e-9 * bound
        assert not bad.any(), f"{what}: {int(bad.sum())} sums off the componentwise bar"
    else:
        assert_close(got, want, what=what)


def _rcn(hidden, classes, n_in, seed):
    m = _m()
    model = m.RCN(classes, [], hidden)
    model.load_weights_and_bias(n_in)
    net = O.Net(model.layer_shapes)
    params = _params(net.shapes, np.random.default_rng(seed))
    model.set_params(params)
    return model, net, params


def _inputs(B, n_in, classes, seed):
    rng = np.random.default_rng(seed)
    return rng.standard_normal((B, n_in)), rng.integers(0, classes, B).astype(np.int64)


def _check_step(model, net, params, X, labels, what, extra=None):
    """classify_features, evaluate and one train_batch against the oracle, every layer's activations and deltas of every
    sample, and the launches against the restated plan.  Returns the post-step parameters."""
    B = X.shape[0]
    shapes = net.shapes
    classes = shapes[-1][0]
    Y = np.eye(classes)[labels]
    p = plan(shapes, B)
    print(what, "B", B, shapes, p)
    assert any(r > 32 for r, _ in shapes) and off_tensor_cores(shapes, B)

    want_out = net.forward(params, X)
    lab, k = _profile(lambda: model.classify_features(X))
    assert k == forward_kernels(shapes, B) + Counter({"argmax_last_kernel": 1}), k
    assert np.array_equal(lab, O.argmax_last(want_out)), f"{what}: labels"
    hits, k = _profile(lambda: model.evaluate(X, labels))
    assert k == forward_kernels(shapes, B) + Counter({"batch_stats_kernel": 1}), k
    assert hits == O.accuracy(want_out, labels), f"{what}: evaluate"

    want_params, want_grads = net.train_batch(params, X, Y, ETA, n_threads=1)
    _, k = _profile(lambda: model.train_batch(X, ETA, labels=labels))
    assert k == train_kernels(shapes, B) + Counter(extra or {}), (k, train_kernels(shapes, B))
    _assert_generic(k)

    acts, deltas, bound = _np_step(net, params, X, Y)
    for l in range(len(shapes)):
        assert_close(model.activations(l), acts[l], what=f"{what}: a[{l}]")
        assert_close(model.deltas(l), deltas[l], what=f"{what}: delta[{l}]")
    for b in sorted({0, B // 2, B - 1}):
        _, _, oa, od = net.backprop(params, X[b], Y[b])
        o = 0
        for l, (r, _) in enumerate(shapes):
            assert_close(model.activations(l)[b], oa[o:o + r], what=f"{what}: oracle a[{l}][{b}]")
            assert_close(model.deltas(l)[b], od[o:o + r], what=f"{what}: oracle delta[{l}][{b}]")
            o += r
    _grads_close(model.get_gradients(), want_grads, bound, B, f"{what}: sum dW / db")
    assert_close(model.get_params(), want_params, what=f"{what}: post-step params")
    cost, hits = model.last_batch_stats()
    assert hits == O.accuracy(want_out, labels), f"{what}: hits"
    assert abs(cost - 0.5 * np.sum((want_out - Y) ** 2)) <= 1e-9 * abs(cost), (what, cost)
    return want_params


# -- 1. skinny kernels at every row count ------------------------------------------------------------------------------------
SKINNY_KS = (512, 640, 1152)          # K / 8 per warp = 4, 5 and 9 sixteen-wide blocks
SKINNY_BS = (1, 31, 33, 333)


@pytest.mark.gpu
@pytest.mark.parametrize("M", range(1, SK_MAX_ROWS + 1))
def test_skinny_output_layer_every_row_count(M):
    K, B = SKINNY_KS[M % 3], SKINNY_BS[M % 4]
    model, net, params = _rcn([K], M, 64, seed=100 + M)
    try:
        p = plan(net.shapes, B)[1]
        assert p["fwd"] == "skinny" and p["wgrad"]["engine"] == "skinny" and plan(net.shapes, B)[0]["bwd"] == "skinny"
        X, labels = _inputs(B, 64, M, 200 + M)
        _check_step(model, net, params, X, labels, f"skinny M={M} K={K}")
    finally:
        model.close()


@pytest.mark.gpu
def test_skinny_hidden_layer():
    """512 -> [16, 64] -> 10: the skinny forward without an output delta, and a hidden layer's skinny weight gradient."""
    model, net, params = _rcn([16, 64], 10, 512, seed=7)
    try:
        p = plan(net.shapes, 333)
        assert p[0]["fwd"] == "skinny" and p[0]["wgrad"]["engine"] == "skinny" and p[1]["fwd"] != "skinny"
        X, labels = _inputs(333, 512, 10, 8)
        _check_step(model, net, params, X, labels, "skinny hidden")
    finally:
        model.close()


@pytest.mark.gpu
@pytest.mark.parametrize("M,K", [(17, 512), (16, 384), (16, 520)], ids=["M17-K512", "M16-K384", "M16-K520"])
def test_shapes_that_leave_the_skinny_path(M, K):
    """The DMMA GEMMs run, and no skinny_* kernel does (the launch multiset of _check_step)."""
    model, net, params = _rcn([K], M, 64, seed=M + K)
    try:
        assert plan(net.shapes, 100)[1] == dict(fwd=(32, 128), bwd=None, wgrad=wgrad_plan(M, K, 100))
        assert plan(net.shapes, 100)[0]["bwd"] == (64, 64) and wgrad_plan(M, K, 100)["engine"] == (32, 128)
        X, labels = _inputs(100, 64, M, K)
        _check_step(model, net, params, X, labels, f"not skinny M={M} K={K}")
    finally:
        model.close()


@pytest.mark.gpu
@pytest.mark.parametrize("B", [333, 334])
def test_skinny_forward_on_a_misaligned_input(B):
    """[33, 512] -> 10: layer 2 reads act(1) at 33 * B doubles.  At B = 333 that is 8 bytes off a 16-byte boundary, and
    the layer takes the DMMA GEMM; at B = 334 the skinny kernel.  The skinny backward kernels run at both."""
    model, net, params = _rcn([33, 512], 10, 64, seed=B)
    try:
        p = plan(net.shapes, B)
        assert p[2]["fwd"] == ("skinny" if B % 2 == 0 else (32, 128))
        assert p[1]["bwd"] == "skinny" and p[2]["wgrad"]["engine"] == "skinny"
        X, labels = _inputs(B, 64, 10, B + 1)
        _check_step(model, net, params, X, labels, f"misaligned B={B}")
    finally:
        model.close()


def _pool_features(x):
    """Max pool 2 x 2 (Same padding on an even map) of NHWC images, flattened per image."""
    B, H, W, C = x.shape
    return x.reshape(B, H // 2, 2, W // 2, 2, C).max(axis=(2, 4)).reshape(B, -1)


def _softmax_ref(net, p, x, labels):
    """numpy f64 softmax-head step on a pool-only ConvNet: grads, cost (and sum of |per-sample terms|), hits, labels, dX."""
    Ws, bs = [], []
    for name, sl, shp in net.param_slices():
        (Ws.append(p[sl].reshape(shp[1], shp[0]).T) if name.endswith(".W") else bs.append(p[sl]))
    feats = _pool_features(x)
    acts = [feats]
    for W, b in zip(Ws[:-1], bs[:-1]):
        acts.append(_sigmoid(acts[-1] @ W.T + b))
    z = acts[-1] @ Ws[-1].T + bs[-1]
    B, n = z.shape
    zm = z.max(axis=1, keepdims=True)
    lse = zm[:, 0] + np.log(np.exp(z - zm).sum(axis=1))
    prob = np.exp(z - lse[:, None])
    loss = lse - z[np.arange(B), labels]
    onehot = np.eye(n)[labels]
    deltas = [None] * len(Ws)
    deltas[-1] = prob - onehot
    for l in range(len(Ws) - 2, -1, -1):
        deltas[l] = (deltas[l + 1] @ Ws[l + 1]) * acts[l + 1] * (1 - acts[l + 1])
    grads, bound = [], []
    for d, a in zip(deltas, acts):
        grads += [(d.T @ a).T.ravel(), d.sum(0)]
        bound += [(np.abs(d).T @ np.abs(a)).T.ravel(), np.abs(d).sum(0)]
    hits = int(np.sum(np.all((z == z.max(axis=1, keepdims=True)) == (onehot == 1.0), axis=1)))
    lab = n - 1 - np.argmax(z[:, ::-1], axis=1)                 # last maximal element
    return dict(grads=np.concatenate(grads), bound=np.concatenate(bound), cost=float(loss.sum()),
                abs_cost=float(np.abs(loss).sum()), hits=hits, labels=lab, dX=deltas[0] @ Ws[0], ff=[W.shape for W in Ws])


def _softmax_net(ff, classes, seed, shape=(4, 4, 4)):
    m = _m()
    net = m.ConvNet(shape, [m.Pool(m.Pooling.Max, m.Padding.Same)], ff, classes, head=m.Head.SoftmaxCrossEntropy)
    rng = np.random.default_rng(seed)
    p = np.zeros(net.n_params)
    for name, sl, shp in net.param_slices():
        p[sl] = rng.standard_normal(sl.stop - sl.start) * (1 / np.sqrt(shp[1]) if name.endswith(".W") else 0.1)
    net.set_params(p)
    return net, p


def _check_softmax_step(net, p, x, labels, what, want_kernels):
    B = x.shape[0]
    want = _softmax_ref(net, p, x, labels)
    shapes = [(r, c) for r, c in want["ff"]]
    print(what, "B", B, shapes, plan(shapes, B))
    assert any(r > 32 for r, _ in shapes) and off_tensor_cores(shapes, B)
    _, k = _profile(lambda: (net.accumulate_gradients_images(x, labels), net.synchronize()))
    for name in want_kernels:
        assert k[name] == 1, (name, k)
    assert k["softmax_xent_head_kernel"] == 1 and "batch_stats_kernel" not in k, k
    _assert_generic(k)
    got = net.get_gradients()
    if B >= 20000:
        _grads_close(got, want["grads"], want["bound"], B, f"{what}: grads")
    else:
        assert_close(got, want["grads"], what=f"{what}: grads")
    assert_close(net.input_gradient(), want["dX"], what=f"{what}: per-sample dX = W0^T delta0")
    cost, hits = net.last_batch_stats()
    assert hits == want["hits"], (what, hits, want["hits"])
    assert abs(cost - want["cost"]) <= 1e-9 * want["abs_cost"], (what, cost, want["cost"])
    acc, ecost, lab = net.evaluate_images(x, labels, want_labels=True)
    assert acc == hits and ecost == cost, (what, acc, ecost, hits, cost)
    assert np.array_equal(lab, want["labels"]), f"{what}: labels"
    assert np.array_equal(net.classify_images(x), want["labels"]), f"{what}: classify labels"
    return want


@pytest.mark.gpu
@pytest.mark.parametrize("B", [333, 334])
def test_skinny_logits_on_a_misaligned_input(B):
    """ConvNet with ff [33, 512] and the softmax head: the logits layer reads act(1) at 33 * B doubles, so B = 333 takes
    dense_logits_gemm and B = 334 skinny_forward_kernel(logits)."""
    net, p = _softmax_net([33, 512], 10, seed=B)
    try:
        rng = np.random.default_rng(B)
        x, labels = rng.standard_normal((B, 4, 4, 4)), rng.integers(0, 10, B).astype(np.int64)
        logits = "skinny_forward_kernel(logits)" if B % 2 == 0 else "dense_logits_gemm"
        _check_softmax_step(net, p, x, labels, f"softmax misaligned B={B}",
                            [logits, "skinny_backward_data_kernel", "skinny_backward_weight_kernel"])
        _, k = _profile(lambda: net.classify_images(x))
        assert k[logits] == 1, k
    finally:
        net.close()


# -- 2. DMMA dense plans -------------------------------------------------------------------------------------------------------
TILE_CASES = {
    # id: (n_in, hidden, classes, B)
    "tile32-64": (48, [129, 65, 64, 33, 20], 10, 200),     # forward / backward-data at M = 129, 65, 64, 33 and 20, 10
    "tile128": (384, [1152, 384], 10, 2048),               # 9 x 16 = 144 big tiles: forward and backward-data of layer 0
}


@pytest.mark.gpu
@pytest.mark.parametrize("cid", list(TILE_CASES))
def test_dmma_tiles(cid):
    n_in, hidden, classes, B = TILE_CASES[cid]
    model, net, params = _rcn(hidden, classes, n_in, seed=len(cid))
    try:
        p = plan(net.shapes, B)
        fwd = {r: q["fwd"] for (r, _), q in zip(net.shapes, p)}
        if cid == "tile32-64":
            assert all(fwd[r] == (64, 64) for r in (129, 65, 64, 33)) and fwd[20] == fwd[10] == (32, 128)
            assert [q["bwd"] for q in p[:-1]] == [(64, 64)] * 4 + [(32, 128)]
        else:
            assert p[0]["fwd"] == p[0]["bwd"] == (128, 128) and p[0]["wgrad"]["engine"] == (128, 128)
        X, labels = _inputs(B, n_in, classes, B)
        _check_step(model, net, params, X, labels, cid)
    finally:
        model.close()


WGRAD_CASES = {
    # id: (n_in, hidden, classes, B, layer, expected (engine, splits))
    "one-split": (1024, [640], 10, 333, 0, ((64, 64), 1)),             # 10 x 16 = 160 tiles >= 148
    "capped-by-batch": (64, [200], 10, 200, 0, ((64, 64), 3)),          # 200 / 64 = 3 splits
    "cap-64": (1024, [256], 10, 4096, 1, ((32, 128), 64)),             # c3's last layer: 148 -> 64
    "s_big": (1024, [256], 10, 4096, 0, ((128, 128), 9)),              # c3's dW0: one wave of 16 big tiles x 9
    "lowered": (64, [100], 10, 1000, 1, ((32, 128), 13)),              # 15 splits -> split_plan -> 13
}


@pytest.mark.gpu
@pytest.mark.parametrize("cid", list(WGRAD_CASES))
def test_dmma_weight_gradient_splits(cid):
    n_in, hidden, classes, B, layer, (engine, splits) = WGRAD_CASES[cid]
    model, net, params = _rcn(hidden, classes, n_in, seed=len(cid) + 50)
    try:
        w = plan(net.shapes, B)[layer]["wgrad"]
        assert (w["engine"], w["splits"]) == (engine, splits), w
        X, labels = _inputs(B, n_in, classes, B + 3)
        _check_step(model, net, params, X, labels, cid)
        g1 = model.get_gradients()
        model.set_params(params)
        model.train_batch(X, ETA, labels=labels)
        assert np.array_equal(model.get_gradients(), g1), "split-K weight gradient is not run-to-run identical"
    finally:
        model.close()


# -- 3. reductions and their tickets ---------------------------------------------------------------------------------------
BIAS_CASES = {
    # id: (hidden, classes, B): the rows and bias plans each covers
    "M1-M255-S1": ([255], 1, 200),
    "M1-M255-S8": ([255], 1, 2000),
    "M256-M257-S1": ([256, 257], 10, 64),
    "M256-M257-S32": ([256, 257], 10, 2000),
}


@pytest.mark.gpu
@pytest.mark.parametrize("cid", list(BIAS_CASES))
def test_bias_gradient_variants(cid):
    hidden, classes, B = BIAS_CASES[cid]
    model, net, params = _rcn(hidden, classes, 48, seed=len(cid) + 70)
    try:
        bias = {r: wgrad_plan(r, c, B)["bias"] for r, c in net.shapes}
        many = not cid.endswith("S1")
        for r in (1, 255, 256, 257):
            if r in bias:
                assert bias[r][0] == ("wide" if r >= 256 else "narrow") and (bias[r][1] > 1) == many, bias
        X, labels = _inputs(B, 48, classes, B + 5)
        _check_step(model, net, params, X, labels, cid)
    finally:
        model.close()


@pytest.mark.gpu
def test_large_bias_tickets_reset_across_batches():
    """One model trained at B = 333, 20 000, 333: the skinny layer's bias reduction uses 2, 79 and 2 column splits on the
    same row block, and the 512-row layer's 6, 250 and 6, so a ticket left set by one launch would break the next.  The
    20 000-sample step also reduces 250 skinny weight-gradient splits (not a multiple of 8)."""
    model, net, params = _rcn([512], 10, 64, seed=90)
    try:
        plans = [wgrad_plan(10, 512, B) for B in (333, 20000)]
        assert [q["bias"] for q in plans] == [("narrow", 2), ("narrow", 79)] and plans[1]["splits"] == 250
        assert [bias_plan(512, B) for B in (333, 20000)] == [("wide", 6), ("wide", 250)]
        p = params
        for i, B in enumerate((333, 20000, 333)):
            X, labels = _inputs(B, 64, 10, 300 + i)
            p = _check_step(model, net, p, X, labels, f"ticket step {i}")
            model.set_params(p)       # the next step starts from the oracle's parameters
    finally:
        model.close()


# -- 4. heads and statistics -----------------------------------------------------------------------------------------------
def _saturating_net(B, seed):
    """40 -> [40] -> 10 whose output units saturate to exactly 1.0 where a feature is 1: hidden unit c = sigmoid(100 x_c
    - 50), output c = sigmoid(100 h_c - 40 + small) (z near 60: exactly 1.0; near -40: tiny).  Samples of kind 2 saturate
    two classes (label = the later one: never a hit), kind 1 one class (a hit iff it is the label), kind 0 none
    (x_c = 0.5 gives moderate outputs)."""
    rng = np.random.default_rng(seed)
    C, H, L = 10, 40, 40
    W0 = np.zeros((H, L))
    W0[np.arange(C), np.arange(C)] = 100.0
    W0[C:, C:] = rng.standard_normal((H - C, L - C)) / np.sqrt(L - C)
    b0 = np.zeros(H)
    b0[:C] = -50.0
    W1 = rng.standard_normal((C, H)) * 0.05
    W1[np.arange(C), np.arange(C)] = 100.0
    b1 = np.full(C, -40.0)
    net = O.Net([(H, L), (C, H)])
    params = net.pack([W0, W1], [b0, b1])
    X = np.zeros((B, L))
    X[:, C:] = rng.standard_normal((B, L - C))
    kind = rng.integers(0, 3, B)
    labels = rng.integers(0, C, B).astype(np.int64)
    for b in range(B):
        if kind[b] == 2:
            c1, c2 = sorted(rng.choice(C, 2, replace=False))
            X[b, [c1, c2]] = 1.0
            labels[b] = c2
        elif kind[b] == 1:
            c = rng.integers(0, C)
            X[b, c] = 1.0
            if rng.random() < 0.5:
                labels[b] = c
        else:
            X[b, :C] = 0.5 * (rng.random(C) < 0.5)
    return net, params, X, labels, kind


@pytest.mark.gpu
def test_batch_stats_with_saturated_outputs():
    B = 600                                        # three batch_stats CTAs
    net, params, X, labels, kind = _saturating_net(B, 11)
    out = net.forward(params, X)
    n_one = (out == 1.0).sum(axis=1)
    assert np.array_equal(n_one, kind), "construction: saturation to exactly 1.0 where intended"
    want_hits = O.accuracy(out, labels)
    assert want_hits == int(np.sum((kind == 1) & (out[np.arange(B), labels] == 1.0)) +
                            np.sum((kind == 0) & (O.argmax_last(out) == labels)))
    model = _m().RCN(10, [], [40])
    try:
        model.load_weights_and_bias(40)
        model.set_params(params)
        _check_step(model, net, params, X, labels, "saturated stats")
    finally:
        model.close()


@pytest.mark.gpu
def test_large_argmax_past_one_pass():
    """classify_features at B = 200 000: argmax_last_kernel's 1 184 x 128 threads take two grid-stride passes; samples
    with two outputs at exactly 1.0 check the last-maximum rule on both passes."""
    B = 200000
    net, params, X, labels, kind = _saturating_net(B, 12)
    model = _m().RCN(10, [], [40])
    try:
        model.load_weights_and_bias(40)
        model.set_params(params)
        want = O.argmax_last(net.forward(params, X))
        lab, k = _profile(lambda: model.classify_features(X))
        assert k == Counter({"dense_forward_gemm": 2, "argmax_last_kernel": 1}), k
        assert np.array_equal(lab, want)
        assert (want[kind == 2] == labels[kind == 2]).all()     # the later of the two saturated classes
    finally:
        model.close()


@pytest.mark.gpu
@pytest.mark.parametrize("classes", [1, 32, 33, 1000])
def test_large_softmax_head_past_one_pass(classes):
    """softmax_xent_head_kernel at B = 9 500: 1 184 CTAs x 8 warps hold 9 472 samples, so 28 warps add a second sample
    to their cost and hits."""
    B = 9500
    net, p = _softmax_net([40], classes, seed=classes)
    try:
        rng = np.random.default_rng(classes + 1)
        x, labels = rng.standard_normal((B, 4, 4, 4)), rng.integers(0, classes, B).astype(np.int64)
        _check_softmax_step(net, p, x, labels, f"softmax classes={classes}", ["dense_logits_gemm"])
    finally:
        net.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 32, 33])
def test_ext_softmax_xent_past_one_pass(n):
    from mercer_research_b200 import ext
    B = 20000
    rng = np.random.default_rng(n)
    z = rng.standard_normal((B, n)) * 4
    labels = rng.integers(0, n, B).astype(np.int64)
    (prob, loss, delta), k = _profile(lambda: ext.softmax_xent(z, labels=labels))
    assert k == Counter({"ext_softmax_xent_kernel": 1}), k
    zm = z.max(axis=1, keepdims=True)
    lse = zm[:, 0] + np.log(np.exp(z - zm).sum(axis=1))
    want_p = np.exp(z - lse[:, None])
    assert_close(prob, want_p, what="p")
    assert_close(loss, lse - z[np.arange(B), labels], what="loss")
    assert_close(delta, want_p - np.eye(n)[labels], what="delta")
