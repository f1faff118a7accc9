"""The convolutional network with the softmax cross-entropy head (``ConvNet(..., head=Head.SoftmaxCrossEntropy)``,
``rcn_cuda_cnn_create_with_head``): an affine output layer, p = softmax(z), cost sum_b (log s + m) - z_label, delta_L = p - y,
hits and labels decided on the logits.

Oracle: oracle/ext.py (conv, pool, activation and softmax_xent from ext_oracle.cpp) composed with a numpy dense stack (sigmoid
hidden layers, affine output layer).  Dense weights are drawn N(0, 1/fan_in) so the logits stay moderate (|z| of a few units):
p, delta and the cost then carry the 1e-9 bar of conftest.assert_close like every other quantity."""
import ctypes as C
import os
import shutil
import socket
import subprocess
import tempfile

import numpy as np
import pytest

from conftest import assert_close

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ETA = 0.5


def _m():
    import mercer_research_b200 as m
    return m


def _profile(fn):
    from mercer_research_b200 import _lib
    _lib.profile_enable(True)
    fn()
    rep = _lib.profile_report()
    _lib.profile_enable(False)
    return sorted(rep)


def _init(net, seed):
    """He-scaled conv weights, dense weights N(0, 1/fan_in) and biases N(0, 0.01): moderate logits."""
    rng = np.random.default_rng(seed)
    p = np.zeros(net.n_params)
    for name, sl, shp in net.param_slices():
        n = sl.stop - sl.start
        if name.startswith("conv") and name.endswith(".w"):
            p[sl] = rng.standard_normal(n) * np.sqrt(2.0 / (shp[1] * shp[2] * shp[3]))
        elif name.endswith(".W"):
            p[sl] = rng.standard_normal(n) / np.sqrt(shp[1])
        elif name.startswith("dense"):
            p[sl] = rng.standard_normal(n) * 0.1
    net.set_params(p)
    return p


def _unpack(net, p):
    conv, Ws, bs = [], [], []
    for name, sl, shp in net.param_slices():
        v = p[sl]
        if name.endswith(".w"):
            conv.append([v.reshape(shp)])
        elif name.startswith("conv"):
            conv[-1].append(v.copy())
        elif name.endswith(".W"):
            Ws.append(v.reshape(shp[1], shp[0]).T.copy())
        else:
            bs.append(v.copy())
    return conv, Ws, bs


def _sigmoid(z):
    return 1.0 / (1.0 + np.exp(-z))


def oracle_forward(net, p, x):
    """Stack outputs, features (B, L), dense activations [a_0 = feats^T, ..., hidden], logits (classes, B)."""
    from oracle import ext as E
    conv, Ws, bs = _unpack(net, p)
    outs, ams, a, ci = [], [], x, 0
    for l in net.layers:
        if isinstance(l, _m().Conv):
            w, b = conv[ci]
            ci += 1
            a = E.conv2d_forward(a, w, b, int(l.padding), E.ACT_RELU)
            ams.append(None)
        else:
            a, am = E.pool2d_forward(a, int(l.padding), int(l.pooling))
            ams.append(am)
        outs.append(a)
    feats = a.reshape(x.shape[0], -1)
    acts = [feats.T]
    for W, b in zip(Ws[:-1], bs[:-1]):
        acts.append(_sigmoid(W @ acts[-1] + b[:, None]))
    z = Ws[-1] @ acts[-1] + bs[-1][:, None]
    return outs, ams, acts, z


def oracle_step(net, p, x, labels, eta):
    """One train_batch with the softmax head on f64 NHWC images."""
    from oracle import ext as E
    conv, Ws, bs = _unpack(net, p)
    outs, ams, acts, z = oracle_forward(net, p, x)
    B = x.shape[0]
    probs, loss, delta = E.softmax_xent(z.T, labels=labels)
    cost = float(np.sum(loss))
    onehot = np.zeros_like(z)
    ok = (labels >= 0) & (labels < z.shape[0])
    onehot[labels[ok], np.arange(B)[ok]] = 1.0
    hits = int(np.sum(np.all((z == z.max(axis=0)) == (onehot == 1.0), axis=0)))
    deltas = [None] * len(Ws)
    deltas[-1] = delta.T
    for l in range(len(Ws) - 2, -1, -1):
        a = acts[l + 1]
        deltas[l] = (Ws[l + 1].T @ deltas[l + 1]) * (a * (1.0 - a))
    gW = [d @ a.T for d, a in zip(deltas, acts)]
    gb = [d.sum(axis=1) for d in deltas]
    dX = (Ws[0].T @ deltas[0]).T
    g = dX.reshape(outs[-1].shape)
    conv_grads = []
    first_conv = min([i for i, l in enumerate(net.layers) if isinstance(l, _m().Conv)], default=len(net.layers))
    ci = len(conv)
    for li in range(len(net.layers) - 1, -1, -1):
        l = net.layers[li]
        x_in = x if li == 0 else outs[li - 1]
        if isinstance(l, _m().Pool):
            if li <= first_conv:
                break
            g = E.pool2d_backward(g, ams[li], x_in.shape[1:3], int(l.padding), int(l.pooling))
            continue
        ci -= 1
        dz = E.activation_backward(outs[li], g, E.ACT_RELU)
        dw, db = E.conv2d_backward_weight(x_in, dz, l.kh, l.kw, int(l.padding))
        conv_grads.insert(0, (dw, db))
        if li <= first_conv:
            break
        g = E.conv2d_backward_data(dz, conv[ci][0], x_in.shape[1:3], int(l.padding))
    flat = []
    for dw, db in conv_grads:
        flat += [dw.ravel(), db]
    for dw, db in zip(gW, gb):
        flat += [dw.T.ravel(), db]
    grads = np.concatenate(flat)
    return dict(grads=grads, new=p - (eta / B) * grads, cost=cost, hits=hits, outs=outs, dX=dX, z=z, acts=acts,
                deltas=deltas, p=probs.T, Ws=Ws, bs=bs)


def _argmax_last(z):
    from oracle import rcn_oracle_np as R
    return np.array([R.argmax_last(z[:, b]) for b in range(z.shape[1])], dtype=np.int64)


def _images(rng, B, shape, u8):
    if u8:
        return rng.integers(0, 256, size=(B,) + shape[:2], dtype=np.uint8)
    return rng.standard_normal((B,) + shape)


CASES = {
    # the narrow head that takes kernels A/B with the sigmoid head runs the generic path
    "u8_ff8": dict(shape=(12, 11, 1), u8=True, B=16, ff=[8], classes=10,
                   layers=lambda m: [m.Conv(4, 3, 3, m.Padding.Same), m.Pool(m.Pooling.Max, m.Padding.Same)],
                   kernels=["softmax_xent_head_kernel", "dense_logits_gemm", "conv2d_direct_small_u8_kernel",
                            "dense_input_grad_gemm"]),
    # no hidden layer: delta_0 is p - y itself; L = 8 * 8 * 5 = 320 (not a skinny shape)
    "f64_avg_ff0": dict(shape=(16, 16, 3), u8=False, B=64, ff=[], classes=10,
                        layers=lambda m: [m.Conv(5, 3, 3, m.Padding.Same), m.Pool(m.Pooling.Average, m.Padding.Same)],
                        kernels=["softmax_xent_head_kernel", "dense_logits_gemm", "dense_input_grad_gemm"]),
    # 10 x 512 output layer: the skinny forward kernel's logits instantiation
    "skinny": dict(shape=(8, 8, 2), u8=False, B=64, ff=[512], classes=10,
                   layers=lambda m: [m.Conv(4, 3, 3, m.Padding.Same), m.Pool(m.Pooling.Max, m.Padding.Same)],
                   kernels=["softmax_xent_head_kernel", "skinny_forward_kernel(logits)"]),
    # lanes stride the classes past 32
    "classes40": dict(shape=(12, 12, 1), u8=True, B=32, ff=[16], classes=40,
                      layers=lambda m: [m.Conv(4, 3, 3, m.Padding.Same), m.Pool(m.Pooling.Max, m.Padding.Same)],
                      kernels=["softmax_xent_head_kernel", "dense_logits_gemm"]),
    # p = 1: zero cost, delta = 0 for label 0
    "classes1": dict(shape=(8, 8, 1), u8=True, B=16, ff=[8], classes=1,
                     layers=lambda m: [m.Conv(2, 3, 3, m.Padding.Same), m.Pool(m.Pooling.Max, m.Padding.Same)],
                     kernels=["softmax_xent_head_kernel", "dense_logits_gemm"]),
}


def _build(case, seed=7, head=None):
    m = _m()
    c = CASES[case]
    head = m.Head.SoftmaxCrossEntropy if head is None else head
    net = m.ConvNet(c["shape"], c["layers"](m), c["ff"], c["classes"], head=head)
    return net, _init(net, seed)


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(CASES))
def test_softmax_step_matches_oracle(case):
    c = CASES[case]
    rng = np.random.default_rng(200 + len(case))
    net, p = _build(case)
    batches = [(_images(rng, c["B"], c["shape"], c["u8"]), rng.integers(0, c["classes"], c["B"]).astype(np.int64))
               for _ in range(3)]
    f64 = lambda img: img.astype(np.float64)[..., None] if c["u8"] else img

    img, lab = batches[0]
    kernels = _profile(lambda: (net.accumulate_gradients_images(img, lab), net.synchronize()))
    for k in c["kernels"]:
        assert any(n.startswith(k) for n in kernels), (k, kernels)
    for k in ("smallnet_", "batch_stats_kernel"):
        assert not any(n.startswith(k) for n in kernels), (k, kernels)
    want = oracle_step(net, p, f64(img), lab, ETA)
    got_g = net.get_gradients()
    for name, sl, _ in net.param_slices():
        assert_close(got_g[sl], want["grads"][sl], what=f"{case} sum d{name}")
    for i in range(len(net.layers)):
        assert_close(net.layer_output(i), want["outs"][i], what=f"{case} layer {i} output")
    assert_close(net.input_gradient(), want["dX"], what=f"{case} dX")
    cost, hits = net.last_batch_stats()
    assert hits == want["hits"]
    assert_close(cost, want["cost"], what=f"{case} batch cost")

    acc, ecost, labels_out = net.evaluate_images(img, lab, want_labels=True)
    assert np.array_equal(labels_out, _argmax_last(want["z"]))
    assert acc == want["hits"]
    assert_close(ecost, want["cost"], what=f"{case} evaluate cost")
    assert np.array_equal(net.classify_images(img), labels_out)

    net.apply_gradients(ETA, c["B"])
    p1 = net.get_params()
    assert_close(p1, want["new"], what=f"{case} params after one step")
    net2, _ = _build(case)
    net2.train_batch_images(img, lab, ETA)
    assert np.array_equal(net2.get_params(), p1), "accumulate + apply must equal train_batch"

    ref = want["new"]
    for img, lab in batches[1:]:
        net.train_batch_images(img, lab, ETA)
        ref = oracle_step(net, ref, f64(img), lab, ETA)["new"]
    assert_close(net.get_params(), ref, what=f"{case} params after three steps")


@pytest.mark.gpu
def test_softmax_tcgen05_logits():
    """ff [2048] -> 512 classes at B = 4096: the output layer's logits, its weight gradient and the hidden layer's
    backward-data GEMM take the tcgen05 integer-slice path; the rest runs in f64 (DMMA, direct conv).  Every quantity is held
    to the error bound that follows from the engines' documented guarantees (test_gpu_ozaki.py, DESIGN.md section 2), carried
    through the step as a per-element magnitude G of the possible error, in units of 1e-9:
      logits       the digit truncation is relative to the operand scales, so an error in z_i is bounded by the terms
                   T_i = (|W| |a| + |b|)_i, not by |z_i|;
      head         delta_i = p_i - y_i then moves by at most D_L = |delta| + p (T + sum_j p_j T_j); the batch cost by
                   sum_b (T_label + sum_i p_i T_i);
      tcgen05 GEMM the scale-unit bar, amax(A row) . sum|B col| + sum|A row| . amax(B col): the backward data D_0 =
                   unit(|W_1|^T, D_L) a (1 - a), and the output layer's dW = unit(D_L, |a|^T) (its delta rows are not alike
                   inside their unit: p ~ 1/512 for most samples and a -1 spike for each sample of that class);
      f64 GEMMs    componentwise on the carried bounds: the hidden dW = D_0 |a_0|^T, dX = |W_0|^T D_0, and the conv gradients
                   the conv backward-weight of |x| with dX through the pool backward and ReLU' (f64 rounding is far inside);
      biases       row sums of D.
    The post-step parameters p - (eta / B) g then differ from the oracle's by at most 1e-9 |p_new| (the update's own
    rounding) plus (eta / B) 1e-9 G.  conftest.assert_close alone would ask 1e-9 of a near-zero weight's own size, which the
    integer-slice engines do not guarantee (measured on B200: 9 of 1.1 M parameters, worst 1.9e-12 at a weight of -1.05e-4).
    Hits and labels are exact (no two top logits lie within the error)."""
    from oracle import ext as E
    m = _m()
    B = 4096
    net = m.ConvNet((8, 8, 1), [m.Conv(2, 3, 3, m.Padding.Same), m.Pool(m.Pooling.Max, m.Padding.Same)], [2048], 512,
                    head=m.Head.SoftmaxCrossEntropy)
    p = _init(net, 41)
    rng = np.random.default_rng(42)
    img = rng.integers(0, 256, size=(B, 8, 8), dtype=np.uint8)
    lab = rng.integers(0, 512, B).astype(np.int64)
    kernels = _profile(lambda: (net.accumulate_gradients_images(img, lab), net.synchronize()))
    for k in ("dense_logits_gemm(tcgen05", "dense_backward_data_gemm(tcgen05", "softmax_xent_head_kernel"):
        assert any(n.startswith(k) for n in kernels), (k, kernels)
    x = img.astype(np.float64)[..., None]
    want = oracle_step(net, p, x, lab, ETA)
    Ws, bs, acts, P = want["Ws"], want["bs"], want["acts"], want["p"]

    def unit(A, Bm):      # scale-unit bar of A @ Bm for nonnegative A, Bm: A's unit is a row, Bm's a column
        return A.max(axis=1)[:, None] * Bm.sum(axis=0)[None, :] + A.sum(axis=1)[:, None] * Bm.max(axis=0)[None, :]

    T = np.abs(Ws[-1]) @ np.abs(acts[-1]) + np.abs(bs[-1])[:, None]
    D_L = np.abs(want["deltas"][-1]) + P * (T + np.sum(P * T, axis=0))
    a1 = acts[1]
    D_0 = unit(np.abs(Ws[1]).T, D_L) * (a1 * (1.0 - a1))
    G = np.zeros(net.n_params)
    sl = {n: s for n, s, _ in net.param_slices()}
    G[sl["dense0.W"]] = (D_0 @ np.abs(acts[0]).T).T.ravel()            # column-major rows x cols
    G[sl["dense0.b"]] = D_0.sum(axis=1)
    G[sl["dense1.W"]] = unit(D_L, np.abs(acts[1]).T).T.ravel()
    G[sl["dense1.b"]] = D_L.sum(axis=1)
    outs, ams, _, _ = oracle_forward(net, p, x)
    conv, pool = net.layers
    dx = (np.abs(Ws[0]).T @ D_0).T.reshape(outs[1].shape)
    dz = E.activation_backward(outs[0], E.pool2d_backward(dx, ams[1], (8, 8), int(pool.padding), int(pool.pooling)), E.ACT_RELU)
    dw, db = E.conv2d_backward_weight(x, dz, conv.kh, conv.kw, int(conv.padding))
    G[sl["conv0.w"]] = dw.ravel()
    G[sl["conv0.b"]] = db

    g = net.get_gradients()
    for name, s in sl.items():
        ratio = np.abs(g[s] - want["grads"][s]) / np.maximum(G[s], 1e-300)
        assert np.all(ratio <= 1e-9), (f"sum d{name}", float(np.max(ratio)))
    cost, hits = net.last_batch_stats()
    assert hits == want["hits"]
    cost_terms = float(np.sum(T[lab, np.arange(B)] + np.sum(P * T, axis=0)))
    assert abs(cost - want["cost"]) <= 1e-9 * cost_terms, (cost, want["cost"], cost_terms)
    assert np.array_equal(net.classify_images(img), _argmax_last(want["z"]))
    net.apply_gradients(ETA, B)
    err = np.abs(net.get_params() - want["new"])
    bound = 1e-9 * np.abs(want["new"]) + (ETA / B) * 1e-9 * G
    assert np.all(err <= bound), ("params after one step", int(np.sum(err > bound)), float(np.max(err / bound)))


@pytest.mark.gpu
def test_softmax_gradient_is_the_cost_derivative():
    """Central differences of the evaluate_images batch cross-entropy agree with the gradient sums for conv weights, conv
    biases and dense weights of a tiny f64 network."""
    m = _m()
    net = m.ConvNet((8, 8, 2), [m.Conv(3, 3, 3, m.Padding.Same), m.Pool(m.Pooling.Max, m.Padding.None_),
                                m.Conv(2, 3, 3, m.Padding.Same), m.Pool(m.Pooling.Average, m.Padding.Same)], [5], 3,
                    head=m.Head.SoftmaxCrossEntropy)
    p = _init(net, 11)
    rng = np.random.default_rng(12)
    x = rng.standard_normal((4, 8, 8, 2))
    lab = rng.integers(0, 3, 4).astype(np.int64)
    net.accumulate_gradients_images(x, lab)
    g = net.get_gradients()

    def cost(q):
        net.set_params(q)
        return net.evaluate_images(x, lab)[1]

    sl = {n: s for n, s, _ in net.param_slices()}
    conv_w = [i for n, s in sl.items() if n.startswith("conv") and n.endswith(".w") for i in range(s.start, s.stop)]
    dense_w = [i for n, s in sl.items() if n.endswith(".W") for i in range(s.start, s.stop)]
    pick = (sorted(conv_w, key=lambda i: -abs(g[i]))[:4] + [sl["conv0.b"].start, sl["conv2.b"].start]
            + sorted(dense_w, key=lambda i: -abs(g[i]))[:4])
    h = 1e-5
    for i in pick:
        qp, qm = p.copy(), p.copy()
        qp[i] += h
        qm[i] -= h
        fd = (cost(qp) - cost(qm)) / (2 * h)
        assert abs(fd - g[i]) <= 1e-6 * max(abs(g[i]), abs(fd)) + 1e-9, (i, fd, g[i])


@pytest.mark.gpu
def test_softmax_stats_and_hit_rule():
    """last_batch_stats equals evaluate on the same batch bit for bit, classify equals evaluate's labels; the hit rule and
    the labels are decided on the logits: z = (0, 2^-60) rounds to p = (0.5, 0.5) but only label 1 is a hit, and with
    equal logits neither label is a hit and the label is the last tied class."""
    m = _m()
    net, _ = _build("classes40", seed=3)
    rng = np.random.default_rng(5)
    img = rng.integers(0, 256, size=(32, 12, 12), dtype=np.uint8)
    lab = rng.integers(0, 40, 32).astype(np.int64)
    net.accumulate_gradients_images(img, lab)
    cost, hits = net.last_batch_stats()
    acc, ecost, labels_out = net.evaluate_images(img, lab, want_labels=True)
    assert (acc, ecost) == (hits, cost)
    assert np.array_equal(net.classify_images(img), labels_out)

    tiny = m.ConvNet((4, 4, 1), [m.Pool(m.Pooling.Max, m.Padding.Same)], [], 2, head=m.Head.SoftmaxCrossEntropy)
    x = rng.standard_normal((2, 4, 4, 1))
    y = np.array([1, 0], dtype=np.int64)
    q = np.zeros(tiny.n_params)
    q[-1] = 2.0 ** -60
    tiny.set_params(q)
    acc, c, labels = tiny.evaluate_images(x, y, want_labels=True)
    assert acc == 1 and list(labels) == [1, 1]
    assert_close(c, 2 * np.log(2.0), what="cost of p = (0.5, 0.5)")
    tiny.accumulate_gradients_images(x[:1], y[:1])
    assert tiny.last_batch_stats()[1] == 1
    tiny.accumulate_gradients_images(x[1:], y[1:])
    assert tiny.last_batch_stats()[1] == 0
    q[-1] = 0.0
    tiny.set_params(q)
    acc, _, labels = tiny.evaluate_images(x, y, want_labels=True)
    assert acc == 0 and list(labels) == [1, 1]


def _dev(*arrays):
    import torch
    return [torch.as_tensor(a).cuda() for a in arrays]


@pytest.mark.gpu
@pytest.mark.parametrize("use_perm", [True, False], ids=["perm", "identity"])
@pytest.mark.parametrize("case", ["u8_ff8", "f64_avg_ff0"])
def test_softmax_epoch_steps_equal_train_batch(case, use_perm):
    """8 epoch steps over N = 3B + 5 samples (two wraps) equal train_batch_images on the chunks, bit for bit."""
    import torch
    c = CASES[case]
    B = c["B"]
    n, steps = 3 * B + 5, 8
    rng = np.random.default_rng(1)
    x = _images(rng, n, c["shape"], c["u8"])
    y = rng.integers(0, c["classes"], n).astype(np.int64)
    perm = np.random.default_rng(2).permutation(n) if use_perm else np.arange(n)
    xd, yd = _dev(x, y)
    pd = torch.as_tensor(perm).cuda() if use_perm else None
    (net, _), (ref, _) = _build(case), _build(case)
    net.epoch_bind(xd, yd, B, pd)
    pos = 0
    for k in range(steps):
        net.epoch_step(ETA)
        idx = perm[pos:pos + B]
        ref.train_batch_images(x[idx], y[idx], ETA)
        assert np.array_equal(net.get_params(), ref.get_params()), f"{case}: step {k} differs"
        assert net.last_batch_stats() == ref.last_batch_stats()
        pos += B
        if pos + B > n:
            pos = 0
        assert net.epoch_position() == pos


@pytest.mark.gpu
def test_softmax_graph_replay():
    """A captured epoch step replayed equals eager epoch steps bit for bit."""
    import torch
    c = CASES["f64_avg_ff0"]
    B, n = c["B"], 4 * c["B"]
    rng = np.random.default_rng(21)
    x = rng.standard_normal((n,) + c["shape"])
    y = rng.integers(0, 10, n).astype(np.int64)
    xd, yd = _dev(x, y)
    (eager, _), (graphed, _) = _build("f64_avg_ff0", seed=5), _build("f64_avg_ff0", seed=5)
    for net in (eager, graphed):
        net.epoch_bind(xd, yd, B)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        graphed.set_stream(side.cuda_stream)
        graphed.epoch_accumulate()            # sizes the buffers outside the capture
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        graphed.set_stream(torch.cuda.current_stream().cuda_stream)
        graphed.epoch_step(ETA)
    graphed.set_stream(-1)
    for _ in range(6):
        graph.replay()
        eager.epoch_step(ETA)
    torch.cuda.synchronize()
    assert np.array_equal(graphed.get_params(), eager.get_params())
    assert graphed.epoch_position() == eager.epoch_position()


@pytest.mark.gpu
def test_softmax_train_arrays_learns():
    """train_arrays with the softmax head lifts test accuracy on a separable set: the class is the brightest quadrant."""
    m = _m()
    rng = np.random.default_rng(9)

    def make(n):
        lab = rng.integers(0, 4, n).astype(np.int64)
        img = rng.integers(0, 64, size=(n, 12, 12)).astype(np.uint8)
        for i, c in enumerate(lab):
            r, s = divmod(int(c), 2)
            img[i, 6 * r:6 * r + 6, 6 * s:6 * s + 6] += 160
        return img, lab

    tr_x, tr_y = make(2048)
    te_x, te_y = make(512)
    net = m.ConvNet((12, 12, 1), [m.Conv(4, 3, 3, m.Padding.Same), m.Pool(m.Pooling.Max, m.Padding.Same)], [16], 4,
                    head=m.Head.SoftmaxCrossEntropy)
    _init(net, 10)
    before, _ = net.evaluate_images(te_x, te_y)
    hist = net.train_arrays(tr_x, tr_y, te_x, te_y, batch_size=64, epochs=3, eta=0.05, seed=3, log=None)
    assert hist[-1] >= 0.9 * len(te_y) and hist[-1] > before, (before, hist)


def _nccl_worker(rank, world, port, out_dir):
    import sys
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import torch
    import torch.distributed as dist
    from mercer_research_b200.trainer import DataParallelTrainer
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world,
                            device_id=torch.device("cuda", rank))
    m = _m()
    c = CASES["f64_avg_ff0"]
    net = m.ConvNet(c["shape"], c["layers"](m), c["ff"], c["classes"], device=rank, head=m.Head.SoftmaxCrossEntropy)
    _init(net, 31)
    trainer = DataParallelTrainer(net, eta=ETA, exchange="nccl")
    rng = np.random.default_rng(32)
    for _ in range(2):
        x = rng.standard_normal((128,) + c["shape"])
        y = rng.integers(0, 10, 128).astype(np.int64)
        trainer.step_global_images(torch.tensor(x, device="cuda"), torch.tensor(y, device="cuda"))
    torch.cuda.synchronize()
    np.save(os.path.join(out_dir, f"params_{rank}.npy"), net.get_params())
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.gpu
def test_softmax_nccl_two_gpus(tmp_path):
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mp.spawn(_nccl_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    p0, p1 = np.load(tmp_path / "params_0.npy"), np.load(tmp_path / "params_1.npy")
    assert np.array_equal(p0, p1), "replicas must stay bit-identical"
    m = _m()
    c = CASES["f64_avg_ff0"]
    ref = m.ConvNet(c["shape"], c["layers"](m), c["ff"], c["classes"], head=m.Head.SoftmaxCrossEntropy)
    _init(ref, 31)
    rng = np.random.default_rng(32)
    for _ in range(2):
        x = rng.standard_normal((128,) + c["shape"])
        y = rng.integers(0, 10, 128).astype(np.int64)
        ref.train_batch_images(x, y, ETA)
    assert_close(p0, ref.get_params(), rtol=1e-12, what="2-GPU NCCL vs 1 GPU on the global batch")


@pytest.mark.gpu
def test_default_head_is_the_plain_create():
    """create_with_head(..., SigmoidQuadratic) and rcn_cuda_cnn_create give bit-identical steps with the same kernels
    (kernels A/B on the narrow head)."""
    from mercer_research_b200 import _lib
    m = _m()
    c = CASES["u8_ff8"]

    def plain():
        net = m.ConvNet(c["shape"], c["layers"](m), c["ff"], c["classes"])
        net._lib.rcn_cuda_cnn_destroy(net._h)
        spec = [v for l in net.layers for v in l.spec()]
        ff = (C.c_size_t * 1)(*c["ff"])
        h = C.c_void_p()
        _lib.check(net._lib.rcn_cuda_cnn_create(0, 12, 11, 1, (C.c_int32 * len(spec))(*spec), len(net.layers), ff, 1, 10,
                                                C.byref(h)))
        net._h = h
        return net

    rng = np.random.default_rng(4)
    img = rng.integers(0, 256, size=(16, 12, 11), dtype=np.uint8)
    lab = rng.integers(0, 10, 16).astype(np.int64)
    runs = []
    for net in (m.ConvNet(c["shape"], c["layers"](m), c["ff"], c["classes"], head=m.Head.SigmoidQuadratic), plain()):
        _init(net, 8)
        ks = _profile(lambda: (net.train_batch_images(img, lab, ETA), net.synchronize()))
        runs.append((ks, net.get_params(), net.last_batch_stats()))
    assert runs[0][0] == runs[1][0]
    assert any(k.startswith("smallnet_fwd_bwd_kernel") for k in runs[0][0]), runs[0][0]
    assert np.array_equal(runs[0][1], runs[1][1]) and runs[0][2] == runs[1][2]


# -- CPU ----------------------------------------------------------------------------------------------------------------
def test_unknown_head_is_invalid_needs_no_gpu(built_library):
    """An unknown head is refused with RCN_ERR_INVALID before any device work."""
    lib = built_library
    spec = (C.c_int32 * 5)(0, 4, 3, 3, 1)
    ff = (C.c_size_t * 1)(8)
    for head in (2, -1, 100):
        h = C.c_void_p()
        assert lib.rcn_cuda_cnn_create_with_head(0, 8, 8, 1, spec, 1, ff, 1, 10, head, C.byref(h)) == 1, head
        assert not h.value
    with pytest.raises(ValueError):
        _m().ConvNet((8, 8, 1), [_m().Conv(4)], [8], 10, head=2)


def test_cpp_wrapper_takes_the_head():
    gxx = shutil.which("g++")
    if not gxx:
        pytest.skip("g++ not available")
    src = r'''
#include "rcn.hpp"
int main() {
    using L = rcn::ConvNet::Layer;
    rcn::ConvNet net(12, 11, 1, {L::conv(4, 3, 3, rcn::Padding::Same), L::pool(rcn::Pooling::Max, rcn::Padding::Same)}, {8}, 10, 0,
                     rcn::Head::SoftmaxCrossEntropy);
    std::vector<uint8_t> img(16 * 12 * 11);
    std::vector<int64_t> lab(16);
    net.train_batch(img.data(), RCN_PIXELS_U8_ROWMAJOR, lab.data(), 16, 12, 11, 0.5);
    return (int)(net.last_batch_stats().second + net.get_params().size());
}
'''
    with tempfile.TemporaryDirectory() as d:
        p = os.path.join(d, "head.cpp")
        open(p, "w").write(src)
        r = subprocess.run([gxx, "-std=c++17", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), "-c", p, "-o",
                            os.path.join(d, "head.o")], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
