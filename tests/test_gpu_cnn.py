"""The convolutional network handle (csrc/cnn.cu, mercer_research_b200/cnn.py): learned conv / pool layers trained through
the extension kernels in front of the reference's dense stack.

Oracle: oracle/ext.py (conv, pool, activation from ext_oracle.cpp) composed with oracle/rcn_oracle_np for the dense part and
numpy for dX = W0^T delta0.  The case with the tcgen05 conv paths is checked against the library's own ops instead, bit for
bit (the integer-slice kernels have their own bars in test_gpu_ozaki.py)."""
import os
import shutil
import socket
import subprocess

import numpy as np
import pytest

from conftest import assert_close

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _m():
    import mercer_research_b200 as m
    return m


# -- oracle composition ---------------------------------------------------------------------------------------------------
def _unpack(net, p):
    """conv [(w, b)] in stack order, dense ([W], [b]) with W rows x cols."""
    conv, Ws, bs = [], [], []
    for name, sl, shp in net.param_slices():
        v = p[sl]
        if name.endswith(".w"):
            conv.append([v.reshape(shp)])
        elif name.startswith("conv"):
            conv[-1].append(v.copy())
        elif name.endswith(".W"):
            Ws.append(v.reshape(shp[1], shp[0]).T.copy())     # column-major rows x cols
        else:
            bs.append(v.copy())
    return conv, Ws, bs


def oracle_step(net, p, x, labels, eta):
    """One train_batch of the network on f64 NHWC images: (grads, new params, cost, hits, layer outputs, dX)."""
    from oracle import ext as E
    from oracle import rcn_oracle_np as R
    conv, Ws, bs = _unpack(net, p)
    B = x.shape[0]
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
    feats = a.reshape(B, -1)
    Y = np.eye(net.classes)[labels]
    gW = [np.zeros_like(W) for W in Ws]
    gb = [np.zeros_like(b) for b in bs]
    dX = np.zeros_like(feats)
    cost, hits = 0.0, 0
    for i in range(B):
        db, dw, _, acts, deltas = R.backprop(Ws, bs, feats[i], Y[i])
        gW = [g + d for g, d in zip(gW, dw)]
        gb = [g + d for g, d in zip(gb, db)]
        dX[i] = Ws[0].T @ deltas[0]
        cost += 0.5 * float(np.sum((acts[-1] - Y[i]) ** 2))
        hits += int(R.accuracy_hit(acts[-1], labels[i]))
    # down the stack
    g = dX.reshape(outs[-1].shape)
    conv_grads = []
    first_conv = min(i for i, l in enumerate(net.layers) if isinstance(l, _m().Conv))
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
    new = p - (eta / B) * grads
    return grads, new, cost, hits, outs, dX


def _rng_images(rng, B, shape, u8):
    if u8:
        return rng.integers(0, 256, size=(B,) + shape[:2], dtype=np.uint8)
    return rng.standard_normal((B,) + shape)


def _profile(fn):
    from mercer_research_b200 import _lib
    _lib.profile_enable(True)
    fn()
    kernels = sorted(_lib.profile_report())
    _lib.profile_enable(False)
    return kernels


CASES = {
    # direct conv kernel reading u8 pixels, fused narrow dense head (kernels A/B)
    "A": dict(shape=(12, 11, 1), u8=True, B=16, ff=[8], classes=10,
              layers=lambda m: [m.Conv(4, 3, 3, m.Padding.Same), m.Pool(m.Pooling.Max, m.Padding.Same)],
              kernels=["conv2d_direct_small_u8_kernel", "smallnet_fwd_bwd_kernel", "ext_pool_backward_kernel",
                       "conv2d_backward_weight_igemm", "dense_input_grad_gemm"]),
    # direct conv + DMMA implicit GEMM, generic dense path
    "B": dict(shape=(16, 16, 3), u8=False, B=64, ff=[64], classes=10,
              layers=lambda m: [m.Conv(16, 3, 3, m.Padding.Same), m.Pool(m.Pooling.Max, m.Padding.None_),
                                m.Conv(32, 3, 3, m.Padding.None_), m.Pool(m.Pooling.Average, m.Padding.Same)],
              kernels=["conv2d_direct_small_kernel", "conv2d_forward_igemm", "conv2d_backward_data_igemm",
                       "dense_forward_gemm", "dense_input_grad_gemm", "activation_backward_kernel"]),
}


def _build(case, seed=7):
    m = _m()
    c = CASES[case]
    net = m.ConvNet(c["shape"], c["layers"](m), c["ff"], c["classes"])
    p = net.init_params(np.random.default_rng(seed))
    return net, p


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(CASES))
def test_cnn_step_matches_oracle(case):
    c = CASES[case]
    rng = np.random.default_rng(100 + ord(case))
    net, p = _build(case)
    eta = 0.5
    batches = [(_rng_images(rng, c["B"], c["shape"], c["u8"]), rng.integers(0, c["classes"], c["B"]).astype(np.int64))
               for _ in range(3)]
    f64 = lambda img: img.astype(np.float64)[..., None] if c["u8"] else img

    # one accumulate: gradients, taps, stats, and which kernels ran
    img, lab = batches[0]
    kernels = _profile(lambda: (net.accumulate_gradients_images(img, lab), net.synchronize()))
    for k in c["kernels"]:
        assert any(n.startswith(k) for n in kernels), (k, kernels)
    want_g, want_p, want_cost, want_hits, want_outs, want_dx = oracle_step(net, p, f64(img), lab, eta)
    got_g = net.get_gradients()
    for name, sl, _ in net.param_slices():
        assert_close(got_g[sl], want_g[sl], what=f"case {case} sum d{name}")
    for i in range(len(net.layers)):
        assert_close(net.layer_output(i), want_outs[i], what=f"case {case} layer {i} output")
    for i, l in enumerate(net.layers):    # the max pool picks the same element of the handle's own conv output
        if isinstance(l, _m().Pool) and l.pooling == _m().Pooling.Max:
            from oracle import ext as E
            below = net.layer_output(i - 1) if i else f64(img)
            y, _ = E.pool2d_forward(below, int(l.padding), int(l.pooling))
            assert np.array_equal(net.layer_output(i), y), f"case {case} pool {i}"
    assert_close(net.input_gradient(), want_dx, what=f"case {case} dX")
    cost, hits = net.last_batch_stats()
    assert hits == want_hits
    assert_close(cost, want_cost, what=f"case {case} batch cost")

    # evaluate: cost, hits, labels; the gradients stay as they were
    g_before = net.get_gradients()
    acc, ecost, labels_out = net.evaluate_images(img, lab, want_labels=True)
    assert np.array_equal(net.get_gradients(), g_before), "evaluate must leave the gradients untouched"
    from oracle import rcn_oracle_np as R
    _, Ws, bs = _unpack(net, p)
    feats = want_outs[-1].reshape(c["B"], -1)
    outs = [R.classify_test(Ws, bs, f) for f in feats]
    assert np.array_equal(labels_out, [R.argmax_last(o) for o in outs])
    assert acc == want_hits
    assert_close(ecost, want_cost, what=f"case {case} evaluate cost")
    assert np.array_equal(net.classify_images(img), labels_out)

    # accumulate + apply == train_batch, bit for bit
    net.apply_gradients(eta, c["B"])
    p1 = net.get_params()
    assert_close(p1, want_p, what=f"case {case} params after one step")
    net2, _ = _build(case)
    net2.train_batch_images(img, lab, eta)
    assert np.array_equal(net2.get_params(), p1), "accumulate + apply must equal train_batch"

    # three steps
    ref = want_p
    for img, lab in batches[1:]:
        net.train_batch_images(img, lab, eta)
        _, ref, *_ = oracle_step(net, ref, f64(img), lab, eta)
    assert_close(net.get_params(), ref, what=f"case {case} params after three steps")


@pytest.mark.gpu
def test_cnn_wide_tcgen05_wiring():
    """Case C: 32x32x64 -> Conv(128, 3x3, Same) -> MaxPool; the conv forward and weight gradient take the tcgen05
    integer-slice implicit GEMMs.  Every check but dX is bit for bit against the library's own ops on the same data."""
    import torch
    m = _m()
    from mercer_research_b200 import ext
    B, eta = 64, 0.25
    net = m.ConvNet((32, 32, 64), [m.Conv(128, 3, 3, m.Padding.Same), m.Pool(m.Pooling.Max, m.Padding.Same)], [32], 10)
    p = net.init_params(np.random.default_rng(3))
    rng = np.random.default_rng(4)
    x = rng.standard_normal((B, 32, 32, 64))
    lab = rng.integers(0, 10, B).astype(np.int64)
    kernels = _profile(lambda: (net.accumulate_gradients_images(x, lab), net.synchronize()))
    assert any(k.startswith("conv2d_forward_igemm(tcgen05") for k in kernels), kernels
    assert any(k.startswith("conv2d_backward_weight_igemm(tcgen05") for k in kernels), kernels
    nw = 128 * 9 * 64
    w, b = p[:nw].reshape(128, 3, 3, 64), p[nw:nw + 128]
    y = ext.conv2d_forward(x, w, b, m.Padding.Same, ext.Activation.ReLU)
    yp, am = ext.pool2d_forward(y, m.Padding.Same, m.Pooling.Max)
    assert np.array_equal(net.layer_output(0), y)
    assert np.array_equal(net.layer_output(1), yp)
    # dense part: an RCN driven by hand on the handle's own features
    L = net.feature_len
    dense = m.RCN(10, [], [32])
    dense.load_weights_and_bias_shapes([(32, L), (10, 32)])
    dense.set_params(p[nw + 128:])
    feats = net.layer_output(1).reshape(B, L)
    dense.accumulate_gradients(feats, labels=lab)
    g = net.get_gradients()
    assert np.array_equal(g[nw + 128:], dense.get_gradients())
    assert net.last_batch_stats() == dense.last_batch_stats()
    # conv part, fed with the handle's own dX
    dx = net.input_gradient()
    d_pool = ext.pool2d_backward(dx.reshape(yp.shape), am, (32, 32), m.Padding.Same, m.Pooling.Max)
    dz = ext.activation_backward(y, d_pool, ext.Activation.ReLU)
    dw, db = ext.conv2d_backward_weight(x, dz, 3, 3, m.Padding.Same)
    assert np.array_equal(g[:nw], dw.ravel()) and np.array_equal(g[nw:nw + 128], db)
    # dX against numpy W0^T delta0
    W0 = p[nw + 128:nw + 128 + 32 * L].reshape(L, 32).T
    assert_close(dx, dense.deltas(0) @ W0, what="case C dX")
    # the step
    net.apply_gradients(eta, B)
    dense.apply_gradients(eta, B)
    got = net.get_params()
    assert np.array_equal(got[nw + 128:], dense.get_params())
    assert np.array_equal(got[:nw + 128], p[:nw + 128] - (eta / B) * g[:nw + 128])
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_cnn_gradient_is_the_cost_derivative():
    """Central differences of the batch quadratic cost sum_b 0.5*|a_b - y_b|^2 for a few conv weights and biases of a tiny
    f64 network agree with the handle's gradient sums (independent of the oracle's composition)."""
    m = _m()
    net = m.ConvNet((8, 8, 2), [m.Conv(3, 3, 3, m.Padding.Same), m.Pool(m.Pooling.Max, m.Padding.None_),
                                m.Conv(2, 3, 3, m.Padding.Same), m.Pool(m.Pooling.Average, m.Padding.Same)], [5], 3)
    p = net.init_params(np.random.default_rng(11))
    rng = np.random.default_rng(12)
    x = rng.standard_normal((4, 8, 8, 2))
    lab = rng.integers(0, 3, 4).astype(np.int64)
    net.accumulate_gradients_images(x, lab)
    g = net.get_gradients()

    def cost(q):
        net.set_params(q)
        return net.evaluate_images(x, lab)[1]

    conv_idx = [i for name, sl, _ in net.param_slices() if name.startswith("conv") for i in range(sl.start, sl.stop)]
    pick = sorted(conv_idx, key=lambda i: -abs(g[i]))[:6] + [s.start for n, s, _ in net.param_slices() if n.endswith(".b")][:2]
    h = 1e-5
    for i in pick:
        qp, qm = p.copy(), p.copy()
        qp[i] += h
        qm[i] -= h
        fd = (cost(qp) - cost(qm)) / (2 * h)
        assert abs(fd - g[i]) <= 1e-6 * max(abs(g[i]), abs(fd)) + 1e-9, (i, fd, g[i])


@pytest.mark.gpu
def test_cnn_step_graph_capture():
    """After one eager step, accumulate + apply with device inputs captured into a CUDA graph and replayed three times
    equal three eager steps bit for bit."""
    import torch
    m = _m()
    c = CASES["B"]
    rng = np.random.default_rng(21)
    data = [(torch.tensor(rng.standard_normal((c["B"],) + c["shape"]), device="cuda"),
             torch.tensor(rng.integers(0, 10, c["B"]), device="cuda")) for _ in range(4)]
    eager, _ = _build("B", seed=5)
    graphed, _ = _build("B", seed=5)
    for net in (eager, graphed):
        net.accumulate_gradients_images(*data[0])
        net.apply_gradients(0.5, c["B"])
    x_in, y_in = data[0][0].clone(), data[0][1].clone()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        graphed.accumulate_gradients_images(x_in, y_in)
        graphed.apply_gradients(0.5, c["B"])
    for x, y in data[1:]:
        x_in.copy_(x)
        y_in.copy_(y)
        graph.replay()
        eager.accumulate_gradients_images(x, y)
        eager.apply_gradients(0.5, c["B"])
    torch.cuda.synchronize()
    assert np.array_equal(graphed.get_params(), eager.get_params())


def _nccl_cnn_worker(rank, world, port, out_dir):
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
    c = CASES["B"]
    net = m.ConvNet(c["shape"], c["layers"](m), c["ff"], c["classes"], device=rank)
    net.init_params(np.random.default_rng(31))
    trainer = DataParallelTrainer(net, eta=0.5, exchange="nccl")
    assert not trainer.p2p
    rng = np.random.default_rng(32)
    for _ in range(2):
        x = rng.standard_normal((128,) + c["shape"])
        y = rng.integers(0, 10, 128).astype(np.int64)
        trainer.step_global_images(torch.tensor(x, device="cuda"), torch.tensor(y, device="cuda"))
    torch.cuda.synchronize()
    np.save(os.path.join(out_dir, f"cnn_params_{rank}.npy"), net.get_params())
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.gpu
def test_cnn_nccl_two_gpus(tmp_path):
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mp.spawn(_nccl_cnn_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    p0, p1 = np.load(tmp_path / "cnn_params_0.npy"), np.load(tmp_path / "cnn_params_1.npy")
    assert np.array_equal(p0, p1), "replicas must stay bit-identical"
    m = _m()
    c = CASES["B"]
    ref = m.ConvNet(c["shape"], c["layers"](m), c["ff"], c["classes"])
    ref.init_params(np.random.default_rng(31))
    rng = np.random.default_rng(32)
    for _ in range(2):
        x = rng.standard_normal((128,) + c["shape"])
        y = rng.integers(0, 10, 128).astype(np.int64)
        ref.train_batch_images(x, y, 0.5)
    assert_close(p0, ref.get_params(), what="2-GPU NCCL vs 1 GPU on the global batch")


# -- CPU ----------------------------------------------------------------------------------------------------------------
def test_cnn_layer_spec_validation_needs_no_gpu(built_library):
    """Malformed stacks are refused with the ext ops' status codes before any device work (on a machine without a GPU a
    valid stack then fails with RCN_ERR_CUDA)."""
    m = _m()
    P, Q = m.Padding, m.Pooling
    cases = [
        ((8, 8, 1), [m.Conv(4, 2, 2, P.Same)], [8], 10, 2),                   # even kernel with Same
        ((4, 4, 1), [m.Conv(4, 5, 5, P.None_)], [8], 10, 2),                  # kernel larger than its map
        ((4, 4, 1), [m.Pool(Q.Max, P.None_), m.Pool(Q.Max, P.None_), m.Pool(Q.Max, P.None_)], [8], 10, 2),  # pool on 1x1
        ((8, 8, 1), [m.Conv(0, 3, 3, P.Same)], [8], 10, 1),                   # zero output channels
        ((8, 8, 0), [m.Conv(4, 3, 3, P.Same)], [8], 10, 1),                   # zero input channels
        ((8, 8, 1), [], [8], 10, 1),                                          # nothing in front of the dense stack
        ((8, 8, 1), [m.Conv(4, 3, 3, P.Same)], [0], 10, 1),                   # zero-width dense layer
        ((8, 8, 1), [m.Conv(4, 3, 3, P.Same)], [8], 0, 1),                    # zero classes
    ]
    for shape, layers, ff, classes, status in cases:
        with pytest.raises(m.RcnCudaError) as e:
            m.ConvNet(shape, layers, ff, classes)
        assert e.value.status == status, (layers, e.value)


def test_cnn_cpp_wrapper_compiles():
    gxx = shutil.which("g++")
    if not gxx:
        pytest.skip("g++ not available")
    src = r'''
#include "rcn.hpp"
int main() {
    using L = rcn::ConvNet::Layer;
    rcn::ConvNet net(12, 11, 1, {L::conv(4, 3, 3, rcn::Padding::Same), L::pool(rcn::Pooling::Max, rcn::Padding::Same)}, {8}, 10);
    std::vector<uint8_t> img(16 * 12 * 11);
    std::vector<int64_t> lab(16);
    net.train_batch(img.data(), RCN_PIXELS_U8_ROWMAJOR, lab.data(), 16, 12, 11, 0.5);
    auto st = net.last_batch_stats();
    auto ev = net.evaluate(img.data(), RCN_PIXELS_U8_ROWMAJOR, lab.data(), 16, 12, 11);
    return (int)(st.second + ev.first + net.get_params().size());
}
'''
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        p = os.path.join(d, "cnn.cpp")
        open(p, "w").write(src)
        r = subprocess.run([gxx, "-std=c++17", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), "-c", p, "-o",
                            os.path.join(d, "cnn.o")], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
