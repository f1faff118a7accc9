"""GPU parity tests of the dense layers / backprop / SGD step through the C ABI.
Tolerance: 1e-9 relative (the reference computes in f64, BASELINE.json north_star); labels bit-exact."""
import os

import numpy as np
import pytest

import oracle as O
from conftest import assert_close

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
CP = [1, 3]


@pytest.fixture(scope="module")
def api(built_library):
    import mercer_research_b200 as m
    return m


def make_model(api, sizes, classes, n_in, seed=0xC0FFEE, scale=1.0):
    """Model with no convpool layers so the first dense layer takes n_in directly (4^0/2^0 * l)."""
    model = api.RCN(classes, [], sizes)
    model.load_weights_and_bias(n_in)
    net = O.Net(model.layer_shapes)
    params = np.random.default_rng(seed).standard_normal(net.n_params) * scale
    model.set_params(params)
    return model, net, params


def test_kat_mlp_step(api):
    """SURVEY.md Appendix B 3-2-2 MLP."""
    model = api.RCN(2, [], [2])
    model.load_weights_and_bias(3)
    assert model.layer_shapes == [(2, 3), (2, 2)]
    model.set_weights(0, [[0.1, -0.2, 0.3], [0.4, 0.5, -0.6]]); model.set_bias(0, [0.01, -0.02])
    model.set_weights(1, [[0.7, -0.8], [-0.9, 1.0]]); model.set_bias(1, [0.03, 0.04])
    x = np.array([[1.0, 0.5, -1.5]]); y = np.array([[0.0, 1.0]])
    model.train_batch(x, 3.0, onehot=y)
    assert_close(model.activations(0), [[0.3917409692534856, 0.8220063142137535]], what="a1")
    assert_close(model.activations(1), [[0.41256147606104177, 0.6246750573701205]], what="a2")
    assert_close(model.deltas(1), [[0.099986132119507, -0.08799723356765517]], what="d2")
    assert_close(model.deltas(0), [[0.035548466979736765, -0.024578376854694016]], what="d1")
    assert_close(model.get_weights(1), [[0.5824940070747917, -1.046567695808136], [-0.7965836352917443, 1.217002844877865]], what="W2'")
    assert_close(model.get_bias(1), [-0.26995839635852104, 0.3039917007029655], what="b2'")
    assert_close(model.get_weights(0), [[-0.006645400939210289, -0.25332270046960514, 0.45996810140881544],
                                        [0.47373513056408206, 0.536867565282041, -0.710602695846123]], what="W1'")
    assert_close(model.get_bias(0), [-0.0966454009392103, 0.05373513056408204], what="b1'")


def test_golden_dense_mnist8(api):
    g = np.load(os.path.join(GOLD, "dense_mnist8.npz"))
    model = api.RCN(10, [], [30])
    model.load_weights_and_bias(784)
    model.set_params(g["params"])
    assert_close(model.classify_test(g["X"]), g["acts"], what="acts")
    assert np.array_equal(model.classify_features(g["X"]), g["pred"])
    model.train_batch(g["X"], 3.0, labels=g["labels"])
    assert_close(model.get_gradients(), g["grads"], what="grads")
    assert_close(model.get_params(), g["new_params"], what="params'")
    assert_close(model.deltas(0)[0], g["sample0_deltas"][:30], what="delta1[0]")


SHAPES = [
    # (n_in, hidden sizes, classes, B)
    (784, [30], 10, 32),          # config C1
    (784, [30], 10, 1024),        # config C2
    (1024, [256], 10, 512),       # config C3 network
    (37, [13, 7], 3, 5),          # odd everything
    (12, [7, 5], 3, 1),           # single sample
    (300, [129, 65, 33], 17, 200),
    (640, [384, 256], 10, 2048),  # exercises the 128x128 tiles and split-K
    (200, [640], 10, 333),        # 640 -> 10: the skinny output-layer kernels (rows <= 16, K % 128 == 0), ragged batch
    (96, [512], 16, 1000),        # 512 -> 16: skinny kernels at their row limit
    (64, [1024], 3, 50),          # 1024 -> 3: fewer samples than one forward CTA holds
]


@pytest.mark.parametrize("n_in,hidden,classes,B", SHAPES)
def test_train_batch_parity(api, n_in, hidden, classes, B):
    model, net, params = make_model(api, hidden, classes, n_in, scale=1.0 if n_in < 100 else 0.05)
    rng = np.random.default_rng(B)
    X = np.maximum(rng.standard_normal((B, n_in)), 0)
    labels = (np.arange(B) % classes).astype(np.int64)
    Y = np.eye(classes)[labels]
    want_params, want_grads = net.train_batch(params, X, Y, 3.0, n_threads=1)
    want_acts = net.forward(params, X)
    got_acts = model.classify_test(X)
    assert_close(got_acts, want_acts, what="forward")
    assert np.array_equal(model.classify_features(X), O.argmax_last(want_acts))
    assert model.evaluate(X, labels) == O.accuracy(want_acts, labels)
    model.train_batch(X, 3.0, labels=labels)
    # per-sample taps for a few samples
    for b in sorted({0, B // 2, B - 1}):
        _, zs, acts, deltas = net.backprop(params, X[b], Y[b])
        o = 0
        for l, (r, _) in enumerate(net.shapes):
            assert_close(model.activations(l)[b], acts[o:o + r], what=f"a[{l}][{b}]")
            assert_close(model.deltas(l)[b], deltas[o:o + r], what=f"delta[{l}][{b}]")
            o += r
    assert_close(model.get_gradients(), want_grads, what="sum dW/db")
    assert_close(model.get_params(), want_params, what="post-step params")
    cost, hits = model.last_batch_stats()
    assert hits == O.accuracy(want_acts, labels)
    assert abs(cost - 0.5 * np.sum((want_acts - Y) ** 2)) <= 1e-9 * max(1.0, cost)
    # one-hot targets give the same step as labels
    model2, _, _ = make_model(api, hidden, classes, n_in, scale=1.0 if n_in < 100 else 0.05)
    model2.train_batch(X, 3.0, onehot=Y)
    assert np.array_equal(model2.get_params(), model.get_params())


def test_saturated_units_unscaled_init(api):
    """The reference draws N(0,1) weights unscaled (rcn.rs:509), so 784-wide layers saturate: sigmoid' = a*(1-a)
    cancels catastrophically and parity requires cancelling identically (DESIGN.md 'faithful quirks')."""
    model, net, params = make_model(api, [30], 10, 784, scale=1.0)
    rng = np.random.default_rng(5)
    X = np.maximum(rng.standard_normal((256, 784)), 0)
    labels = (np.arange(256) % 10).astype(np.int64)
    want_params, want_grads = net.train_batch(params, X, np.eye(10)[labels], 3.0)
    model.train_batch(X, 3.0, labels=labels)
    assert_close(model.get_gradients(), want_grads, what="grads")
    assert_close(model.get_params(), want_params, what="params")


def test_dmma_matches_simt_kernels(api, tmp_path):
    """The DMMA tensor path and the plain SIMT cross-check kernels must agree to rounding."""
    import subprocess
    import sys
    code = r'''
import numpy as np, sys
sys.path.insert(0, %r)
import mercer_research_b200 as m
model = m.RCN(10, [], [384, 256]); model.load_weights_and_bias(640)
model.set_params(np.random.default_rng(1).standard_normal(model.n_params) * 0.05)
X = np.maximum(np.random.default_rng(2).standard_normal((512, 640)), 0)
model.train_batch(X, 3.0, labels=(np.arange(512) %% 10).astype(np.int64))
np.save(sys.argv[1], model.get_params())
''' % os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    outs = []
    for impl in ("dmma", "simt"):
        path = str(tmp_path / f"rcn_gemm_{impl}.npy")
        env = dict(os.environ, RCN_CUDA_GEMM=impl)
        subprocess.run([sys.executable, "-c", code, path], check=True, env=env)
        outs.append(np.load(path))
    assert_close(outs[0], outs[1], rtol=1e-11, what="dmma vs simt")


def test_generic_gemm_path_on_the_canonical_net(api):
    """784-30-10 normally takes the fused small-network kernels; RCN_CUDA_SMALLNET=0 forces the generic tiled GEMM
    path, which must meet the same bar."""
    import subprocess
    import sys
    code = r'''
import numpy as np, sys
sys.path.insert(0, %r); sys.path.insert(0, %r + '/tests')
import mercer_research_b200 as m
import oracle as O
from conftest import assert_close
model = m.RCN(10, [], [30]); model.load_weights_and_bias(784)
net = O.Net(model.layer_shapes)
params = np.random.default_rng(1).standard_normal(net.n_params) * 0.05
model.set_params(params)
X = np.maximum(np.random.default_rng(2).standard_normal((300, 784)), 0)
labels = (np.arange(300) %% 10).astype(np.int64)
want, grads = net.train_batch(params, X, np.eye(10)[labels], 3.0)
model.train_batch(X, 3.0, labels=labels)
assert_close(model.get_gradients(), grads, what="grads")
assert_close(model.get_params(), want, what="params")
print("ok")
''' % ((os.path.dirname(os.path.dirname(os.path.abspath(__file__))),) * 2)
    env = dict(os.environ, RCN_CUDA_SMALLNET="0")
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr


def test_full_pipeline_config_c2(api):
    """BASELINE.json configs[1]: MNIST-shaped CNN, batch 1024, images -> features -> fwd -> bwd -> SGD."""
    rng = np.random.default_rng(0x5EED)
    B = 1024
    imgs = rng.integers(0, 256, size=(B, 28, 28), dtype=np.uint8)
    labels = (np.arange(B) % 10).astype(np.int64)
    model = api.RCN(10, [api.RCNLayer.Convolve2D(api.Padding.Same), api.RCNLayer.Pool2D(api.Pooling.Max)], [30])
    raw = O.features_u8(CP, imgs)
    mean, sd = O.gen_scales(raw)
    model.scale_set = (mean, sd)
    model.load_weights_and_bias(model.feature_len(28, 28))
    assert model.layer_shapes == [(30, 784), (10, 30)]
    net = O.Net(model.layer_shapes)
    params = np.random.default_rng(0xC0FFEE).standard_normal(net.n_params)
    model.set_params(params)
    X = O.standardise(raw, mean, sd)
    Y = np.eye(10)[labels]
    want_params, want_grads = net.train_batch(params, X, Y, 3.0)
    pred_before = model.classify_images(imgs)
    assert np.array_equal(pred_before, O.argmax_last(net.forward(params, X)))          # labels bit-exact
    model.train_batch_images(imgs, labels, 3.0)
    assert_close(model.get_gradients(), want_grads, what="grads")
    assert_close(model.get_params(), want_params, what="params")
    assert np.array_equal(model.classify_images(imgs), O.argmax_last(net.forward(want_params, X)))
    # threaded CPU reduction (the reference's rayon+mutex order) stays within tolerance of the GPU too
    thr_params, _ = net.train_batch(params, X, Y, 3.0, n_threads=8)
    assert_close(model.get_params(), thr_params, what="params vs threaded oracle")


@pytest.mark.parametrize("cfg,hw,B", [([1, 3], (28, 28), 1021), ([1, 3, 1, 3], (28, 28), 203), ([1, 3, 1, 3, 1, 3], (32, 32), 64),
                                       ([1, 3], (12, 20), 5), ([1, 3, 1, 3], (20, 12), 77), ([1, 3], (30, 28), 9)])
def test_fused_front_end_variants(api, cfg, hw, B):
    """Kernel A's staged front end (bulk-async image loads, zero-framed tiles) on stacks / sizes / ragged batches beyond the
    canonical one; (30, 28) has H*W % 16 != 0 and takes the generic fused front end.  Features bit-exact, step <= 1e-9."""
    rng = np.random.default_rng(B * 7 + hw[0])
    imgs = rng.integers(0, 256, size=(B,) + hw, dtype=np.uint8)
    labels = rng.integers(0, 10, B).astype(np.int64)
    lay = [api.RCNLayer.Convolve2D(api.Padding.Same) if c == 1 else api.RCNLayer.Pool2D(api.Pooling.Max) for c in cfg]
    model = api.RCN(10, lay, [30])
    raw = O.features_u8(cfg, imgs)
    mean, sd = O.gen_scales(raw)
    model.scale_set = (mean, sd)
    model.load_weights_and_bias(model.feature_len(*hw))
    net = O.Net(model.layer_shapes)
    params = np.random.default_rng(5).standard_normal(net.n_params) * 0.2
    model.set_params(params)
    X = O.standardise(raw, mean, sd)
    want_params, want_grads = net.train_batch(params, X, np.eye(10)[labels], 3.0)
    model.train_batch_images(imgs, labels, 3.0)
    assert_close(model.get_gradients(), want_grads, what="grads")
    assert_close(model.get_params(), want_params, what="params")


def test_multi_step_training_tracks_oracle(api):
    """20 consecutive SGD steps: errors must not compound beyond tolerance."""
    model, net, params = make_model(api, [16], 4, 40, scale=0.3)
    rng = np.random.default_rng(8)
    p = params.copy()
    for step in range(20):
        X = np.maximum(rng.standard_normal((24, 40)), 0)
        labels = rng.integers(0, 4, 24).astype(np.int64)
        p, _ = net.train_batch(p, X, np.eye(4)[labels], 3.0)
        model.train_batch(X, 3.0, labels=labels)
    assert_close(model.get_params(), p, rtol=1e-9, what="params after 20 steps")


def test_split_phase_equals_train_batch(api):
    """accumulate on two half batches + external sum + apply(global batch) == one train_batch (the DP contract)."""
    import torch
    model, net, params = make_model(api, [30], 10, 784, scale=0.05)
    rng = np.random.default_rng(12)
    X = np.maximum(rng.standard_normal((64, 784)), 0)
    labels = (np.arange(64) % 10).astype(np.int64)
    want, _ = net.train_batch(params, X, np.eye(10)[labels], 3.0)
    g = torch.zeros(model.n_params, dtype=torch.float64, device="cuda")
    model.bind_gradient_buffer(g)
    model.accumulate_gradients(X[:32], labels=labels[:32])
    model.synchronize()
    g0 = g.clone()
    model.accumulate_gradients(X[32:], labels=labels[32:])
    model.synchronize()
    g += g0
    torch.cuda.synchronize()
    model.apply_gradients(3.0, 64)
    assert_close(model.get_params(), want, what="split-phase params")


def test_shape_quirk_and_state_errors(api):
    """rcn.rs:443: one conv + two pools gives 4/16*l = 0 input columns -> `w * a` dimension mismatch."""
    model = api.RCN(10, [api.RCNLayer.Convolve2D(api.Padding.Same), api.RCNLayer.Pool2D(api.Pooling.Max),
                         api.RCNLayer.Pool2D(api.Pooling.Max)], [30])
    with pytest.raises(api.RcnCudaError):
        model.classify_test(np.zeros((1, 196)))            # parameters not initialised
    L = model.feature_len(28, 28)
    assert L == 4 * 7 * 7
    model.load_weights_and_bias(L)
    assert model.layer_shapes[0] == (30, 0)
    imgs = np.zeros((2, 28, 28), dtype=np.uint8)
    with pytest.raises(api.RcnCudaError) as e:
        model.train_batch_images(imgs, np.zeros(2, dtype=np.int64), 3.0)
    assert e.value.status == 2
    empty_ff = api.RCN(10, [], [])
    with pytest.raises(api.RcnCudaError):
        empty_ff.load_weights_and_bias(10)                 # feedforward_cfg[0] (rcn.rs:444)


def test_train_arrays_epoch_driver(api):
    """RCN::train semantics on in-memory images: chunks_exact drops the remainder, scale_set ends up holding the
    TEST set's statistics (rcn.rs:134-137), accuracy uses the exact-one-hot rule."""
    rng = np.random.default_rng(4)
    tr = rng.integers(0, 256, size=(53, 28, 28), dtype=np.uint8)
    te = rng.integers(0, 256, size=(20, 28, 28), dtype=np.uint8)
    trl = (np.arange(53) % 10).astype(np.int64)
    tel = (np.arange(20) % 10).astype(np.int64)
    model = api.RCN(10, [api.RCNLayer.Convolve2D(api.Padding.Same), api.RCNLayer.Pool2D(api.Pooling.Max)], [30])
    lines = []
    hist = model.train_arrays(tr, trl, te, tel, batch_size=10, epochs=2, eta=3.0, seed=1, log=lines.append)
    assert len(hist) == 2 and lines[0].startswith("Epoch 0: ") and lines[0].endswith("%]")
    te_raw = O.features_u8(CP, te)
    m, s = O.gen_scales(te_raw)
    gm, gs = model.scale_set
    assert abs(gm - m) <= 1e-12 * m and abs(gs - s) <= 1e-12 * s


def test_epoch_mode_and_cuda_graph(api):
    """Epoch mode (device-side cursor + perm, rcn.rs:144-149) eager and as a replayed CUDA graph must equal
    explicit train_batch_images calls on the same chunks, including the chunks_exact wrap-around."""
    import torch
    from mercer_research_b200.trainer import DataParallelTrainer
    rng = np.random.default_rng(77)
    N, B = 1000, 96                      # 10 full chunks, remainder 40 dropped
    imgs = rng.integers(0, 256, size=(N, 28, 28), dtype=np.uint8)
    labels = rng.integers(0, 10, N).astype(np.int64)
    perm = rng.permutation(N).astype(np.int64)
    cfg = [api.RCNLayer.Convolve2D(api.Padding.Same), api.RCNLayer.Pool2D(api.Pooling.Max)]

    def fresh():
        m = api.RCN(10, cfg, [30])
        m.scale_set = (20.0, 35.0)
        m.load_weights_and_bias(784)
        m.set_params(np.random.default_rng(3).standard_normal(m.n_params) * 0.05)
        return m

    ref = fresh()
    n_steps = 13                          # wraps after 10
    for k in range(n_steps):
        pos = (k % 10) * B
        idx = perm[pos:pos + B]
        ref.train_batch_images(imgs[idx], labels[idx], 3.0)
    want = ref.get_params()

    d_imgs, d_labels, d_perm = torch.from_numpy(imgs).cuda(), torch.from_numpy(labels).cuda(), torch.from_numpy(perm).cuda()
    eager = fresh()
    eager.epoch_bind(d_imgs, d_labels, B, perm=d_perm)
    for k in range(n_steps):
        eager.epoch_step(3.0)
    assert eager.epoch_position() == 3 * B
    assert np.array_equal(eager.get_params(), want)

    graphed = fresh()
    tr = DataParallelTrainer(graphed, eta=3.0)
    tr.bind_dataset(d_imgs, d_labels, B, perm=d_perm)
    tr.capture(warmup=2)
    # (capture() restores parameters and cursor after its own warm-up steps)
    for k in range(n_steps):
        tr.epoch_step()
    torch.cuda.synchronize()
    assert np.array_equal(graphed.get_params(), want)
    assert graphed.epoch_position() == 3 * B


@pytest.mark.parametrize("B,N,n_steps", [(1024, 5000, 7), (96, 1000, 5)])
def test_epoch_run_equals_steps_and_oracle(api, B, N, n_steps):
    """rcn_cuda_epoch_run (n iterations of the chunks_exact loop, rcn.rs:147-149, in one call) == n epoch_step calls, bit
    for bit, including the cursor wrap-around and a second call that continues; and both track the oracle's literal loop."""
    import torch
    rng = np.random.default_rng(B + n_steps)
    imgs = rng.integers(0, 256, size=(N, 28, 28), dtype=np.uint8)
    labels = rng.integers(0, 10, N).astype(np.int64)
    perm = rng.permutation(N).astype(np.int64)
    cfg = [api.RCNLayer.Convolve2D(api.Padding.Same), api.RCNLayer.Pool2D(api.Pooling.Max)]
    d_imgs, d_labels, d_perm = torch.from_numpy(imgs).cuda(), torch.from_numpy(labels).cuda(), torch.from_numpy(perm).cuda()

    def fresh():
        m = api.RCN(10, cfg, [30])
        m.scale_set = (20.0, 35.0)
        m.load_weights_and_bias(784)
        m.set_params(np.random.default_rng(3).standard_normal(m.n_params) * 0.05)
        m.epoch_bind(d_imgs, d_labels, B, perm=d_perm)
        return m

    stepwise = fresh()
    for k in range(n_steps + 2):
        stepwise.epoch_step(3.0)
    run = fresh()
    run.epoch_run(3.0, n_steps)
    run.epoch_run(3.0, 2)
    assert run.epoch_position() == stepwise.epoch_position()
    assert np.array_equal(run.get_params(), stepwise.get_params())
    assert run.last_batch_stats() == stepwise.last_batch_stats()
    raw = O.features_u8(CP, imgs)
    X = O.standardise(raw, 20.0, 35.0)
    net = O.Net([(30, 784), (10, 30)])
    p = np.random.default_rng(3).standard_normal(net.n_params) * 0.05
    pos = 0
    for k in range(n_steps + 2):
        idx = perm[pos:pos + B]
        p, _ = net.train_batch(p, X[idx], np.eye(10)[labels[idx]], 3.0)
        pos = pos + B if pos + 2 * B <= N else 0
    assert_close(run.get_params(), p, rtol=1e-9, what="params vs oracle epoch loop")


def test_train_epoch_host_equals_step_by_step(api):
    """The pipelined host-dataset loop (double-buffered H2D on a copy stream) == train_batch_images chunk by chunk,
    remainder dropped like chunks_exact (rcn.rs:147-149); per-step (cost, hits) equal last_batch_stats."""
    rng = np.random.default_rng(21)
    B, N = 64, 64 * 5 + 17
    images = rng.integers(0, 256, size=(N, 28, 28), dtype=np.uint8)
    labels = rng.integers(0, 10, size=N).astype(np.int64)
    cfg = [api.RCNLayer.Convolve2D(api.Padding.Same), api.RCNLayer.Pool2D(api.Pooling.Max)]
    params = None
    results = []
    import torch
    pinned = torch.from_numpy(images).pin_memory()       # pinned host memory takes the streaming (zero-copy prefetch) path
    pinned_labels = torch.from_numpy(labels).pin_memory()
    for mode in ("loop", "epoch", "epoch-pinned", "epoch-pinned-again"):
        model = api.RCN(10, cfg, [30])
        model.load_weights_and_bias(784)
        if params is None:
            params = np.random.default_rng(22).standard_normal(model.n_params)
        model.set_params(params)
        model.scale_set = (40.0, 60.0)
        if mode == "loop":
            stats = []
            for k in range(N // B):
                model.train_batch_images(images[k * B:(k + 1) * B], labels[k * B:(k + 1) * B], 3.0)
                stats.append(model.last_batch_stats())
            cost = np.array([s[0] for s in stats]); hits = np.array([s[1] for s in stats], dtype=np.uint64)
        elif mode == "epoch":
            cost, hits = model.train_epoch_host(images, labels, B, 3.0)
            assert len(cost) == N // B
        else:
            if mode.endswith("again"):                   # second epoch on the same handle replays the cached graph
                model.train_epoch_host(pinned.numpy(), pinned_labels.numpy(), B, 3.0)
                model.set_params(params)
            cost, hits = model.train_epoch_host(pinned.numpy(), pinned_labels.numpy(), B, 3.0)
            assert len(cost) == N // B
        results.append((model.get_params(), cost, hits))
    for other in results[1:]:
        assert np.array_equal(results[0][0], other[0]), "same kernels, same order: parameters must be bit-identical"
        assert np.array_equal(results[0][1], other[1]) and np.array_equal(results[0][2], other[2])


def test_train_epoch_host_streaming_large_chunks(api):
    """Same equality at a chunk size where every prefetch thread carries several 16-byte loads and the last round is
    ragged (B=1000: 49 000 uint4 per chunk over 8192 threads)."""
    import torch
    rng = np.random.default_rng(23)
    B, N = 1000, 1000 * 4 + 123
    images = torch.from_numpy(rng.integers(0, 256, size=(N, 28, 28), dtype=np.uint8)).pin_memory()
    labels = torch.from_numpy(rng.integers(0, 10, size=N).astype(np.int64)).pin_memory()
    cfg = [api.RCNLayer.Convolve2D(api.Padding.Same), api.RCNLayer.Pool2D(api.Pooling.Max)]
    out = []
    for mode in ("loop", "epoch-pinned"):
        model = api.RCN(10, cfg, [30])
        model.load_weights_and_bias(784)
        model.set_params(np.random.default_rng(24).standard_normal(model.n_params) * 0.1)
        model.scale_set = (40.0, 60.0)
        if mode == "loop":
            stats = []
            for k in range(N // B):
                model.train_batch_images(images.numpy()[k * B:(k + 1) * B], labels.numpy()[k * B:(k + 1) * B], 3.0)
                stats.append(model.last_batch_stats())
            cost = np.array([s[0] for s in stats]); hits = np.array([s[1] for s in stats], dtype=np.uint64)
        else:
            cost, hits = model.train_epoch_host(images.numpy(), labels.numpy(), B, 3.0)
        out.append((model.get_params(), cost, hits))
    assert np.array_equal(out[0][0].view(np.uint64), out[1][0].view(np.uint64))
    assert np.array_equal(out[0][1], out[1][1]) and np.array_equal(out[0][2], out[1][2])


HOST_COPY_SCRIPT = r'''
import numpy as np, sys, torch
sys.path.insert(0, %(root)r)
import mercer_research_b200 as m
rng = np.random.default_rng(31)
B, steps = 16, 151
N = B * steps + 5
images = torch.from_numpy(rng.integers(0, 256, size=(N, 28, 28), dtype=np.uint8)).pin_memory()
labels = torch.from_numpy(rng.integers(0, 10, size=N).astype(np.int64)).pin_memory()
cfg = [m.RCNLayer.Convolve2D(m.Padding.Same), m.RCNLayer.Pool2D(m.Pooling.Max)]
out = []
for mode in ("loop", "epoch", "epoch-again"):
    model = m.RCN(10, cfg, [30]); model.load_weights_and_bias(784)
    model.set_params(np.random.default_rng(32).standard_normal(model.n_params) * 0.1)
    model.scale_set = (40.0, 60.0)
    if mode == "loop":
        st = []
        for k in range(steps):
            model.train_batch_images(images.numpy()[k * B:(k + 1) * B], labels.numpy()[k * B:(k + 1) * B], 3.0)
            st.append(model.last_batch_stats())
        cost = np.array([x[0] for x in st]); hits = np.array([x[1] for x in st], dtype=np.uint64)
    else:
        if mode == "epoch-again":
            model.train_epoch_host(images.numpy()[:7 * B], labels.numpy()[:7 * B], B, 3.0)
            model.set_params(np.random.default_rng(32).standard_normal(model.n_params) * 0.1)
        cost, hits = model.train_epoch_host(images.numpy(), labels.numpy(), B, 3.0)
        assert len(cost) == steps
    out.append((model.get_params(), cost, hits))
for o in out[1:]:
    assert np.array_equal(out[0][0].view(np.uint64), o[0].view(np.uint64)), "parameters differ"
    assert np.array_equal(out[0][1], o[1]) and np.array_equal(out[0][2], o[2]), "per-step results differ"
print("ok")
'''


@pytest.mark.parametrize("copy_mode,spg", [("dma", "0"), ("dma", "1"), ("dma", "7"), ("pull", "0"), ("pull", "3")])
def test_train_epoch_host_copy_modes(api, copy_mode, spg):
    """Both ways the streamed epoch moves its images over PCIe (copy engine into a 64-chunk ring with an arrival counter
    kernel A waits on / SM-issued zero-copy loads on a graph branch), at several steps per graph ("0" = the mode's default:
    40 / 2): 151 steps wrap the ring twice and leave a remainder of 20-, 10- and single-step launches; bit-identical to train_batch_images chunk by chunk
    (rcn.rs:147-149)."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, RCN_CUDA_HOST_COPY=copy_mode, RCN_CUDA_HOST_STEPS_PER_GRAPH=spg)
    r = subprocess.run([sys.executable, "-c", HOST_COPY_SCRIPT % {"root": root}], env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


@pytest.mark.parametrize("same_device", [True, False])
@pytest.mark.parametrize("single_call", [True, False])
def test_dp_peer_memory_exchange_two_ranks(api, single_call, same_device):
    """Two ranks in one process -- on two GPUs of this box (peer access over NVLink) or BOTH ON DEVICE 0 (the protocol is
    the same: receive slots, sentinels, step parity, rank-ordered sum; this variant runs on a 1-GPU lease): the exchange +
    update -- as its own kernel after accumulate (split calls) or behind the weight-gradient kernel's pushes
    (train_batch_images, one call) -- keeps the replicas bit-identical and equals single-GPU training on the global minibatch
    within summation order (rcn.rs:190-222)."""
    import torch
    if not same_device and torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import threading
    rng = np.random.default_rng(23)
    Bg, steps = 128, 6
    images = rng.integers(0, 256, size=(steps, Bg, 28, 28), dtype=np.uint8)
    labels = rng.integers(0, 10, size=(steps, Bg)).astype(np.int64)
    cfg = [api.RCNLayer.Convolve2D(api.Padding.Same), api.RCNLayer.Pool2D(api.Pooling.Max)]
    ref = api.RCN(10, cfg, [30], device=0)
    ref.load_weights_and_bias(784)
    params = np.random.default_rng(24).standard_normal(ref.n_params)
    ref.set_params(params); ref.scale_set = (40.0, 60.0)
    for k in range(steps):
        ref.train_batch_images(images[k], labels[k], 3.0)
    want = ref.get_params()
    ranks = []
    for r in range(2):
        m = api.RCN(10, cfg, [30], device=0 if same_device else r)
        m.load_weights_and_bias(784)
        m.set_params(params); m.scale_set = (40.0, 60.0)
        m.dp_init(2, r)
        ranks.append(m)
    for m in ranks:
        m.dp_connect_local(ranks)
    half = Bg // 2
    errors = []

    def work(r):
        try:
            m = ranks[r]
            for k in range(steps):
                if single_call:    # the shard is this rank's batch; the library scales by the global batch (rcn.rs:214)
                    m.train_batch_images(images[k, r * half:(r + 1) * half], labels[k, r * half:(r + 1) * half], 3.0)
                else:
                    m.accumulate_gradients_images(images[k, r * half:(r + 1) * half], labels[k, r * half:(r + 1) * half])
                    m.apply_gradients(3.0, Bg)
            m.synchronize()
            m.dp_check()
        except Exception as e:   # noqa: BLE001
            errors.append((r, repr(e)))

    th = [threading.Thread(target=work, args=(r,)) for r in range(2)]
    [t.start() for t in th]
    [t.join(timeout=90) for t in th]
    assert not any(t.is_alive() for t in th), "ranks did not finish (exchange deadlock?)"
    assert not errors, errors
    p0, p1 = ranks[0].get_params(), ranks[1].get_params()
    assert np.array_equal(p0, p1), "replicas must stay bit-identical"
    assert_close(p0, want, rtol=1e-9, what="2-rank parameters vs single GPU")
    g0, g1 = ranks[0].get_gradients(), ranks[1].get_gradients()
    assert np.array_equal(g0, g1), "gradient buffers hold the same global sum on every rank"
    for m in ranks:
        m.dp_shutdown()


@pytest.mark.parametrize("graph", [False, True])
def test_dp_epoch_steps_two_ranks_prewait(api, graph):
    """The data-parallel EPOCH step as the bench runs it -- device cursor, kernel B pushing to the peer and advancing the
    cursor, the small exchange kernel, and the next step's kernel A running its front end ahead of griddepcontrol.wait --
    queued back to back without any host synchronisation in between (so consecutive steps really overlap), eagerly or as 4
    steps per CUDA graph.  Needs TWO GPUs: with both ranks on ONE device the peer's weight-gradient kernel (a thread-block-
    cluster launch) was measured NOT to start while this rank's exchange kernel is resident (device timeline, round 2: it
    started 5 us after the spinning kernel gave up), so a rank that runs ahead starves the other -- an artefact of sharing a
    device, which one process per GPU never does.  (bench.py checks the same path across processes in its `parity` block.)
    Replicas bit-identical, parameters equal to single-GPU training on the concatenated global batches, cursor wraps."""
    import threading
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    devs = (0, 1)
    rng = np.random.default_rng(77)
    B, n_chunks, steps = 64, 5, 12            # per-rank batch; 5 chunks per epoch -> the cursor wraps twice
    N = B * n_chunks + 17                      # chunks_exact drops the remainder
    shard = [rng.integers(0, 256, size=(N, 28, 28), dtype=np.uint8) for _ in range(2)]
    shard_labels = [rng.integers(0, 10, size=N).astype(np.int64) for _ in range(2)]
    cfg = [api.RCNLayer.Convolve2D(api.Padding.Same), api.RCNLayer.Pool2D(api.Pooling.Max)]
    params = np.random.default_rng(78).standard_normal(23860) * 0.05
    ref = api.RCN(10, cfg, [30], device=0)
    ref.load_weights_and_bias(784); ref.set_params(params); ref.scale_set = (40.0, 60.0)
    pos = 0
    for k in range(steps):
        gi = np.concatenate([shard[0][pos:pos + B], shard[1][pos:pos + B]])
        gl = np.concatenate([shard_labels[0][pos:pos + B], shard_labels[1][pos:pos + B]])
        ref.train_batch_images(gi, gl, 3.0)
        pos = pos + B if pos + 2 * B <= N else 0
    want = ref.get_params()
    ranks, streams, graphs, data = [], [], [], []
    for r in range(2):
        m = api.RCN(10, cfg, [30], device=devs[r])
        m.load_weights_and_bias(784); m.set_params(params); m.scale_set = (40.0, 60.0)
        m.dp_init(2, r)
        ranks.append(m)
    for m in ranks:
        m.dp_connect_local(ranks)
    for r, m in enumerate(ranks):
        # graph=True captures on a torch stream (one per device).  The eager variant keeps each model on the non-blocking
        # stream it created itself: two MORE streams on this one device can end up sharing a hardware queue with the other
        # rank's (CUDA_DEVICE_MAX_CONNECTIONS = 8), and a queue shared by both ranks serialises the peer behind a spinning
        # exchange kernel -- a one-process artefact (one process per GPU, the deployed shape, has a queue set per rank).
        st = torch.cuda.Stream(device=devs[r]) if graph else None
        streams.append(st)
        di, dl = torch.from_numpy(shard[r]).cuda(devs[r]), torch.from_numpy(shard_labels[r]).cuda(devs[r])
        data.append((di, dl))
        if graph:
            m.set_stream(st.cuda_stream)
        m.epoch_bind(di, dl, B)
    for d in set(devs):
        torch.cuda.synchronize(d)
    errors = []

    # Warm-up with SPLIT calls and a host barrier in between: the first step sizes every scratch buffer, and a cudaMalloc /
    # cudaFree synchronises the whole device -- on which, in this one-process test, the peer's exchange kernel may already
    # be spinning for our pushes (one process per GPU, the deployed shape, has no such coupling).  After the warm-up no call
    # allocates, so the steps below run back to back.
    gate = threading.Barrier(2)

    def warm(r):
        try:
            ranks[r].epoch_accumulate()
            ranks[r].synchronize()
            gate.wait(timeout=60)
            ranks[r].epoch_apply(3.0, 2 * B)
            ranks[r].synchronize()
        except Exception as e:   # noqa: BLE001
            errors.append((r, repr(e)))

    th = [threading.Thread(target=warm, args=(r,)) for r in range(2)]
    [t.start() for t in th]
    [t.join(timeout=90) for t in th]
    assert not any(t.is_alive() for t in th) and not errors, errors
    for m in ranks:
        m.set_params(params)
        m.epoch_seek(0)
    # graph=True: capture 4 steps per rank (capture executes nothing); both graphs are then replayed 3 times from two threads
    for r, m in enumerate(ranks):
        if not graph:
            break
        with torch.cuda.device(devs[r]):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=streams[r]):
                m.set_stream(streams[r].cuda_stream)
                for _ in range(4):
                    m.epoch_step(3.0)
        graphs.append(g)

    def work(r):
        try:
            if graph:
                with torch.cuda.device(devs[r]), torch.cuda.stream(streams[r]):
                    for _ in range(steps // 4):
                        graphs[r].replay()
                streams[r].synchronize()
            else:
                for _ in range(steps):              # no host synchronisation between the steps
                    ranks[r].epoch_step(3.0)
                ranks[r].synchronize()
            ranks[r].dp_check()
        except Exception as e:   # noqa: BLE001
            errors.append((r, repr(e)))

    th = [threading.Thread(target=work, args=(r,)) for r in range(2)]
    [t.start() for t in th]
    [t.join(timeout=90) for t in th]
    assert not any(t.is_alive() for t in th), "ranks did not finish (exchange deadlock?)"
    assert not errors, errors
    p0, p1 = ranks[0].get_params(), ranks[1].get_params()
    assert np.array_equal(p0, p1), "replicas must stay bit-identical"
    assert_close(p0, want, rtol=1e-9, what="2-rank graph-replayed epoch steps vs single GPU")
    assert ranks[0].epoch_position() == pos and ranks[1].epoch_position() == pos
    for m in ranks:
        m.dp_shutdown()


DP_TIMEOUT_SCRIPT = r"""
import json, sys, time
import numpy as np
sys.path.insert(0, %(root)r)
from mercer_research_b200 import RCN, Padding, Pooling, RCNLayer, _lib
cfg = [RCNLayer.Convolve2D(Padding.Same), RCNLayer.Pool2D(Pooling.Max)]
ranks = []
for r in range(2):
    m = RCN(10, cfg, [30], device=0)
    m.load_weights_and_bias(784)
    m.set_params(np.random.default_rng(1).standard_normal(m.n_params) * 0.05)
    m.dp_init(2, r)
    ranks.append(m)
for m in ranks:
    m.dp_connect_local(ranks)
rng = np.random.default_rng(2)
images = rng.integers(0, 256, size=(32, 28, 28), dtype=np.uint8)
labels = rng.integers(0, 10, size=32)
t0 = time.time()
ranks[0].train_batch_images(images, labels, 3.0)        # rank 1 never steps: its pushes never arrive
raised = ""
try:
    ranks[0].dp_check()
except _lib.RcnCudaError as e:
    raised = str(e)
print(json.dumps({"seconds": time.time() - t0, "raised": raised, "params_nan": bool(np.isnan(ranks[0].get_params()).any())}))
"""


def test_dp_exchange_times_out_instead_of_hanging(built_library):
    """ADVICE r1: a rank whose peer never pushes (died, raised before its launch, ran fewer steps) must not spin in a GPU
    kernel forever: the receive is bounded, sets the block's error word, and the host gets RCN_ERR_STATE."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, RCN_CUDA_DP_TIMEOUT_MS="300")
    out = subprocess.run([sys.executable, "-c", DP_TIMEOUT_SCRIPT % {"root": root}], env=env, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    r = json.loads(out.stdout.strip().splitlines()[-1])
    assert "timed out" in r["raised"], r
    assert r["params_nan"], r
    assert r["seconds"] < 60, r


def test_checkpoint_round_trip_on_device(api, tmp_path):
    """rcn.bin (bincode layout, serialization.py): save a trained model, reload it, same predictions and parameters."""
    rng = np.random.default_rng(41)
    cfg = [api.RCNLayer.Convolve2D(api.Padding.Same), api.RCNLayer.Pool2D(api.Pooling.Max)]
    model = api.RCN(10, cfg, [30], "images/train", "images/test")
    model.load_weights_and_bias(784)
    model.set_params(rng.standard_normal(model.n_params))
    model.scale_set = (41.5, 63.25)
    images = rng.integers(0, 256, size=(32, 28, 28), dtype=np.uint8)
    model.train_batch_images(images, rng.integers(0, 10, size=32), 3.0)
    path = str(tmp_path / "rcn.bin")
    model.save(path)
    back = api.RCN.load(path)
    assert back.layer_shapes == model.layer_shapes and back.scale_set == model.scale_set
    assert back.training_path == "images/train" and back.testing_path == "images/test"
    assert np.array_equal(back.get_params(), model.get_params())
    assert np.array_equal(back.classify_images(images), model.classify_images(images))


@pytest.mark.parametrize("graph", [True, False])
def test_train_arrays_matches_oracle_epoch_loop(api, graph):
    """The device-resident epoch driver (device-side shuffle indirection + cursor, optional CUDA graph) against the
    oracle running rcn.rs:144-165 literally: same permutations, same batches, train/test statistics applied the same way."""
    rng = np.random.default_rng(51)
    n, nt, B, epochs = 77, 40, 16, 3
    tr = rng.integers(0, 256, size=(n, 28, 28), dtype=np.uint8)
    te = rng.integers(0, 256, size=(nt, 28, 28), dtype=np.uint8)
    trl = rng.integers(0, 10, size=n).astype(np.int64)
    tel = rng.integers(0, 10, size=nt).astype(np.int64)
    model = api.RCN(10, [api.RCNLayer.Convolve2D(api.Padding.Same), api.RCNLayer.Pool2D(api.Pooling.Max)], [30])
    model.load_weights_and_bias(784)
    net = O.Net(model.layer_shapes)
    params = np.random.default_rng(52).standard_normal(net.n_params) * 0.1
    model.set_params(params)
    hist = model.train_arrays(tr, trl, te, tel, batch_size=B, epochs=epochs, eta=0.5, seed=7, log=None, cuda_graph=graph)
    # oracle
    ftr, fte = O.features_u8(CP, tr), O.features_u8(CP, te)
    mtr, mte = O.gen_scales(ftr), O.gen_scales(fte)
    xtr, xte = O.standardise(ftr, *mtr), O.standardise(fte, *mte)
    r2 = np.random.default_rng(7)
    p = params.copy()
    want_hist = []
    for _ in range(epochs):
        perm = r2.permutation(n)
        for s in range(0, n - B + 1, B):
            idx = perm[s:s + B]
            p, _ = net.train_batch(p, xtr[idx], np.eye(10)[trl[idx]], 0.5)
        want_hist.append(O.accuracy(net.forward(p, xte), tel))
    assert hist == want_hist
    assert_close(model.get_params(), p, rtol=1e-9, what="parameters after the epoch loop")
    gm, gs = model.scale_set
    assert abs(gm - mte[0]) <= 1e-12 * mte[0] and abs(gs - mte[1]) <= 1e-12 * mte[1]


def test_cached_step_graphs_survive_buffer_growth(api):
    """Device pointers are baked into the cached step graphs (the library's host-streaming graphs, the trainer's captured
    step). When a later call needs more scratch than any call before it (a longer epoch: the label stage grows; a bigger
    inference batch: features / activations grow) the grow-only buffers move and the graphs must be re-captured, not
    replayed with freed pointers. Results stay bit-identical to chunk-by-chunk training."""
    import torch
    from mercer_research_b200 import _lib
    from mercer_research_b200.trainer import DataParallelTrainer
    rng = np.random.default_rng(31)
    B, N = 64, 64 * 40
    images = torch.from_numpy(rng.integers(0, 256, size=(N, 28, 28), dtype=np.uint8)).pin_memory()
    labels = torch.from_numpy(rng.integers(0, 10, size=N).astype(np.int64)).pin_memory()
    big = rng.integers(0, 256, size=(6000, 28, 28), dtype=np.uint8)
    cfg = [api.RCNLayer.Convolve2D(api.Padding.Same), api.RCNLayer.Pool2D(api.Pooling.Max)]
    hi, hl = images.numpy(), labels.numpy()

    def fresh():
        m = api.RCN(10, cfg, [30])
        m.load_weights_and_bias(784)
        m.set_params(np.random.default_rng(32).standard_normal(m.n_params) * 0.1)
        m.scale_set = (40.0, 60.0)
        return m

    ref = fresh()
    for k in range(2 + 40 + 3):                  # the three epochs below, chunk by chunk
        j = k if k < 2 else (k - 2 if k < 42 else k - 42)
        ref.train_batch_images(hi[j * B:(j + 1) * B], hl[j * B:(j + 1) * B], 3.0)
        if k == 41:
            want_pred = ref.classify_images(big)  # labels under the parameters after the first two epochs
    want = ref.get_params()

    model = fresh()
    g0 = _lib.allocation_generation()
    model.train_epoch_host(hi[:2 * B], hl[:2 * B], B, 3.0)        # short epoch: graphs captured, small label stage
    assert _lib.allocation_generation() > g0
    model.train_epoch_host(hi, hl, B, 3.0)                        # 20x longer epoch: the label stage moves
    pred = model.classify_images(big)                             # much bigger batch: features / activations move
    model.train_epoch_host(hi[:3 * B], hl[:3 * B], B, 3.0)
    assert np.array_equal(model.get_params().view(np.uint64), want.view(np.uint64))
    assert np.array_equal(pred, want_pred)

    # the trainer's captured epoch step: replay, grow a buffer in between, replay again
    d_imgs, d_labels = images.cuda(), labels.cuda()
    ref2 = fresh()
    for k in range(6):
        ref2.train_batch_images(hi[k * B:(k + 1) * B], hl[k * B:(k + 1) * B], 3.0)
    graphed = fresh()
    tr = DataParallelTrainer(graphed, eta=3.0)
    tr.bind_dataset(d_imgs, d_labels, B)
    tr.capture(warmup=1, steps_per_graph=2)
    # (capture() restores parameters and cursor after its own warm-up steps)
    tr.epoch_steps(2)
    gen = tr._graph_generation
    graphed.classify_images(torch.from_numpy(big).cuda())         # grows the model's feature / activation buffers
    assert _lib.allocation_generation() != gen
    tr.epoch_steps(4)
    torch.cuda.synchronize()
    assert tr._graph_generation == _lib.allocation_generation()   # re-captured
    assert graphed.epoch_position() == 6 * B
    assert np.array_equal(graphed.get_params().view(np.uint64), ref2.get_params().view(np.uint64))


def test_cached_step_graphs_follow_scale_set(api):
    """scale_set travels by value in the captured kernel arguments: after set_scale / gen_scales changed it, the cached
    host-streaming graphs and the trainer's captured step must be re-captured (rcn.rs:406-412 standardises with the
    CURRENT scale_set), not replayed with the old (mean, sd)."""
    import torch
    from mercer_research_b200.trainer import DataParallelTrainer
    rng = np.random.default_rng(41)
    B, N = 64, 64 * 6
    images = torch.from_numpy(rng.integers(0, 256, size=(N, 28, 28), dtype=np.uint8)).pin_memory()
    labels = torch.from_numpy(rng.integers(0, 10, size=N).astype(np.int64)).pin_memory()
    hi, hl = images.numpy(), labels.numpy()
    cfg = [api.RCNLayer.Convolve2D(api.Padding.Same), api.RCNLayer.Pool2D(api.Pooling.Max)]

    def fresh():
        m = api.RCN(10, cfg, [30])
        m.load_weights_and_bias(784)
        m.set_params(np.random.default_rng(42).standard_normal(m.n_params) * 0.1)
        return m

    ref = fresh()
    for scale in ((40.0, 60.0), (25.0, 45.0)):
        ref.scale_set = scale
        for k in range(N // B):
            ref.train_batch_images(hi[k * B:(k + 1) * B], hl[k * B:(k + 1) * B], 3.0)
    want = ref.get_params()

    model = fresh()
    for scale in ((40.0, 60.0), (25.0, 45.0)):
        model.scale_set = scale
        model.train_epoch_host(hi, hl, B, 3.0)
    assert np.array_equal(model.get_params().view(np.uint64), want.view(np.uint64))

    graphed = fresh()
    graphed.scale_set = (40.0, 60.0)
    tr = DataParallelTrainer(graphed, eta=3.0)
    tr.bind_dataset(images.cuda(), labels.cuda(), B)
    tr.capture(warmup=1, steps_per_graph=3)
    # (capture() restores parameters and cursor after its own warm-up steps)
    tr.epoch_steps(6)
    graphed.scale_set = (25.0, 45.0)
    tr.epoch_steps(6)
    torch.cuda.synchronize()
    assert np.array_equal(graphed.get_params().view(np.uint64), want.view(np.uint64))


def test_train_epoch_host_contract(api):
    """Argument contract of the host-dataset loop: chunks_exact drops a short tail entirely (rcn.rs:147), device buffers are
    rejected, a wrong feature width is the reference's dimension-mismatch panic, state errors come back as status codes."""
    import torch
    cfg = [api.RCNLayer.Convolve2D(api.Padding.Same), api.RCNLayer.Pool2D(api.Pooling.Max)]
    model = api.RCN(10, cfg, [30])
    images = np.zeros((5, 28, 28), dtype=np.uint8)
    labels = np.zeros(5, dtype=np.int64)
    with pytest.raises(api.RcnCudaError) as e:
        model.train_epoch_host(images, labels, 4, 3.0)                       # no parameters yet
    assert e.value.status == 5
    model.load_weights_and_bias(784)
    before = model.get_params()
    cost, hits = model.train_epoch_host(images, labels, 8, 3.0)              # fewer samples than one batch: no step at all
    assert len(cost) == 0 and np.array_equal(model.get_params(), before)
    cost, hits = model.train_epoch_host(images, labels, 2, 3.0)              # 5 samples, batch 2 -> 2 steps, last sample dropped
    assert len(cost) == 2 and hits.dtype == np.uint64
    with pytest.raises(api.RcnCudaError) as e:
        api._lib.check(model._lib.rcn_cuda_train_epoch_host(model._h, torch.zeros(4, 28, 28, dtype=torch.uint8, device="cuda").data_ptr(),
                                                            0, labels.ctypes.data, 4, 28, 28, 2, 3.0, 0, None, None, None))
    assert e.value.status == 1
    wrong = api.RCN(10, cfg, [30])
    wrong.load_weights_and_bias(100)                                        # first layer expects 100 inputs, features are 784
    with pytest.raises(api.RcnCudaError) as e:
        wrong.train_epoch_host(images, labels, 2, 3.0)
    assert e.value.status == 2 and "mismatch" in e.value.message


def test_dp_group_contract(api):
    cfg = [api.RCNLayer.Convolve2D(api.Padding.Same), api.RCNLayer.Pool2D(api.Pooling.Max)]
    model = api.RCN(10, cfg, [30])
    with pytest.raises(api.RcnCudaError) as e:
        model.dp_init(2, 0)                                                  # needs parameters (the block is sized by them)
    assert e.value.status == 5
    model.load_weights_and_bias(784)
    for world, rank in [(0, 0), (2, 2), (17, 0), (2, -1)]:
        with pytest.raises(api.RcnCudaError) as e:
            model.dp_init(world, rank)
        assert e.value.status == 1
    handle = model.dp_init(1, 0)
    assert len(handle) == 64
    model.dp_connect_ipc([handle])                                          # a world of one is a no-op group
    model.set_params(np.zeros(model.n_params))
    model.train_batch_images(np.zeros((4, 28, 28), dtype=np.uint8), np.zeros(4, dtype=np.int64), 3.0)
    model.dp_shutdown()
    other = api.RCN(10, cfg, [30])
    other.load_weights_and_bias(784)
    with pytest.raises(api.RcnCudaError) as e:
        other.dp_connect_ipc([handle])                                      # connect before init
    assert e.value.status == 5


def test_wide_layer_beyond_exact_int32_range_stays_on_dmma(api):
    """K > 16384 cannot use the integer-slice path (int32 accumulation bound): the layer runs on DMMA and still matches."""
    from mercer_research_b200 import ext
    rng = np.random.default_rng(71)
    a = rng.standard_normal((130, 16500))
    b = rng.standard_normal((16500, 70))
    got = ext.gemm_f64(a, b, impl=0)
    assert_close(got, a @ b, rtol=1e-9, what="dmma, deep K")
    with pytest.raises(api.RcnCudaError) as e:
        ext.gemm_f64(a, b, impl=1)
    assert e.value.status == 1 and "exact int32" in e.value.message


def _nccl_numpy_worker(rank, world, port, out_dir):
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    import torch
    import torch.distributed as dist
    import mercer_research_b200 as m
    from mercer_research_b200.trainer import DataParallelTrainer, shard_bounds
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world,
                            device_id=torch.device("cuda", rank))
    rng = np.random.default_rng(51)
    Bg, steps = 256, 5
    images = rng.integers(0, 256, size=(steps, Bg, 28, 28), dtype=np.uint8)
    labels = rng.integers(0, 10, size=(steps, Bg)).astype(np.int64)
    cfg = [m.RCNLayer.Convolve2D(m.Padding.Same), m.RCNLayer.Pool2D(m.Pooling.Max)]
    model = m.RCN(10, cfg, [30], device=rank)
    model.load_weights_and_bias(784)
    model.set_params(np.random.default_rng(52).standard_normal(model.n_params) * 0.05)
    model.scale_set = (40.0, 60.0)
    trainer = DataParallelTrainer(model, eta=3.0, exchange="nccl")
    assert not trainer.p2p
    lo, hi = shard_bounds(Bg, rank, world)
    for k in range(steps):   # numpy (host) inputs: the library used to run these on its private stream, unordered with NCCL
        trainer.step_images_host(images[k, lo:hi], labels[k, lo:hi])
    torch.cuda.synchronize()
    np.save(os.path.join(out_dir, f"nccl_params_{rank}.npy"), model.get_params())
    dist.barrier()
    dist.destroy_process_group()


def test_nccl_exchange_with_host_inputs_two_gpus(api, tmp_path):
    """ADVICE r1: the NCCL path with numpy inputs must order the library's kernels, the all-reduce and the update on one
    stream (DataParallelTrainer binds the model to torch's current stream before every sequence). 2 processes x 1 GPU."""
    import socket
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mp.spawn(_nccl_numpy_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    p0, p1 = np.load(tmp_path / "nccl_params_0.npy"), np.load(tmp_path / "nccl_params_1.npy")
    assert np.array_equal(p0, p1), "replicas must stay bit-identical"
    rng = np.random.default_rng(51)
    images = rng.integers(0, 256, size=(5, 256, 28, 28), dtype=np.uint8)
    labels = rng.integers(0, 10, size=(5, 256)).astype(np.int64)
    cfg = [api.RCNLayer.Convolve2D(api.Padding.Same), api.RCNLayer.Pool2D(api.Pooling.Max)]
    ref = api.RCN(10, cfg, [30], device=0)
    ref.load_weights_and_bias(784)
    ref.set_params(np.random.default_rng(52).standard_normal(ref.n_params) * 0.05)
    ref.scale_set = (40.0, 60.0)
    for k in range(5):
        ref.train_batch_images(images[k], labels[k], 3.0)
    assert_close(p0, ref.get_params(), rtol=1e-9, what="2-GPU NCCL (host inputs) vs single GPU")
