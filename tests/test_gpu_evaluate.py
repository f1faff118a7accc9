"""RCN.evaluate_images / rcn_cuda_evaluate_images: test-set evaluation (rcn.rs:152-157) straight from images, on one GPU.
The canonical network ([Conv Same, Pool Max], 28x28 u8, 784-30-10) runs the inference variant of kernel A
(smallnet_infer_kernel); everything else the existing feature, forward and statistics kernels.  Checked against the
oracle (features_u8 + standardise + Net.forward, accuracy, argmax_last) and, bit for bit, against the training step's
statistics, classify_images and evaluate on features."""
import ctypes as C
import os
import socket

import numpy as np
import pytest

import oracle as O

pytestmark = pytest.mark.gpu

CFG = [1, 3]
INFER_FUSED = "smallnet_infer_kernel(fused features)"                       # staged front end (FUSED 2)
INFER_GENERIC = "smallnet_infer_kernel(fused features, generic front end)"  # H*W not a multiple of 16 (FUSED 1)


@pytest.fixture(scope="module")
def api(built_library):
    import mercer_research_b200 as m
    return m


def make_model(api, ff=(30,), L=784, seed=0xC0FFEE, scale=(40.0, 60.0)):
    model = api.RCN(10, [api.RCNLayer.Convolve2D(api.Padding.Same), api.RCNLayer.Pool2D(api.Pooling.Max)], list(ff), device=0)
    model.load_weights_and_bias(L)
    params = np.random.default_rng(seed).standard_normal(model.n_params) * 0.1
    model.set_params(params)
    model.scale_set = scale
    return model, params


def oracle_eval(model, params, images, labels):
    """(accept, cost, argmax labels) of the oracle for u8 images (B, H, W)."""
    mean, sd = model.scale_set
    z = O.standardise(O.features_u8(CFG, images), mean, sd)
    acts = O.Net(model.layer_shapes).forward(params, z)
    y = np.zeros_like(acts)
    ok = (labels >= 0) & (labels < acts.shape[1])
    y[np.nonzero(ok)[0], labels[ok]] = 1.0
    return O.accuracy(acts, labels), 0.5 * float(np.sum((acts - y) ** 2)), O.argmax_last(acts)


def dataset(model, params, B, H=28, W=28, seed=7):
    """Seeded u8 images; half the labels are the oracle's prediction (so there are hits to count), half random."""
    rng = np.random.default_rng(seed + B)
    images = rng.integers(0, 256, size=(B, H, W), dtype=np.uint8)
    labels = rng.integers(0, 10, size=B).astype(np.int64)
    _, _, pred = oracle_eval(model, params, images, labels)
    labels[: B // 2] = pred[: B // 2]
    return images, labels


@pytest.mark.parametrize("device_inputs", [False, True], ids=["host", "device"])
@pytest.mark.parametrize("B", [1, 7, 64, 1000, 1024, 10000])
def test_canonical_network_against_oracle(api, B, device_inputs):
    import torch
    model, params = make_model(api)
    images, labels = dataset(model, params, B)
    want_acc, want_cost, want_lab = oracle_eval(model, params, images, labels)
    x, y = (torch.from_numpy(images).cuda(), torch.from_numpy(labels).cuda()) if device_inputs else (images, labels)
    acc, cost, lab = model.evaluate_images(x, y, want_labels=True)
    lab = lab.cpu().numpy() if device_inputs else lab
    assert acc == want_acc
    assert abs(cost - want_cost) <= 1e-9 * abs(want_cost), (cost, want_cost)
    assert np.array_equal(lab, want_lab)
    assert model.evaluate_images(x, y) == (acc, cost)


@pytest.mark.parametrize("B", [1000, 1024])
def test_bit_identical_to_the_existing_paths(api, B):
    model, params = make_model(api)
    images, labels = dataset(model, params, B)
    model.accumulate_gradients_images(images, labels)
    train_stats = model.last_batch_stats()
    grads = model.get_gradients()
    acc, cost, lab = model.evaluate_images(images, labels, want_labels=True)
    assert (cost, acc) == train_stats, "cost and hits must equal the training step's, bit for bit"
    assert np.array_equal(lab, model.classify_images(images))
    odd = labels.copy()
    odd[::5], odd[1::7] = -1, 10                                  # outside [0, classes): never a hit
    acc_odd, _ = model.evaluate_images(images, odd)
    assert acc_odd == model.evaluate(model.flatten_feature_set(images, standardise=True), odd)
    assert np.array_equal(model.get_params(), params)
    assert np.array_equal(model.get_gradients(), grads)
    assert model.last_batch_stats() == train_stats


def launches(api, fn):
    from mercer_research_b200 import _lib
    import torch
    torch.cuda.synchronize()
    _lib.profile_enable(True)
    try:
        out = fn()
        got = {name: v["launches"] for name, v in _lib.profile_report().items()}
    finally:
        _lib.profile_enable(False)
    return got, out


@pytest.mark.parametrize("B", [1, 64, 1000, 10000])
def test_route_canonical_u8(api, B):
    model, params = make_model(api)
    images, labels = dataset(model, params, B)
    got, _ = launches(api, lambda: model.evaluate_images(images, labels, want_labels=True))
    assert got == {INFER_FUSED: 1}, got


def test_route_generic_front_end_30x30(api):
    model, params = make_model(api, L=900)
    images, labels = dataset(model, params, 100, H=30, W=30)
    want_acc, want_cost, want_lab = oracle_eval(model, params, images, labels)
    got, (acc, cost, lab) = launches(api, lambda: model.evaluate_images(images, labels, want_labels=True))
    assert got == {INFER_GENERIC: 1}, got
    assert acc == want_acc and np.array_equal(lab, want_lab)
    assert abs(cost - want_cost) <= 1e-9 * abs(want_cost)


@pytest.mark.parametrize("case", ["f64_pixels", "wide_network"])
def test_route_existing_kernels(api, case):
    """f64 pixels, or a layer wider than 32: features + forward + batch_stats_kernel (+ argmax_last_kernel)."""
    model, params = make_model(api, ff=(256,) if case == "wide_network" else (30,))
    images, labels = dataset(model, params, 300)
    want_acc, want_cost, want_lab = oracle_eval(model, params, images, labels)
    x = images.astype(np.float64) if case == "f64_pixels" else images
    got, (acc, cost, lab) = launches(api, lambda: model.evaluate_images(x, labels, want_labels=True))
    assert not any(k.startswith("smallnet_infer_kernel") for k in got), got
    assert got.get("batch_stats_kernel") == 1 and got.get("argmax_last_kernel") == 1, got
    assert acc == want_acc and np.array_equal(lab, want_lab)
    assert abs(cost - want_cost) <= 1e-9 * abs(want_cost)


def test_device_outputs_capture_and_replay(api):
    """With cost and accept in device memory the call only enqueues work: it is captured into a CUDA graph, and every
    replay evaluates the images the buffer holds at that time (the last CTA resets the ticket)."""
    import torch
    from mercer_research_b200 import _lib
    model, params = make_model(api)
    B = 1000
    img = torch.zeros((B, 28, 28), dtype=torch.uint8, device="cuda")
    lab = torch.zeros(B, dtype=torch.int64, device="cuda")
    cost = torch.zeros(1, dtype=torch.float64, device="cuda")
    acc = torch.zeros(1, dtype=torch.int64, device="cuda")
    out = torch.zeros(B, dtype=torch.int64, device="cuda")

    def call():
        model.set_stream(torch.cuda.current_stream().cuda_stream)
        _lib.check(model._lib.rcn_cuda_evaluate_images(model._h, img.data_ptr(), _lib.PIXELS_U8_ROWMAJOR, lab.data_ptr(), B,
                                                       28, 28, cost.data_ptr(), acc.data_ptr(), out.data_ptr()))

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        call()                                        # warm-up outside the capture: buffers, kernel attributes
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        call()
    model.set_stream(torch.cuda.current_stream().cuda_stream)
    for seed in (11, 12):
        images, labels = dataset(model, params, B, seed=seed)
        img.copy_(torch.from_numpy(images))
        lab.copy_(torch.from_numpy(labels))
        graph.replay()
        torch.cuda.synchronize()
        want_acc, want_cost, want_lab = oracle_eval(model, params, images, labels)
        assert int(acc.item()) == want_acc
        assert abs(cost.item() - want_cost) <= 1e-9 * abs(want_cost)
        assert np.array_equal(out.cpu().numpy(), want_lab)


def test_batch_above_the_kernel_limit_runs_in_chunks(api):
    import torch
    n_max = 1 << 22                                     # smallnet_max_batch()
    B = n_max + 1000
    free, _ = torch.cuda.mem_get_info()
    if free < 40 * (1 << 30):
        pytest.skip("needs ~40 GB of free device memory")
    model, _ = make_model(api)
    g = torch.Generator(device="cuda").manual_seed(5)
    images = torch.randint(0, 256, (B, 28, 28), dtype=torch.uint8, device="cuda", generator=g)
    labels = torch.randint(0, 10, (B,), dtype=torch.int64, device="cuda", generator=g)
    got, (acc, cost) = launches(api, lambda: model.evaluate_images(images, labels))
    assert sum(v for k, v in got.items() if k.startswith("smallnet_infer_kernel")) == 2, got
    a0, c0 = model.evaluate_images(images[:n_max], labels[:n_max])
    a1, c1 = model.evaluate_images(images[n_max:], labels[n_max:])
    assert acc == a0 + a1
    assert cost == c0 + c1, "costs are added in chunk order"


def test_errors(api):
    from mercer_research_b200 import _lib
    lib = _lib.load()
    images = np.zeros((4, 28, 28), dtype=np.uint8)
    labels = np.zeros(4, dtype=np.int64)
    cost, acc = C.c_double(1.0), C.c_uint64(1)
    fresh = api.RCN(10, [api.RCNLayer.Convolve2D(api.Padding.Same), api.RCNLayer.Pool2D(api.Pooling.Max)], [30], device=0)
    with pytest.raises(_lib.RcnCudaError) as e:
        fresh.evaluate_images(images, labels)
    assert e.value.status == 5                                          # RCN_ERR_STATE: no parameters
    model, _ = make_model(api)
    h, ip, lp = model._h, images.ctypes.data, labels.ctypes.data
    ca, aa = C.addressof(cost), C.addressof(acc)
    assert lib.rcn_cuda_evaluate_images(h, None, 0, lp, 4, 28, 28, ca, aa, None) == 1
    assert lib.rcn_cuda_evaluate_images(h, ip, 0, None, 4, 28, 28, ca, aa, None) == 1
    assert lib.rcn_cuda_evaluate_images(h, ip, 0, lp, 4, 28, 28, None, aa, None) == 1
    assert lib.rcn_cuda_evaluate_images(h, ip, 0, lp, 4, 28, 28, ca, None, None) == 1
    assert lib.rcn_cuda_evaluate_images(h, ip, 7, lp, 4, 28, 28, ca, aa, None) == 1     # unknown pixel format
    assert lib.rcn_cuda_evaluate_images(h, ip, 0, lp, 4, 30, 30, ca, aa, None) == 2     # 900 features into a 784-wide layer
    got, rc = launches(api, lambda: lib.rcn_cuda_evaluate_images(h, None, 0, None, 0, 28, 28, ca, aa, None))
    assert rc == 0 and (cost.value, acc.value) == (0.0, 0) and got == {}
    assert model.evaluate_images(images[:0], labels[:0]) == (0, 0.0)


def test_train_arrays_evaluates_with_one_launch_per_epoch(api):
    model, _ = make_model(api)
    rng = np.random.default_rng(3)
    tr = rng.integers(0, 256, size=(256, 28, 28), dtype=np.uint8)
    te = rng.integers(0, 256, size=(300, 28, 28), dtype=np.uint8)
    tr_y, te_y = rng.integers(0, 10, size=256), rng.integers(0, 10, size=300)
    got, history = launches(api, lambda: model.train_arrays(tr, tr_y, te, te_y, 64, 2, 3.0, log=None))
    assert got.get(INFER_FUSED) == 2, got
    assert len(history) == 2


def _nccl_eval_worker(rank, world, port, out_dir):
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import torch
    import torch.distributed as dist
    import mercer_research_b200 as api
    from mercer_research_b200.trainer import DataParallelTrainer
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    model = api.RCN(10, [api.RCNLayer.Convolve2D(api.Padding.Same), api.RCNLayer.Pool2D(api.Pooling.Max)], [30], device=rank)
    model.load_weights_and_bias(784)
    model.set_params(np.random.default_rng(0xC0FFEE).standard_normal(model.n_params) * 0.1)
    model.scale_set = (40.0, 60.0)
    trainer = DataParallelTrainer(model, eta=3.0, device=torch.device("cuda", rank), exchange="nccl")
    rng = np.random.default_rng(77)
    images = torch.from_numpy(rng.integers(0, 256, size=(1001, 28, 28), dtype=np.uint8)).cuda(rank)
    labels = torch.from_numpy(rng.integers(0, 10, size=1001).astype(np.int64)).cuda(rank)
    acc, cost = trainer.evaluate(images, labels)
    np.save(os.path.join(out_dir, f"eval_{rank}.npy"), np.array([float(acc), cost]))
    dist.barrier()
    dist.destroy_process_group()


def test_data_parallel_evaluate_two_gpus(api, tmp_path):
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mp.spawn(_nccl_eval_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    r0, r1 = np.load(tmp_path / "eval_0.npy"), np.load(tmp_path / "eval_1.npy")
    assert np.array_equal(r0, r1), "every rank must return the same values"
    model, _ = make_model(api)
    rng = np.random.default_rng(77)
    images = rng.integers(0, 256, size=(1001, 28, 28), dtype=np.uint8)
    labels = rng.integers(0, 10, size=1001).astype(np.int64)
    acc, cost = model.evaluate_images(images, labels)
    assert int(r0[0]) == acc
    assert abs(r0[1] - cost) <= 1e-12 * abs(cost)
