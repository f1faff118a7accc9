"""Epoch mode of the convolutional network handle (rcn_cuda_cnn_epoch_*, ConvNet.epoch_* / train_arrays): a dataset
resident in HBM, the device-side cursor and its staging kernel, graph-replayed steps and the data-parallel trainer.

The yardstick is the handle's own batch path: an epoch step must equal train_batch_images on the host-gathered chunk
perm[pos:pos+B], bit for bit (test_gpu_cnn.py checks that path against the oracle)."""
import ctypes as C
import os
import shutil
import socket
import subprocess
import tempfile

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ETA = 0.5


def _m():
    import mercer_research_b200 as m
    return m


# shape, u8 pixels, batch, dense widths, stack
CASES = {
    # 132-byte images: 4-byte accesses; direct u8 conv kernel and the fused narrow head
    "u8_12x11": dict(shape=(12, 11, 1), u8=True, B=16, ff=[8],
                     layers=lambda m: [m.Conv(4, 3, 3, m.Padding.Same), m.Pool(m.Pooling.Max, m.Padding.Same)]),
    # 784-byte images: 16-byte accesses
    "u8_28x28": dict(shape=(28, 28, 1), u8=True, B=32, ff=[16],
                     layers=lambda m: [m.Conv(8, 3, 3, m.Padding.Same), m.Pool(m.Pooling.Max, m.Padding.Same)]),
    # test_gpu_cnn.py case B: two conv layers, the generic dense head
    "f64_16x16x3": dict(shape=(16, 16, 3), u8=False, B=64, ff=[64],
                        layers=lambda m: [m.Conv(16, 3, 3, m.Padding.Same), m.Pool(m.Pooling.Max, m.Padding.None_),
                                          m.Conv(32, 3, 3, m.Padding.None_), m.Pool(m.Pooling.Average, m.Padding.Same)]),
    # 840-byte images: 8-byte accesses
    "f64_5x7x3": dict(shape=(5, 7, 3), u8=False, B=8, ff=[8],
                      layers=lambda m: [m.Conv(4, 3, 3, m.Padding.Same), m.Pool(m.Pooling.Max, m.Padding.Same)]),
    "u8_pool_first": dict(shape=(12, 12, 1), u8=True, B=16, ff=[8],
                          layers=lambda m: [m.Pool(m.Pooling.Max, m.Padding.Same), m.Conv(4, 3, 3, m.Padding.Same)]),
    # no conv parameter: the update kernel still advances the cursor
    "u8_pool_only": dict(shape=(12, 11, 1), u8=True, B=16, ff=[8],
                         layers=lambda m: [m.Pool(m.Pooling.Max, m.Padding.Same)]),
}


def _net(case, seed=7):
    m = _m()
    c = CASES[case]
    net = m.ConvNet(c["shape"], c["layers"](m), c["ff"], 10)
    net.init_params(np.random.default_rng(seed))
    return net


def _data(case, n, seed):
    c = CASES[case]
    rng = np.random.default_rng(seed)
    if c["u8"]:
        x = rng.integers(0, 256, size=(n,) + c["shape"][:2], dtype=np.uint8)
    else:
        x = rng.standard_normal((n,) + c["shape"])
    return x, rng.integers(0, 10, n).astype(np.int64)


def _dev(*arrays):
    import torch
    return [torch.as_tensor(a).cuda() for a in arrays]


def _positions(n, B, steps, start=0):
    """The cursor before each step, and after the last: chunks_exact(B) with wrap-around."""
    pos, out = start, []
    for _ in range(steps + 1):
        out.append(pos)
        pos += B
        if pos + B > n:
            pos = 0
    return out


def _profile(fn):
    from mercer_research_b200 import _lib
    _lib.profile_enable(True)
    fn()
    rep = _lib.profile_report()
    _lib.profile_enable(False)
    return rep


@pytest.mark.gpu
@pytest.mark.parametrize("use_perm", [True, False], ids=["perm", "identity"])
@pytest.mark.parametrize("case", sorted(CASES))
def test_epoch_steps_equal_train_batch(case, use_perm):
    """8 steps over N = 3B + 5 samples (two wraps): parameters after every step equal train_batch_images on the chunk the
    cursor points at, bit for bit, and the cursor follows chunks_exact."""
    import torch
    B = CASES[case]["B"]
    n, steps = 3 * B + 5, 8
    x, y = _data(case, n, 1)
    perm = np.random.default_rng(2).permutation(n) if use_perm else np.arange(n)
    xd, yd = _dev(x, y)
    pd = torch.as_tensor(perm).cuda() if use_perm else None
    net, ref = _net(case), _net(case)
    net.epoch_bind(xd, yd, B, pd)
    pos = _positions(n, B, steps)
    assert net.epoch_position() == 0
    for k in range(steps):
        net.epoch_step(ETA)
        idx = perm[pos[k]:pos[k] + B]
        ref.train_batch_images(x[idx], y[idx], ETA)
        assert np.array_equal(net.get_params(), ref.get_params()), f"{case}: step {k} differs"
        assert net.epoch_position() == pos[k + 1], f"{case}: cursor after step {k}"


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["u8_12x11", "f64_16x16x3"])
def test_epoch_run_accumulate_apply_and_stats(case):
    import torch
    B = CASES[case]["B"]
    n = 3 * B + 5
    x, y = _data(case, n, 3)
    perm = np.random.default_rng(4).permutation(n)
    xd, yd, pd = _dev(x, y, perm)
    # epoch_run(n) == n epoch_step calls
    a, b = _net(case), _net(case)
    a.epoch_bind(xd, yd, B, pd)
    b.epoch_bind(xd, yd, B, pd)
    a.epoch_run(ETA, 5)
    for _ in range(5):
        b.epoch_step(ETA)
    assert np.array_equal(a.get_params(), b.get_params())
    assert a.epoch_position() == b.epoch_position() == _positions(n, B, 5)[-1]
    # accumulate twice (same chunk, same sums) + apply(eta, B) == epoch_step
    p0 = a.get_params()
    a.epoch_accumulate()
    g1 = a.get_gradients()
    a.epoch_accumulate()
    assert np.array_equal(a.get_gradients(), g1), "two accumulates without an apply must stage the same chunk"
    a.epoch_apply(ETA, B)
    b.epoch_step(ETA)
    assert np.array_equal(a.get_params(), b.get_params())
    assert a.epoch_position() == b.epoch_position()
    # last_batch_stats of a step == evaluate_images on that chunk under the pre-step parameters
    pos = a.epoch_position()
    p_pre = a.get_params()
    a.epoch_step(ETA)
    cost, hits = a.last_batch_stats()
    idx = perm[pos:pos + B]
    ev = _net(case)
    ev.set_params(p_pre)
    acc, ecost = ev.evaluate_images(x[idx], y[idx])
    assert hits == acc
    assert abs(cost - ecost) <= 1e-9 * max(1.0, abs(ecost)), (cost, ecost)
    assert not np.array_equal(p0, a.get_params())
    torch.cuda.synchronize()


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["u8_12x11", "u8_pool_first", "f64_5x7x3"])
def test_epoch_step_launch_profile(case):
    """One staging launch per step; no separate widening kernel for u8 images."""
    B = CASES[case]["B"]
    x, y = _data(case, 2 * B, 5)
    xd, yd = _dev(x, y)
    net = _net(case)
    net.epoch_bind(xd, yd, B)
    net.epoch_step(ETA)
    net.synchronize()
    rep = _profile(lambda: (net.epoch_step(ETA), net.synchronize()))
    stage = [k for k in rep if k.startswith("cnn_stage_batch_kernel")]
    assert stage and sum(rep[k]["launches"] for k in stage) == 1, rep
    assert not any("u8_to_f64" in k for k in rep), rep
    if CASES[case]["u8"]:   # the batch path widens u8 images with the same kernel (identity mapping)
        rep = _profile(lambda: (net.train_batch_images(x[:B], y[:B], ETA), net.synchronize()))
        assert sum(v["launches"] for k, v in rep.items() if k.startswith("cnn_stage_batch_kernel")) == 1, rep


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["u8_28x28", "f64_16x16x3"])
def test_epoch_step_graph_replay(case):
    """One captured epoch_step replayed across the wrap equals eager steps; so does DataParallelTrainer's epoch mode,
    whose capture leaves parameters and cursor as it found them."""
    import torch
    from mercer_research_b200.trainer import DataParallelTrainer
    B = CASES[case]["B"]
    n, steps = 3 * B + 5, 8
    x, y = _data(case, n, 6)
    perm = np.random.default_rng(7).permutation(n)
    xd, yd, pd = _dev(x, y, perm)
    eager, graphed = _net(case), _net(case)
    eager.epoch_bind(xd, yd, B, pd)
    graphed.epoch_bind(xd, yd, B, pd)
    graphed.epoch_accumulate()                    # sizes the buffers outside the capture; cursor and parameters stay
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        graphed.set_stream(torch.cuda.current_stream().cuda_stream)
        graphed.epoch_step(ETA)
    graphed.set_stream(torch.cuda.current_stream().cuda_stream)
    for _ in range(steps):
        g.replay()
        eager.epoch_step(ETA)
    torch.cuda.synchronize()
    assert np.array_equal(graphed.get_params(), eager.get_params())
    assert graphed.epoch_position() == eager.epoch_position() == _positions(n, B, steps)[-1]

    net = _net(case)
    trainer = DataParallelTrainer(net, eta=ETA)
    trainer.bind_dataset(xd, yd, B, pd)
    p0 = net.get_params()
    trainer.capture(warmup=2, steps_per_graph=2)
    assert np.array_equal(net.get_params(), p0) and net.epoch_position() == 0, "capture must not advance training"
    trainer.epoch_steps(steps + 1)               # four replays and one eager step
    ref = _net(case)
    ref.epoch_bind(xd, yd, B, pd)
    ref.epoch_run(ETA, steps + 1)
    torch.cuda.synchronize()
    assert np.array_equal(net.get_params(), ref.get_params())
    assert net.epoch_position() == ref.epoch_position()


def _nccl_epoch_worker(rank, world, port, out_dir):
    import sys
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist
    from mercer_research_b200.trainer import DataParallelTrainer
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world,
                            device_id=torch.device("cuda", rank))
    c = CASES["f64_16x16x3"]
    B = c["B"]
    x, y = _data("f64_16x16x3", 3 * B + 5, 40 + rank)
    perm = np.random.default_rng(50 + rank).permutation(3 * B + 5)
    xd, yd, pd = (torch.as_tensor(a).cuda() for a in (x, y, perm))
    net = _net("f64_16x16x3", seed=31)
    trainer = DataParallelTrainer(net, eta=ETA, exchange="nccl")
    assert not trainer.p2p
    trainer.bind_dataset(xd, yd, B, pd)
    trainer.epoch_steps(6)
    torch.cuda.synchronize()
    np.save(os.path.join(out_dir, f"cnn_epoch_params_{rank}.npy"), net.get_params())
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.gpu
def test_epoch_nccl_two_gpus(tmp_path):
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mp.spawn(_nccl_epoch_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    p0, p1 = np.load(tmp_path / "cnn_epoch_params_0.npy"), np.load(tmp_path / "cnn_epoch_params_1.npy")
    assert np.array_equal(p0, p1), "replicas must stay bit-identical"
    B = CASES["f64_16x16x3"]["B"]
    n = 3 * B + 5
    shards = [(_data("f64_16x16x3", n, 40 + r), np.random.default_rng(50 + r).permutation(n)) for r in range(2)]
    ref = _net("f64_16x16x3", seed=31)
    for pos in _positions(n, B, 6)[:-1]:
        xs = np.concatenate([x[p[pos:pos + B]] for (x, _), p in shards])
        ys = np.concatenate([y[p[pos:pos + B]] for (_, y), p in shards])
        ref.train_batch_images(xs, ys, ETA)
    want = ref.get_params()
    assert np.max(np.abs(p0 - want)) <= 1e-9 * max(1.0, np.max(np.abs(want)))


def _hand_loop(net, x, y, tx, ty, B, epochs, eta, seed):
    """train_arrays written out: the same generator, train_batch_images on the permuted chunks, chunked evaluation."""
    rng = np.random.default_rng(seed)
    net.init_params(rng)
    hist = []
    for _ in range(epochs):
        perm = rng.permutation(len(x))
        for k in range(len(x) // B):
            idx = perm[k * B:(k + 1) * B]
            net.train_batch_images(x[idx], y[idx], eta)
        hist.append(sum(net.evaluate_images(tx[i:i + B], ty[i:i + B])[0] for i in range(0, len(tx), B)))
    return hist


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["u8_12x11", "f64_5x7x3"])
def test_train_arrays_equals_hand_written_loop(case):
    B = CASES[case]["B"]
    x, y = _data(case, 5 * B + 3, 8)
    tx, ty = _data(case, 2 * B + 1, 9)
    m = _m()
    c = CASES[case]
    net = m.ConvNet(c["shape"], c["layers"](m), c["ff"], 10)
    lines = []
    hist = net.train_arrays(x, y, tx, ty, B, 3, ETA, seed=5, log=lines.append)
    ref = m.ConvNet(c["shape"], c["layers"](m), c["ff"], 10)
    want = _hand_loop(ref, x, y, tx, ty, B, 3, ETA, 5)
    assert hist == want
    assert np.array_equal(net.get_params(), ref.get_params())
    assert lines[0] == "Epoch 0: {}/{} [{:.2f}%]".format(want[0], len(tx), want[0] / len(tx) * 100.0)


@pytest.mark.gpu
def test_train_arrays_learns_a_separable_set():
    """Four classes told apart by which quadrant of an 8x8 image is bright: three epochs end well above chance."""
    m = _m()
    rng = np.random.default_rng(10)

    def make(n):
        lab = rng.integers(0, 4, n).astype(np.int64)
        img = 0.1 * rng.random((n, 8, 8, 1))
        for i, c in enumerate(lab):
            r, q = divmod(int(c), 2)
            img[i, 4 * r:4 * r + 4, 4 * q:4 * q + 4, 0] += 1.0
        return img, lab

    x, y = make(1024)
    tx, ty = make(256)
    net = m.ConvNet((8, 8, 1), [m.Conv(4, 3, 3, m.Padding.Same), m.Pool(m.Pooling.Max, m.Padding.Same)], [16], 4)
    hist = net.train_arrays(x, y, tx, ty, 16, 3, 3.0, seed=1, log=None)
    assert hist[-1] >= 0.75 * len(tx), hist


@pytest.mark.gpu
def test_epoch_entry_points_reject_bad_calls():
    import torch
    m = _m()
    lib = m._lib.load()
    net = _net("u8_12x11")
    h = net._h
    B = 16
    x, y = _data("u8_12x11", 2 * B, 11)
    xd, yd = _dev(x, y)
    u8 = m._lib.PIXELS_U8_ROWMAJOR
    # a step before bind
    assert lib.rcn_cuda_cnn_epoch_step(h, ETA) == 5
    assert lib.rcn_cuda_cnn_epoch_accumulate(h) == 5
    assert lib.rcn_cuda_cnn_epoch_apply(h, ETA, B) == 5
    assert lib.rcn_cuda_cnn_epoch_run(h, ETA, 1) == 5
    assert lib.rcn_cuda_cnn_epoch_seek(h, 0) == 5
    assert lib.rcn_cuda_cnn_epoch_position(h, C.byref(C.c_size_t())) == 5
    # host pointers
    assert lib.rcn_cuda_cnn_epoch_bind(h, x.ctypes.data, u8, yd.data_ptr(), None, 2 * B, 12, 11, B) == 1
    assert lib.rcn_cuda_cnn_epoch_bind(h, xd.data_ptr(), u8, y.ctypes.data, None, 2 * B, 12, 11, B) == 1
    perm = np.arange(2 * B)
    assert lib.rcn_cuda_cnn_epoch_bind(h, xd.data_ptr(), u8, yd.data_ptr(), perm.ctypes.data, 2 * B, 12, 11, B) == 1
    # shapes and format
    assert lib.rcn_cuda_cnn_epoch_bind(h, xd.data_ptr(), u8, yd.data_ptr(), None, 2 * B, 11, 12, B) == 2
    assert lib.rcn_cuda_cnn_epoch_bind(h, xd.data_ptr(), 7, yd.data_ptr(), None, 2 * B, 12, 11, B) == 1
    # n < B, B == 0
    assert lib.rcn_cuda_cnn_epoch_bind(h, xd.data_ptr(), u8, yd.data_ptr(), None, B - 1, 12, 11, B) == 1
    assert lib.rcn_cuda_cnn_epoch_bind(h, xd.data_ptr(), u8, yd.data_ptr(), None, 2 * B, 12, 11, 0) == 1
    with pytest.raises(ValueError):
        net.epoch_bind(x, y, B)
    # bound: seek past the last whole chunk, zero global batch
    net.epoch_bind(xd, yd, B)
    with pytest.raises(m.RcnCudaError) as e:
        net.epoch_seek(B + 1)
    assert e.value.status == 1
    with pytest.raises(m.RcnCudaError) as e:
        net.epoch_apply(ETA, 0)
    assert e.value.status == 1
    torch.cuda.synchronize()


# -- CPU ----------------------------------------------------------------------------------------------------------------
def test_epoch_entry_points_reject_a_null_handle(built_library):
    from mercer_research_b200 import _lib
    lib = _lib.load()
    calls = [
        lambda: lib.rcn_cuda_cnn_epoch_bind(None, None, 0, None, None, 1, 1, 1, 1),
        lambda: lib.rcn_cuda_cnn_epoch_seek(None, 0),
        lambda: lib.rcn_cuda_cnn_epoch_position(None, C.byref(C.c_size_t())),
        lambda: lib.rcn_cuda_cnn_epoch_accumulate(None),
        lambda: lib.rcn_cuda_cnn_epoch_apply(None, 0.5, 1),
        lambda: lib.rcn_cuda_cnn_epoch_step(None, 0.5),
        lambda: lib.rcn_cuda_cnn_epoch_run(None, 0.5, 1),
    ]
    for fn in calls:
        assert fn() == 1
        assert "null network handle" in lib.rcn_cuda_last_error().decode()


def test_epoch_cpp_wrapper_compiles():
    gxx = shutil.which("g++")
    if not gxx:
        pytest.skip("g++ not available")
    src = r'''
#include "rcn.hpp"
int main() {
    using L = rcn::ConvNet::Layer;
    rcn::ConvNet net(12, 11, 1, {L::conv(4, 3, 3, rcn::Padding::Same), L::pool(rcn::Pooling::Max, rcn::Padding::Same)}, {8}, 10);
    const void* images = nullptr;    // device memory in a real program
    const int64_t* labels = nullptr;
    net.epoch_bind(images, RCN_PIXELS_U8_ROWMAJOR, labels, nullptr, 53, 12, 11, 16);
    net.epoch_seek(0);
    net.epoch_accumulate();
    net.epoch_apply(0.5, 16);
    net.epoch_step(0.5);
    net.epoch_run(0.5, 3);
    return (int)net.epoch_position();
}
'''
    with tempfile.TemporaryDirectory() as d:
        p = os.path.join(d, "cnn_epoch.cpp")
        open(p, "w").write(src)
        r = subprocess.run([gxx, "-std=c++17", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), "-c", p, "-o",
                            os.path.join(d, "cnn_epoch.o")], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
