"""Momentum SGD and AdamW for the convolutional network handle (rcn_cuda_cnn_set_optimizer, ConvNet.set_optimizer).

The yardstick is the header's operation order restated in numpy on the gradients the library reports: parameters and
optimizer state must match it bit for bit.  torch.optim confirms the semantics to 1e-12.  Every path that applies an
update (accumulate + apply, train_batch, epoch steps, epoch_run, graph replay, the data-parallel trainer) must agree bit
for bit, and a network that never picks an optimizer must keep the plain update's kernels."""
import ctypes as C
import os
import shutil
import socket
import subprocess
import tempfile

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _m():
    import mercer_research_b200 as m
    return m


# shape, u8 pixels, batch, dense widths, stack, head
STACKS = {
    # u8 images through the direct conv kernel, the fused narrow dense head
    "u8_narrow": dict(shape=(12, 11, 1), u8=True, B=16, ff=[8], softmax=False,
                      layers=lambda m: [m.Conv(4, 3, 3, m.Padding.Same), m.Pool(m.Pooling.Max, m.Padding.Same)]),
    # two conv layers on f64 images, the generic dense head
    "f64_two_conv": dict(shape=(16, 16, 3), u8=False, B=64, ff=[64], softmax=False,
                         layers=lambda m: [m.Conv(16, 3, 3, m.Padding.Same), m.Pool(m.Pooling.Max, m.Padding.None_),
                                           m.Conv(32, 3, 3, m.Padding.None_), m.Pool(m.Pooling.Average, m.Padding.Same)]),
    # no conv parameter: the first segment of the update is empty
    "pool_only": dict(shape=(12, 11, 1), u8=True, B=16, ff=[8], softmax=False,
                      layers=lambda m: [m.Pool(m.Pooling.Max, m.Padding.Same)]),
    "softmax": dict(shape=(12, 11, 1), u8=True, B=16, ff=[16], softmax=True,
                    layers=lambda m: [m.Conv(4, 3, 3, m.Padding.Same), m.Pool(m.Pooling.Max, m.Padding.Same)]),
}

# name -> (optimizer, eta)
OPTS = {
    "momentum": (lambda m: m.SGD(momentum=0.9), 0.5),
    "nesterov": (lambda m: m.SGD(momentum=0.9, nesterov=True), 0.5),
    "momentum_wd": (lambda m: m.SGD(momentum=0.8, weight_decay=1e-3), 0.5),
    "wd_only": (lambda m: m.SGD(weight_decay=1e-2), 0.5),
    "adamw": (lambda m: m.AdamW(), 0.01),
    "adamw_wd": (lambda m: m.AdamW(beta1=0.85, beta2=0.99, eps=1e-6, weight_decay=1e-2), 0.01),
}


def _net(stack, opt=None, seed=7):
    m = _m()
    c = STACKS[stack]
    head = m.Head.SoftmaxCrossEntropy if c["softmax"] else m.Head.SigmoidQuadratic
    net = m.ConvNet(c["shape"], c["layers"](m), c["ff"], 10, head=head)
    net.init_params(np.random.default_rng(seed))
    if opt is not None:
        net.set_optimizer(OPTS[opt][0](m))
    return net


def _data(stack, n, seed):
    c = STACKS[stack]
    rng = np.random.default_rng(seed)
    if c["u8"]:
        x = rng.integers(0, 256, size=(n,) + c["shape"][:2], dtype=np.uint8)
    else:
        x = rng.standard_normal((n,) + c["shape"])
    return x, rng.integers(0, 10, n).astype(np.int64)


def _dev(*arrays):
    import torch
    return [torch.as_tensor(a).cuda() for a in arrays]


def _positions(n, B, steps):
    pos, out = 0, []
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


def _launches(rep, prefix):
    return sum(v["launches"] for k, v in rep.items() if k.startswith(prefix))


def ref_state(opt, n):
    """The state right after set_optimizer."""
    m = _m()
    if isinstance(opt, m.AdamW):
        return np.concatenate([np.zeros(2 * n), [0.0, 1.0, 1.0]])
    return np.zeros(n) if opt.momentum > 0 else np.zeros(0)


def ref_step(opt, p, g, st, eta, B):
    """rcn_cuda.h's formulas, one rounding per operation (numpy never fuses a multiply-add)."""
    m = _m()
    n = p.size
    B = float(B)
    if isinstance(opt, m.SGD):
        d = g / B + opt.weight_decay * p
        st = st.copy()
        if opt.momentum > 0:
            st = opt.momentum * st + d
            u = d + opt.momentum * st if opt.nesterov else st
        else:
            u = d
        return p - eta * u, st
    mm, v, (t, b1t, b2t) = st[:n], st[n:2 * n], st[2 * n:]
    t, b1, b2 = t + 1.0, b1t * opt.beta1, b2t * opt.beta2
    p = p * (1.0 - eta * opt.weight_decay)
    gh = g / B
    mm = opt.beta1 * mm + (1.0 - opt.beta1) * gh
    v = opt.beta2 * v + (1.0 - opt.beta2) * (gh * gh)
    p = p - eta * ((mm / (1.0 - b1)) / (np.sqrt(v / (1.0 - b2)) + opt.eps))
    return p, np.concatenate([mm, v, [t, b1, b2]])


# -- 1. exact update ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("opt", sorted(OPTS))
@pytest.mark.parametrize("stack", sorted(STACKS))
def test_update_equals_numpy_restatement(stack, opt):
    """Three accumulate + apply steps: parameters and state equal the header's formulas on the reported gradients."""
    m = _m()
    o, eta = OPTS[opt][0](m), OPTS[opt][1]
    B = STACKS[stack]["B"]
    net = _net(stack, opt)
    p = net.get_params()
    st = ref_state(o, p.size)
    assert np.array_equal(net.optimizer_state(), st)
    for k in range(3):
        x, y = _data(stack, B, 20 + k)
        net.accumulate_gradients_images(x, y)
        g = net.get_gradients()
        net.apply_gradients(eta, B)
        p, st = ref_step(o, p, g, st, eta, B)
        assert np.array_equal(net.get_params(), p), f"{stack}/{opt}: parameters differ at step {k}"
        assert np.array_equal(net.optimizer_state(), st), f"{stack}/{opt}: state differs at step {k}"
    if isinstance(o, m.AdamW):
        assert net.optimizer_state()[-3] == 3.0


@pytest.mark.gpu
@pytest.mark.parametrize("opt", sorted(OPTS))
def test_update_matches_torch_optim(opt):
    """The same gradients through torch.optim.SGD / AdamW (float64, CPU) agree to 1e-12: the semantics are torch's."""
    import torch
    m = _m()
    o, eta = OPTS[opt][0](m), OPTS[opt][1]
    stack = "f64_two_conv"
    B = STACKS[stack]["B"]
    net = _net(stack, opt)
    tp = torch.nn.Parameter(torch.tensor(net.get_params()))
    if isinstance(o, m.SGD):
        topt = torch.optim.SGD([tp], lr=eta, momentum=o.momentum, nesterov=o.nesterov, weight_decay=o.weight_decay)
    else:
        topt = torch.optim.AdamW([tp], lr=eta, betas=(o.beta1, o.beta2), eps=o.eps, weight_decay=o.weight_decay)
    for k in range(3):
        x, y = _data(stack, B, 30 + k)
        net.accumulate_gradients_images(x, y)
        g = net.get_gradients()
        net.apply_gradients(eta, B)
        tp.grad = torch.tensor(g / float(B))
        topt.step()
        want = tp.detach().numpy()
        got = net.get_params()
        scale = np.max(np.abs(want))
        assert np.allclose(got, want, rtol=1e-12, atol=1e-12 * scale), (opt, k, np.max(np.abs(got - want)))


# -- 2. paths agree ----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("opt", ["momentum", "adamw_wd"])
@pytest.mark.parametrize("stack", ["u8_narrow", "f64_two_conv", "pool_only"])
def test_train_batch_equals_accumulate_apply(stack, opt):
    B = STACKS[stack]["B"]
    eta = OPTS[opt][1]
    a, b = _net(stack, opt), _net(stack, opt)
    for k in range(3):
        x, y = _data(stack, B, 40 + k)
        a.train_batch_images(x, y, eta)
        b.accumulate_gradients_images(x, y)
        b.apply_gradients(eta, B)
        assert np.array_equal(a.get_params(), b.get_params())
        assert np.array_equal(a.optimizer_state(), b.optimizer_state())
    b.apply_gradients(eta, 0)   # a batch of 0 is a no-op: no update, no step count
    assert np.array_equal(a.get_params(), b.get_params())
    assert np.array_equal(a.optimizer_state(), b.optimizer_state())


@pytest.mark.gpu
@pytest.mark.parametrize("use_perm", [True, False], ids=["perm", "identity"])
@pytest.mark.parametrize("opt", ["nesterov", "adamw"])
@pytest.mark.parametrize("stack", ["u8_narrow", "f64_two_conv", "pool_only", "softmax"])
def test_epoch_steps_equal_train_batch(stack, opt, use_perm):
    """Seven epoch steps over N = 3B + 5 samples (two wraps) equal train_batch_images on the gathered chunks; epoch_run
    equals the same steps."""
    import torch
    B = STACKS[stack]["B"]
    eta = OPTS[opt][1]
    n, steps = 3 * B + 5, 7
    x, y = _data(stack, n, 1)
    perm = np.random.default_rng(2).permutation(n) if use_perm else np.arange(n)
    xd, yd = _dev(x, y)
    pd = torch.as_tensor(perm).cuda() if use_perm else None
    net, ref, run = _net(stack, opt), _net(stack, opt), _net(stack, opt)
    net.epoch_bind(xd, yd, B, pd)
    run.epoch_bind(xd, yd, B, pd)
    pos = _positions(n, B, steps)
    for k in range(steps):
        net.epoch_step(eta)
        idx = perm[pos[k]:pos[k] + B]
        ref.train_batch_images(x[idx], y[idx], eta)
        assert np.array_equal(net.get_params(), ref.get_params()), f"{stack}/{opt}: step {k} differs"
        assert np.array_equal(net.optimizer_state(), ref.optimizer_state()), f"{stack}/{opt}: state after step {k}"
        assert net.epoch_position() == pos[k + 1], f"{stack}/{opt}: cursor after step {k}"
    run.epoch_run(eta, steps)
    assert np.array_equal(run.get_params(), ref.get_params())
    assert np.array_equal(run.optimizer_state(), ref.optimizer_state())
    assert run.epoch_position() == pos[-1]


@pytest.mark.gpu
@pytest.mark.parametrize("opt", ["momentum_wd", "adamw"])
@pytest.mark.parametrize("stack", ["u8_narrow", "f64_two_conv"])
def test_epoch_step_graph_replay(stack, opt):
    """Replays of one captured epoch_step equal eager steps across the wrap; with AdamW k replays leave t = k (every CTA
    reads t before the last one advances it, and the ticket resets for the next replay)."""
    import torch
    B = STACKS[stack]["B"]
    eta = OPTS[opt][1]
    n, steps = 3 * B + 5, 8
    x, y = _data(stack, n, 6)
    perm = np.random.default_rng(7).permutation(n)
    xd, yd, pd = _dev(x, y, perm)
    eager, graphed = _net(stack, opt), _net(stack, opt)
    eager.epoch_bind(xd, yd, B, pd)
    graphed.epoch_bind(xd, yd, B, pd)
    graphed.epoch_accumulate()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        graphed.set_stream(torch.cuda.current_stream().cuda_stream)
        graphed.epoch_step(eta)
    graphed.set_stream(torch.cuda.current_stream().cuda_stream)
    for k in range(steps):
        g.replay()
        eager.epoch_step(eta)
        torch.cuda.synchronize()
        if opt == "adamw":
            assert graphed.optimizer_state()[-3] == k + 1
    assert np.array_equal(graphed.get_params(), eager.get_params())
    assert np.array_equal(graphed.optimizer_state(), eager.optimizer_state())
    assert graphed.epoch_position() == eager.epoch_position() == _positions(n, B, steps)[-1]


# -- 3. the default update is unchanged --------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("stack", ["u8_narrow", "f64_two_conv", "pool_only"])
def test_default_keeps_plain_update_and_its_kernels(stack):
    m = _m()
    B = STACKS[stack]["B"]
    x, y = _data(stack, 3 * B, 50)
    plain, chosen = _net(stack), _net(stack)
    chosen.set_optimizer(m.SGD())
    assert chosen.optimizer_state().size == 0
    for k in range(3):
        xs, ys = x[k * B:(k + 1) * B], y[k * B:(k + 1) * B]
        plain.train_batch_images(xs, ys, 0.5)
        chosen.train_batch_images(xs, ys, 0.5)
        assert np.array_equal(plain.get_params(), chosen.get_params())
    conv = stack != "pool_only"
    for net in (plain, chosen):
        rep = _profile(lambda: (net.train_batch_images(x[:B], y[:B], 0.5), net.synchronize()))
        assert _launches(rep, "sgd_update_kernel") == (2 if conv else 1), rep
        assert _launches(rep, "optim_") == 0, rep
    xd, yd = _dev(x, y)
    for net in (plain, chosen):
        net.epoch_bind(xd, yd, B)
        net.epoch_step(0.5)
        rep = _profile(lambda: (net.epoch_step(0.5), net.synchronize()))
        assert _launches(rep, "sgd_update_kernel") == 2, rep   # the conv launch advances the cursor, with or without parameters
        assert _launches(rep, "optim_") == 0, rep
    assert np.array_equal(plain.get_params(), chosen.get_params())


@pytest.mark.gpu
@pytest.mark.parametrize("opt, kernel", [("wd_only", "optim_sgd_kernel"), ("nesterov", "optim_sgd_kernel"),
                                         ("adamw", "optim_adamw_kernel")])
@pytest.mark.parametrize("stack", ["u8_narrow", "pool_only"])
def test_optimizer_launches_one_kernel_per_apply(stack, opt, kernel):
    B = STACKS[stack]["B"]
    eta = OPTS[opt][1]
    x, y = _data(stack, 2 * B, 51)
    net = _net(stack, opt)
    net.train_batch_images(x[:B], y[:B], eta)
    rep = _profile(lambda: (net.train_batch_images(x[:B], y[:B], eta), net.synchronize()))
    assert _launches(rep, kernel) == 1 and _launches(rep, "optim_") == 1, rep
    assert _launches(rep, "sgd_update_kernel") == 0, rep
    xd, yd = _dev(x, y)
    net.epoch_bind(xd, yd, B)
    net.epoch_step(eta)
    rep = _profile(lambda: (net.epoch_step(eta), net.synchronize()))
    assert _launches(rep, kernel) == 1 and _launches(rep, "optim_") == 1, rep
    assert _launches(rep, "sgd_update_kernel") == 0, rep


# -- 4. resume ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("opt", ["momentum", "adamw_wd"])
def test_resume_in_a_fresh_network(opt):
    from mercer_research_b200 import _lib
    m = _m()
    stack = "f64_two_conv"
    B = STACKS[stack]["B"]
    eta = OPTS[opt][1]
    x, y = _data(stack, 5 * B, 60)
    batches = [(x[k * B:(k + 1) * B], y[k * B:(k + 1) * B]) for k in range(5)]
    whole = _net(stack, opt)
    for xs, ys in batches:
        whole.train_batch_images(xs, ys, eta)
    first = _net(stack, opt)
    for xs, ys in batches[:3]:
        first.train_batch_images(xs, ys, eta)
    params, state = first.get_params(), first.optimizer_state()
    fresh = _net(stack, opt, seed=99)
    fresh.set_params(params)
    gen = _lib.allocation_generation()
    fresh.load_optimizer_state(state)
    assert _lib.allocation_generation() == gen, "loading a state moves no buffer"
    for xs, ys in batches[3:]:
        fresh.train_batch_images(xs, ys, eta)
    assert np.array_equal(fresh.get_params(), whole.get_params())
    assert np.array_equal(fresh.optimizer_state(), whole.optimizer_state())
    # set_optimizer resets the state and asks for a re-capture
    gen = _lib.allocation_generation()
    whole.set_optimizer(OPTS[opt][0](m))
    assert _lib.allocation_generation() != gen
    assert np.array_equal(whole.optimizer_state(), ref_state(OPTS[opt][0](m), whole.n_params))


# -- 5. trainer --------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("opt", ["momentum", "adamw"])
def test_trainer_capture_restores_optimizer_state(opt):
    import torch
    from mercer_research_b200.trainer import DataParallelTrainer
    stack = "u8_narrow"
    B = STACKS[stack]["B"]
    eta = OPTS[opt][1]
    n, steps = 3 * B + 5, 7
    x, y = _data(stack, n, 70)
    perm = np.random.default_rng(71).permutation(n)
    xd, yd, pd = _dev(x, y, perm)
    net = _net(stack, opt)
    trainer = DataParallelTrainer(net, eta=eta)
    trainer.bind_dataset(xd, yd, B, pd)
    trainer.epoch_steps(2)                         # a state that is not the initial one
    torch.cuda.synchronize()
    p0, s0, c0 = net.get_params(), net.optimizer_state(), net.epoch_position()
    trainer.capture(warmup=3, steps_per_graph=2)
    assert np.array_equal(net.get_params(), p0) and net.epoch_position() == c0
    assert np.array_equal(net.optimizer_state(), s0), "capture must not advance the optimizer"
    trainer.epoch_steps(steps)                     # three replays and one eager step
    ref = _net(stack, opt)
    ref.epoch_bind(xd, yd, B, pd)
    ref.epoch_run(eta, 2 + steps)
    torch.cuda.synchronize()
    assert np.array_equal(net.get_params(), ref.get_params())
    assert np.array_equal(net.optimizer_state(), ref.optimizer_state())
    assert net.epoch_position() == ref.epoch_position()


def _nccl_adamw_worker(rank, world, port, out_dir):
    import sys
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist
    from mercer_research_b200.trainer import DataParallelTrainer
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world,
                            device_id=torch.device("cuda", rank))
    stack = "f64_two_conv"
    B = STACKS[stack]["B"]
    x, y = _data(stack, 3 * B + 5, 80 + rank)
    perm = np.random.default_rng(90 + rank).permutation(3 * B + 5)
    xd, yd, pd = (torch.as_tensor(a).cuda() for a in (x, y, perm))
    net = _net(stack, "adamw", seed=31)
    trainer = DataParallelTrainer(net, eta=OPTS["adamw"][1], exchange="nccl")
    assert not trainer.p2p
    trainer.bind_dataset(xd, yd, B, pd)
    trainer.epoch_steps(6)
    torch.cuda.synchronize()
    np.save(os.path.join(out_dir, f"p{rank}.npy"), net.get_params())
    np.save(os.path.join(out_dir, f"s{rank}.npy"), net.optimizer_state())
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.gpu
def test_adamw_nccl_two_gpus(tmp_path):
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mp.spawn(_nccl_adamw_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    assert np.array_equal(np.load(tmp_path / "p0.npy"), np.load(tmp_path / "p1.npy")), "replicas must stay bit-identical"
    s0, s1 = np.load(tmp_path / "s0.npy"), np.load(tmp_path / "s1.npy")
    assert np.array_equal(s0, s1) and s0[-3] == 6.0


# -- 6. learning -------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("opt, eta", [("adamw", 0.01), ("momentum", 0.3)])
def test_train_arrays_learns_with_optimizer(opt, eta):
    """Four classes told apart by which quadrant of an 8x8 image is bright: four epochs end at 75 % or better."""
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
    net.set_optimizer(OPTS[opt][0](m))
    hist = net.train_arrays(x, y, tx, ty, 16, 4, eta, seed=1, log=None)
    assert hist[-1] >= 0.75 * len(tx), hist
    if opt == "adamw":
        assert net.optimizer_state()[-3] == 4 * (1024 // 16)


# -- 7. errors ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_invalid_hyperparameters_and_state_lengths():
    m = _m()
    lib = m._lib.load()
    net = _net("u8_narrow")
    h = net._h
    nan, inf = float("nan"), float("inf")
    bad = [
        (2, 0.0, 0, 0.0, 0.9, 0.999, 1e-8),          # unknown kind
        (0, -0.1, 0, 0.0, 0, 0, 0), (0, 1.0, 0, 0.0, 0, 0, 0), (0, nan, 0, 0.0, 0, 0, 0), (0, inf, 0, 0.0, 0, 0, 0),
        (0, 0.9, 2, 0.0, 0, 0, 0), (0, 0.9, -1, 0.0, 0, 0, 0), (0, 0.0, 1, 0.0, 0, 0, 0),   # nesterov without momentum
        (0, 0.9, 0, -1e-4, 0, 0, 0), (0, 0.9, 0, nan, 0, 0, 0), (0, 0.9, 0, inf, 0, 0, 0),
        (1, 0, 0, 0.0, -0.1, 0.999, 1e-8), (1, 0, 0, 0.0, 1.0, 0.999, 1e-8), (1, 0, 0, 0.0, nan, 0.999, 1e-8),
        (1, 0, 0, 0.0, 0.9, 1.0, 1e-8), (1, 0, 0, 0.0, 0.9, -1.0, 1e-8), (1, 0, 0, 0.0, 0.9, inf, 1e-8),
        (1, 0, 0, 0.0, 0.9, 0.999, 0.0), (1, 0, 0, 0.0, 0.9, 0.999, -1e-8), (1, 0, 0, 0.0, 0.9, 0.999, nan),
        (1, 0, 0, 0.0, 0.9, 0.999, inf), (1, 0, 0, -1.0, 0.9, 0.999, 1e-8), (1, 0, 0, nan, 0.9, 0.999, 1e-8),
    ]
    net.set_optimizer(m.SGD(momentum=0.5))
    for args in bad:
        assert lib.rcn_cuda_cnn_set_optimizer(h, *args) == 1, args
    assert net.optimizer_state().size == net.n_params, "a refused call leaves the optimizer as it was"
    with pytest.raises(TypeError):
        net.set_optimizer("adam")
    n = net.n_params
    for opt, size in [(m.SGD(momentum=0.5), n), (m.AdamW(), 2 * n + 3), (m.SGD(weight_decay=0.1), 0)]:
        net.set_optimizer(opt)
        assert net.optimizer_state().size == size
        for wrong in (size + 1, max(size - 1, 0) if size else 1):
            buf = np.zeros(wrong)
            assert lib.rcn_cuda_cnn_set_optimizer_state(h, buf.ctypes.data, wrong) == 1
            assert lib.rcn_cuda_cnn_get_optimizer_state(h, buf.ctypes.data, wrong) == 1
        with pytest.raises(m.RcnCudaError) as e:
            net.load_optimizer_state(np.zeros(size + 2))
        assert e.value.status == 1


# -- CPU ---------------------------------------------------------------------------------------------------------------
def test_optimizer_entry_points_reject_a_null_handle(built_library):
    from mercer_research_b200 import _lib
    lib = _lib.load()
    n = C.c_size_t()
    calls = [
        lambda: lib.rcn_cuda_cnn_set_optimizer(None, 0, 0.9, 0, 0.0, 0.9, 0.999, 1e-8),
        lambda: lib.rcn_cuda_cnn_optimizer_state_size(None, C.byref(n)),
        lambda: lib.rcn_cuda_cnn_get_optimizer_state(None, None, 0),
        lambda: lib.rcn_cuda_cnn_set_optimizer_state(None, None, 0),
    ]
    for fn in calls:
        assert fn() == 1
        assert "null network handle" in lib.rcn_cuda_last_error().decode()


def test_optimizer_dataclasses_default_to_torch_defaults():
    m = _m()
    assert m.SGD() == m.SGD(momentum=0.0, nesterov=False, weight_decay=0.0)
    assert m.AdamW() == m.AdamW(beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=0.0)


def test_optimizer_cpp_wrapper_compiles():
    gxx = shutil.which("g++")
    if not gxx:
        pytest.skip("g++ not available")
    src = r'''
#include "rcn.hpp"
int main() {
    using L = rcn::ConvNet::Layer;
    rcn::ConvNet net(12, 11, 1, {L::conv(4, 3, 3, rcn::Padding::Same), L::pool(rcn::Pooling::Max, rcn::Padding::Same)}, {8}, 10);
    net.set_optimizer(rcn::Optimizer::sgd(0.9, true, 1e-4));
    net.set_optimizer(rcn::Optimizer::adamw(0.9, 0.999, 1e-8, 1e-2));
    net.set_optimizer(rcn::Optimizer{});
    std::vector<double> state = net.optimizer_state();
    net.set_optimizer_state(state);
    return (int)state.size();
}
'''
    with tempfile.TemporaryDirectory() as d:
        p = os.path.join(d, "cnn_optim.cpp")
        open(p, "w").write(src)
        r = subprocess.run([gxx, "-std=c++17", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), "-c", p, "-o",
                            os.path.join(d, "cnn_optim.o")], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
