"""Which kernels each training entry point launches, on one GPU, for the canonical network ([Conv Same, Pool Max], 28x28 u8
images, 784-30-10).  A fused step is kernel A and kernel B with the SGD update in its epilogue; a split step is kernel A,
kernel B and one sgd_update_kernel.  A step that loses kernel B's update still trains correctly, only one launch slower, so
these counts are what catches it.  The parameters are checked against the oracle as well, so that an update applied twice
cannot pass either."""
import numpy as np
import pytest

import oracle as O
from conftest import assert_close

pytestmark = pytest.mark.gpu

B, STEPS, ETA = 64, 3, 3.0
A_FUSED = "smallnet_fwd_bwd_kernel(fused features)"   # kernel A with the convpool front end
A_FEATS = "smallnet_fwd_bwd_kernel"                   # kernel A on given features
B_UPDATE = "smallnet_wgrad_kernel(+SGD update)"
B_PLAIN = "smallnet_wgrad_kernel"
SGD = "sgd_update_kernel"


@pytest.fixture(scope="module")
def api(built_library):
    import mercer_research_b200 as m
    return m


@pytest.fixture(scope="module")
def data():
    rng = np.random.default_rng(0x1A0C)
    images = rng.integers(0, 256, size=(STEPS * B, 28, 28), dtype=np.uint8)
    labels = rng.integers(0, 10, size=STEPS * B).astype(np.int64)
    feats = O.features_u8([1, 3], images)
    mean, sd = O.gen_scales(feats)
    z = O.standardise(feats, mean, sd)
    return images, labels, z, (mean, sd)


def oracle_params(shapes, data, params, steps):
    _, labels, z, _ = data
    net = O.Net(shapes)
    for k in range(steps):
        s = slice(k * B, (k + 1) * B)
        params, _ = net.train_batch(params, z[s], np.eye(10)[labels[s]], ETA)
    return params


def step_train_batch_images(model, data):
    images, labels, _, _ = data
    model.train_batch_images(images[:B], labels[:B], ETA)


def step_train_batch(model, data):
    _, labels, z, _ = data
    model.train_batch(z[:B], ETA, labels=labels[:B])


def step_accumulate_apply(model, data):
    images, labels, _, _ = data
    model.accumulate_gradients_images(images[:B], labels[:B])
    model.apply_gradients(ETA, B)


def step_epoch_step(model, data):
    model.epoch_step(ETA)


def step_epoch_accumulate_apply(model, data):
    model.epoch_accumulate()
    model.epoch_apply(ETA, B)


def step_train_epoch_host(model, data):
    images, labels, _, _ = data
    model.train_epoch_host(images, labels, B, ETA)   # unpinned numpy: the general double-buffered loop


CASES = {
    "train_batch_images": (step_train_batch_images, 1, {A_FUSED: 1, B_UPDATE: 1}),
    "train_batch": (step_train_batch, 1, {A_FEATS: 1, B_UPDATE: 1}),
    "accumulate_gradients_images+apply_gradients": (step_accumulate_apply, 1, {A_FUSED: 1, B_PLAIN: 1, SGD: 1}),
    "epoch_step": (step_epoch_step, 1, {A_FUSED: 1, B_UPDATE: 1}),
    "epoch_accumulate+epoch_apply": (step_epoch_accumulate_apply, 1, {A_FUSED: 1, B_PLAIN: 1, SGD: 1}),
    "train_epoch_host": (step_train_epoch_host, STEPS, {A_FUSED: STEPS, B_PLAIN: STEPS, SGD: STEPS}),
}


@pytest.mark.parametrize("case", list(CASES))
def test_step_launches(api, data, case):
    import torch
    from mercer_research_b200 import _lib
    step, steps, want = CASES[case]
    images, labels, _, scale = data
    model = api.RCN(10, [api.RCNLayer.Convolve2D(api.Padding.Same), api.RCNLayer.Pool2D(api.Pooling.Max)], [30], device=0)
    model.load_weights_and_bias(784)
    params = np.random.default_rng(0xC0FFEE).standard_normal(model.n_params) * 0.1
    model.set_params(params)
    model.scale_set = scale
    if case.startswith("epoch"):
        model.epoch_bind(torch.from_numpy(images).cuda(), torch.from_numpy(labels).cuda(), B)
    torch.cuda.synchronize()
    _lib.profile_enable(True)
    try:
        step(model, data)
        got = {name: v["launches"] for name, v in _lib.profile_report().items()}
    finally:
        _lib.profile_enable(False)
    assert got == want, f"{case}: launched {got}, expected {want}"
    if case.startswith("epoch"):
        assert model.epoch_position() == B, "the cursor must advance by exactly one batch"
    assert_close(model.get_params(), oracle_params(model.layer_shapes, data, params, steps), what=f"{case}: parameters")
