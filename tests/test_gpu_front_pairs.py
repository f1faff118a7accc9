"""Kernel A's staged front end in both of its forms, bit for bit against the oracle's features.

A one-stage [Conv(Same), Pool(Max)] stack runs on image pairs: the two fp16 lanes of a tile word hold the same pixel of
images g and g + 4 of the CTA's eight, and every intermediate (|v| <= 255 * 4 = 1020) is an exact fp16 integer.  Deeper
stacks (255 * 16 > 2048) keep the int32 tiles.  smallnet_front_select picks the form from the plan; both run under the same
launch names, so the cases below are chosen by their shape: c2's 28x28 and a 32x32 one-stage stack on the pair path, a
two-stage stack on the int32 path.

Kernel A writes the standardised features to the HBM buffer that kernel B's dW0 = sum_b delta0_b f_b^T reads, and to the
shared tile that its layer-0 product reads.  A step from images must therefore give exactly the gradients, activations,
deltas and statistics of the same step fed the oracle's standardised features (kernel A on given features): a feature that
differs in any sample shows up in its column of dW0.  The evaluation kernel shares the front end; its cost and hits must be
the training step's, bit for bit.

Batches: B = 1024; B = 8k + 5, whose last tile has a pair with a missing image; B = 3, fewer images than pairs; and images
that reach the +-1020 bounds (flat, stripes of one and two pixels, 0/255 checkerboards of one and two pixels, each with its
inverse)."""
import zlib

import numpy as np
import pytest

import oracle as O

gpu = pytest.mark.gpu

A_FUSED = "smallnet_fwd_bwd_kernel(fused features)"
A_FEATS = "smallnet_fwd_bwd_kernel"
B_PLAIN = "smallnet_wgrad_kernel"
INFER_STAGED = "smallnet_infer_kernel(fused features)"

CASES = [   # name, cfg, (H, W), hidden, classes, B (None: the bound patterns)
    ("c2-B1024", [1, 3], (28, 28), [30], 10, 1024),
    ("c2-B1029", [1, 3], (28, 28), [30], 10, 1029),
    ("c2-B3", [1, 3], (28, 28), [30], 10, 3),
    ("c2-bounds", [1, 3], (28, 28), [30], 10, None),
    ("32x32-B100", [1, 3], (32, 32), [16], 10, 100),
    ("32x32-bounds", [1, 3], (32, 32), [16], 10, None),
    ("two-stage-28x28-B1029", [1, 3, 1, 3], (28, 28), [30], 10, 1029),
    ("two-stage-28x28-bounds", [1, 3, 1, 3], (28, 28), [30], 10, None),
]


def bound_images(H, W, rng):
    """Flat 0 and 255, stripes and checkerboards of one and two pixels and their inverses, then three random images: 21, so
    the last tile holds five images."""
    r, c = np.meshgrid(np.arange(H), np.arange(W), indexing="ij")
    pats = [np.zeros((H, W), bool), (r // 2) % 2 == 0, (c // 2) % 2 == 0, (r // 2 + c // 2) % 2 == 0, r % 2 == 0, c % 2 == 0,
            (r + c) % 2 == 0, (r // 2) % 2 == (c % 2), (r < H // 2)]
    imgs = [np.where(p, 255, 0) for p in pats] + [np.where(p, 0, 255) for p in pats]
    imgs += list(rng.integers(0, 256, size=(3, H, W)))
    return np.array(imgs, dtype=np.uint8)


def test_bound_images_reach_the_fp16_bound():
    """CPU only: the bound patterns reach |v| = 1020 in every one of the four operators of the first stage."""
    imgs = bound_images(28, 28, np.random.default_rng(0))
    f = O.features_u8([1, 3], imgs).reshape(len(imgs), 4, -1)
    assert f.max() == 1020
    assert all(f[:, k].max() == 1020 for k in range(4))


def launched(fn):
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


@gpu
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_front_end_features_bit_exact(built_library, case):
    import mercer_research_b200 as m

    name, cfg, hw, hidden, classes, B = case
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    images = bound_images(*hw, rng) if B is None else rng.integers(0, 256, size=(B,) + hw, dtype=np.uint8)
    B = len(images)
    raw = O.features_u8(cfg, images)
    mean, sd = O.gen_scales(O.features_u8(cfg, rng.integers(0, 256, size=(32,) + hw, dtype=np.uint8)))
    X = O.standardise(raw, mean, sd)
    model = m.RCN(classes, cfg, hidden, device=0)
    model.load_weights_and_bias(raw.shape[1])
    model.scale_set = (mean, sd)
    params = np.concatenate([rng.standard_normal(r * k) * (2.0 / np.sqrt(k)) if i % 2 == 0 else rng.standard_normal(r) * 0.5
                             for r, k in model.layer_shapes for i in range(2)])
    model.set_params(params)
    labels = rng.integers(0, classes, size=B).astype(np.int64)

    def step(fn):
        got, _ = launched(fn)
        out = dict(grads=model.get_gradients(), stats=model.last_batch_stats(),
                   acts=[model.activations(l) for l in range(len(model.layer_shapes))],
                   dels=[model.deltas(l) for l in range(len(model.layer_shapes))])
        return got, out

    got, from_images = step(lambda: model.accumulate_gradients_images(images, labels))
    assert got == {A_FUSED: 1, B_PLAIN: 1}, got          # the staged front end inside kernel A
    got, from_feats = step(lambda: model.accumulate_gradients(X, labels=labels))
    assert got == {A_FEATS: 1, B_PLAIN: 1}, got
    assert np.array_equal(from_images["grads"].view(np.uint64), from_feats["grads"].view(np.uint64)), \
        "gradients from images differ from those from the oracle's features"
    for l in range(len(model.layer_shapes)):
        assert np.array_equal(from_images["acts"][l], from_feats["acts"][l]), f"activations of layer {l}"
        assert np.array_equal(from_images["dels"][l], from_feats["dels"][l]), f"deltas of layer {l}"
    assert from_images["stats"] == from_feats["stats"]

    got, (hits, cost) = launched(lambda: model.evaluate_images(images, labels))
    assert got == {INFER_STAGED: 1}, got
    assert (cost, hits) == from_images["stats"]
    assert np.array_equal(model.get_params(), params)
