"""The feature stage's less travelled routes (csrc/features.cu), bit for bit against the oracle.

1. The layered path -- map sets too large for shared memory go image -> convert_images_kernel -> one kernel per stage over
   global ping-pong buffers -- at the c4 shape (bench.py's feature leg) and at shapes chosen for the streaming strip kernels'
   geometry: one or several strips, idle threads, empty strips, a row loop of two trips, a map staged in shared memory or
   read from global memory, generic stages between strip stages, the T = double path for u8 input past 10 convs, and the
   grid-stride image loop past gridDim.y = 32768.
2. f64 pixels on the layered and the fused kernel, with non-integer, infinite, huge and NaN pixels.
3. Epoch mode (device cursor + perm) through each stand-alone feature kernel: features_cp_kernel, features_fused_kernel and
   convert_images_kernel + the strip kernels, which must pick image perm[cursor + i] and write its label for the step.
4. gen_scales across blocks, against an exact reference.

The routes are restated below from features.cu's host code so that a CPU-only test keeps the case table honest, and every
GPU case asserts the kernels that ran (the library's launch profile).  The strip kernels' staged / unstaged choice does not
show in the profile; it is derived from the shape by the same rule, and the table covers both sides of it."""
import math
import zlib
from collections import Counter, namedtuple
from fractions import Fraction

import numpy as np
import pytest

import oracle as O
from conftest import assert_close

gpu = pytest.mark.gpu

CONV_NONE, CONV_SAME, POOL_MAX = 0, 1, 3   # RCN_LAYER_* codes
FUSED_SMEM_LIMIT = 200 * 1024              # kFusedSmemLimit
STRIP_STAGE_LIMIT = 48 * 1024              # a strip kernel's map goes through shared memory up to the default 48 KiB
IMAGE_GRID_CAP = 32768                     # gridDim.y of the layered kernels
SCALE_BLOCKS = 148 * 4                     # launch_gen_scales: at most kNumSMs * 4 blocks ...
SCALE_PER_BLOCK = 256 * 8                  # ... of 256 threads, 8 values per thread before the grid is capped

A_FEATS = "smallnet_fwd_bwd_kernel"        # kernel A on given features (no front end)
A_FUSED = "smallnet_fwd_bwd_kernel(fused features)"


# ---- features.cu's host-side routing, restated ----------------------------------------------------------------------
Stage = namedtuple("Stage", "kind same n_in h_in w_in n_out h_out w_out")
Strip = namedtuple("Strip", "rows n_strips sw staged")


def plan(cfg, H, W):
    """plan_features (features.cu:17-73): (stages, n_conv, max_elems).  kind 0 = conv, 1 = conv + pool, 2 = lone pool."""
    st, maps, h, w, i, n_conv, max_elems = [], 0, H, W, 0, 0, H * W
    while i < len(cfg):
        if cfg[i] in (CONV_NONE, CONV_SAME):
            same, n_in, h_in, w_in = cfg[i] == CONV_SAME, maps or 1, h, w
            if not same:
                h, w = h - 2, w - 2
            kind, maps, n_conv = 0, maps * 4 or 4, n_conv + 1
            if i + 1 < len(cfg) and cfg[i + 1] == POOL_MAX:   # a directly following pool is fused into the stage
                kind, h, w, i = 1, (h + 1) // 2, (w + 1) // 2, i + 1
            st.append(Stage(kind, same, n_in, h_in, w_in, maps, h, w))
        elif maps:                                            # pooling an empty feature set is a no-op
            st.append(Stage(2, True, maps, h, w, maps, (h + 1) // 2, (w + 1) // 2))
            h, w = (h + 1) // 2, (w + 1) // 2
        else:
            i += 1
            continue
        max_elems = max(max_elems, st[-1].n_in * st[-1].h_in * st[-1].w_in)
        i += 1
    return st, n_conv, max_elems


def cp_takes(st, n_conv, W):
    """make_cp_plan (features.cu:199-230) plus try_launch_features_cp's shared-memory limit: the staged kernel's stacks."""
    if not 1 <= len(st) <= 8 or n_conv > 10 or W % 4:
        return False
    off = 0
    for s in st:
        if s.kind != 1 or not s.same or s.h_out < 2:
            return False
        off += s.n_in * ((s.h_in + 4) & ~1) * (s.w_in + 3)
        if s.n_in * s.h_out * s.w_out >= 1 << 16 or off > 1 << 20:
            return False
    return True


def strip_geometry(h, w, stride):
    """conv_same_strips / launch_features_t: one CTA per input map, 256 threads as n_strips strips of `rows` rows."""
    rows = min(h, 256)
    n_strips = max(1, 256 // rows)
    staged = h * w * 4 <= STRIP_STAGE_LIMIT and (h * w) % 4 == 0 and stride % 4 == 0
    return Strip(rows, n_strips, -(-w // n_strips), staged)


def route(cfg, H, W, u8=True):
    """(launches of one flatten_feature_set call as a Counter of kernel names, [Strip per strip stage], T's size)."""
    st, n_conv, max_elems = plan(cfg, H, W)
    if u8 and cp_takes(st, n_conv, W):
        return Counter(["features_cp_kernel"]), [], 4
    t_size = 4 if u8 and n_conv <= 10 else 8
    if 2 * max_elems * t_size <= FUSED_SMEM_LIMIT:
        return Counter(["features_fused_kernel"]), [], t_size
    names, strips, stride = ["convert_images_kernel"], [], H * W
    for k, s in enumerate(st):
        last = k == len(st) - 1
        if t_size == 4 and s.kind == 0 and s.same and s.h_in >= 2:
            names.append("conv_same_final_kernel" if last else "conv_same_maps_kernel")
            strips.append(strip_geometry(s.h_in, s.w_in, stride))
        else:
            names.append("stage_final_kernel" if last else "stage_maps_kernel")
        stride = s.n_out * s.h_out * s.w_out
    return Counter(names), strips, t_size


def strip_columns(g, w):
    """[(first, end)] columns of each strip; an empty strip has first >= end."""
    return [(k * g.sw, min(w, k * g.sw + g.sw)) for k in range(g.n_strips)]


# ---- the u8 layered cases ---------------------------------------------------------------------------------------------
Case = namedtuple("Case", "name cfg hw B")
LAYERED = [
    Case("h300-two-row-trips", [1, 1, 1], (300, 40), 3),
    Case("h257-unstaged", [1, 1, 1], (257, 48), 3),
    Case("48KiB-one-strip", [1, 1, 1], (256, 48), 3),
    Case("48KiB-two-strips", [1, 1, 1], (128, 96), 3),
    Case("odd-map-idle-threads", [1, 1, 1], (101, 61), 3),
    Case("85-strips", [1, 1, 1], (3, 2000), 3),
    Case("convert-loops", [1, 1, 1], (130, 130), 3),
    Case("valid-between-strips", [1, 1, 0, 1], (64, 64), 3),
    Case("valid-first", [0, 1, 1, 1], (96, 96), 3),
    Case("leading-pool", [3, 1, 1, 1], (64, 64), 3),
    Case("conv-pool-then-pool", [1, 1, 1, 3, 3], (64, 64), 3),
    Case("ten-convs-int32-limit", [1] * 10, (3, 3), 3),
    Case("eleven-convs-f64", [1] * 11, (3, 3), 1),
]
C4 = Case("c4", [1, 1, 1, 1], (64, 64), 128)
GRID_STRIDE = Case("grid-stride", [1, 1, 3, 3, 3, 3, 3], (81, 81), IMAGE_GRID_CAP + 7)


def test_route_table_pins_what_it_claims():
    """CPU only: every case takes the layered path and reaches the geometry its name claims."""
    for c in LAYERED + [C4, GRID_STRIDE]:
        names, _, _ = route(c.cfg, *c.hw)
        assert "convert_images_kernel" in names, c.name
        n, h, w = O.feature_shape(c.cfg, *c.hw)
        st, _, _ = plan(c.cfg, *c.hw)
        assert n * h * w == st[-1].n_out * st[-1].h_out * st[-1].w_out, c.name
    geo = {c.name: route(c.cfg, *c.hw) for c in LAYERED + [C4, GRID_STRIDE]}

    def strips(name):
        return geo[name][1]

    s = strips("h300-two-row-trips")[0]
    assert s == Strip(256, 1, 40, True) and 300 > s.rows and 300 * 40 * 4 == 48000
    assert [g.staged for g in strips("h257-unstaged")] == [False] * 3 and 257 * 48 * 4 == 49344
    assert strips("48KiB-one-strip") == [Strip(256, 1, 48, True)] * 3
    assert strips("48KiB-two-strips") == [Strip(128, 2, 48, True)] * 3
    s = strips("odd-map-idle-threads")[0]
    assert s == Strip(101, 2, 31, False) and 256 - s.rows * s.n_strips == 54   # threads 202..255 idle
    s = strips("85-strips")[0]
    cols = strip_columns(s, 2000)
    assert s == Strip(3, 85, 24, True)
    assert cols[83] == (1992, 2000) and all(a >= b for a, b in cols[84:])   # a short last strip, then an empty one
    assert 130 * 130 > 64 * 256 and [g.staged for g in strips("convert-loops")] == [False] * 3
    assert geo["valid-between-strips"][0] == Counter({"convert_images_kernel": 1, "conv_same_maps_kernel": 2,
                                                      "stage_maps_kernel": 1, "conv_same_final_kernel": 1})
    assert geo["valid-first"][0] == Counter({"convert_images_kernel": 1, "stage_maps_kernel": 1, "conv_same_maps_kernel": 2,
                                             "conv_same_final_kernel": 1})
    assert geo["leading-pool"][0] == geo["c4"][0] - Counter({"conv_same_maps_kernel": 1})
    assert geo["conv-pool-then-pool"][0] == Counter({"convert_images_kernel": 1, "conv_same_maps_kernel": 2,
                                                     "stage_maps_kernel": 1, "stage_final_kernel": 1})
    s = strips("ten-convs-int32-limit")
    assert geo["ten-convs-int32-limit"][2] == 4 and len(s) == 10 and s[0] == Strip(3, 85, 1, False)
    assert sum(a < b for a, b in strip_columns(s[0], 3)) == 3                    # 82 of the 85 strips are empty
    assert route([1] * 10, 3, 3)[2] == 4 and route([1] * 11, 3, 3)[2] == 8   # int32 up to 10 convs (255 * 4^10)
    assert geo["eleven-convs-f64"][2] == 8 and not strips("eleven-convs-f64")
    assert strips("c4") == [Strip(64, 4, 16, True)] * 4
    assert geo["grid-stride"][0]["conv_same_maps_kernel"] == 1 and geo["grid-stride"][0]["stage_final_kernel"] == 1
    assert GRID_STRIDE.B > IMAGE_GRID_CAP
    all_strips = [g for _, ss, _ in geo.values() for g in ss]
    assert {g.staged for g in all_strips} == {True, False}
    assert {g.n_strips for g in all_strips} >= {1, 2, 4, 85}
    # the fused-kernel f64 case below really is fused, its layered twin really is layered
    assert route(F64_MIXED, 20, 20, u8=False)[0] == Counter(["features_fused_kernel"])
    assert route(F64_MIXED, 64, 64, u8=False)[0]["stage_final_kernel"] == 1
    assert route([1, 1, 1], 64, 64, u8=False)[0] == Counter({"convert_images_kernel": 1, "stage_maps_kernel": 2,
                                                            "stage_final_kernel": 1})


# ---- the exact gen_scales reference -----------------------------------------------------------------------------------
def exact_scales(s1, s2, n, ulp=Fraction(1)):
    """Values v_i = k_i * ulp (k_i integers, ulp a power of two) with s1 = sum k_i, s2 = sum k_i^2: the correctly rounded
    mean m, and sqrt(sum (v_i - m)^2 / n) for that double m, computed exactly and rounded once (plus sqrt's rounding)."""
    m = float(Fraction(s1, n) * ulp)
    K = Fraction(m) / ulp                                      # m = K * ulp exactly
    ss = (s2 - 2 * K * s1 + n * K * K) * ulp * ulp             # sum (v - m)^2, exact
    return m, math.sqrt(float(ss / n))


def int_sums(k):
    """(sum k_i, sum k_i^2, n) in Python integers: exact at any size."""
    k = np.asarray(k, dtype=np.int64).ravel().tolist()
    return sum(k), sum(x * x for x in k), len(k)


def test_exact_scales_reference():
    """CPU only: the reference against brute-force rationals, and against the oracle's sequential sums to rounding."""
    rng = np.random.default_rng(5)
    for n, lo, hi, e in [(1, 0, 65281, 0), (7, 0, 65281, 0), (2049, 0, 65281, 0), (300, -2 ** 40, 2 ** 40, 20)]:
        k = rng.integers(lo, hi, n)
        ulp = Fraction(1, 2 ** e)
        m, sd = exact_scales(*int_sums(k), ulp)
        vs = [int(x) * ulp for x in k]
        assert m == float(sum(vs) / n)
        assert sd == math.sqrt(float(sum((v - Fraction(m)) ** 2 for v in vs) / n))
        om, osd = O.gen_scales((k * float(ulp)).reshape(1, -1))
        scale = abs(m) if lo >= 0 else float(sum(abs(v) for v in vs) / n)
        assert abs(om - m) <= 1e-13 * scale and abs(osd - sd) <= 1e-13 * sd
    # a constant set: sd is exactly zero
    assert exact_scales(*int_sums(np.full(5, 9)))[1] == 0.0


# ---- GPU helpers ------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def api(built_library):
    import mercer_research_b200 as m
    return m


def layers(api, codes):
    return [api.RCNLayer.Convolve2D(api.Padding(c)) if c < 2 else api.RCNLayer.Pool2D(api.Pooling(c - 2)) for c in codes]


def bits_equal(a, b):
    a = np.ascontiguousarray(a, dtype=np.float64)
    b = np.ascontiguousarray(b, dtype=np.float64)
    return a.shape == b.shape and np.array_equal(a.view(np.uint64), b.view(np.uint64))


def dev_bits_equal(a, b):
    """Two torch float64 tensors on the device, bit for bit."""
    import torch
    return a.shape == b.shape and torch.equal(a.contiguous().view(torch.int64), b.contiguous().view(torch.int64))


def launched(fn):
    """(kernel launches by name, fn()) -- the library's launch profile around one call."""
    import torch
    from mercer_research_b200 import _lib
    torch.cuda.synchronize()
    _lib.profile_enable(True)
    try:
        out = fn()
        torch.cuda.synchronize()
        got = Counter({name: v["launches"] for name, v in _lib.profile_report().items()})
    finally:
        _lib.profile_enable(False)
    return got, out


def u8_images(c, seed=None):
    rng = np.random.default_rng(zlib.crc32(c.name.encode()) if seed is None else seed)
    imgs = rng.integers(0, 256, size=(c.B,) + c.hw, dtype=np.uint8)
    if c.B >= 3:                                     # the flat extreme and 255 / 0 stripes, then random images
        imgs[0] = 255
        imgs[1, ::2] = 255
        imgs[1, 1::2] = 0
    return imgs


# ---- 1. the u8 layered path -------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("c", LAYERED, ids=[c.name for c in LAYERED])
def test_layered_u8_bit_exact(api, c):
    imgs = u8_images(c)
    model = api.RCN(10, layers(api, c.cfg), [30])
    got_launches, got = launched(lambda: model.flatten_feature_set(imgs))
    assert got_launches == route(c.cfg, *c.hw)[0], (c.name, got_launches)
    assert bits_equal(got, O.features_u8(c.cfg, imgs)), c.name


@gpu
def test_c4_batch_standardised_into_device_out(api):
    """bench.py's feature leg: B = 128 64x64 images of [Conv(Same)]x4, standardised with (100, 50) into a preallocated
    device buffer; spot images against the oracle, and every image equal to the same image computed alone."""
    import torch
    c = C4
    imgs = u8_images(c)
    model = api.RCN(10, layers(api, c.cfg), [30])
    L = model.feature_len(*c.hw)
    few = imgs[:3]
    assert bits_equal(model.flatten_feature_set(few), O.features_u8(c.cfg, few))
    model.scale_set = (100.0, 50.0)
    d_imgs = torch.from_numpy(imgs).cuda()
    out = torch.empty((c.B, L), dtype=torch.float64, device="cuda")
    got_launches, ret = launched(lambda: model.flatten_feature_set(d_imgs, standardise=True, out=out))
    assert ret is out and got_launches == route(c.cfg, *c.hw)[0]
    spot = [0, 63, 64, 127]
    want = O.standardise(O.features_u8(c.cfg, imgs[spot]), 100.0, 50.0)
    assert bits_equal(out[spot].cpu().numpy(), want)
    one = torch.empty((1, L), dtype=torch.float64, device="cuda")
    for b in range(c.B):
        model.flatten_feature_set(d_imgs[b:b + 1], standardise=True, out=one)
        assert dev_bits_equal(one[0], out[b]), f"image {b} differs from itself computed alone"


@gpu
@pytest.mark.parametrize("cfg,hw,final", [([1, 1, 1], (64, 64), "conv_same_final_kernel"),
                                          ([1, 1, 1], (101, 61), "conv_same_final_kernel"),
                                          ([1, 1, 1, 3, 3], (64, 64), "stage_final_kernel")])
def test_layered_standardise_epilogue(api, cfg, hw, final):
    """The standardise + clamp epilogue of the final strip kernel and of the final generic kernel, with (100, 50) and
    with a perturbed (mean, sd) pair that the fast-division check may reject: IEEE division either way."""
    c = Case("std", cfg, hw, 4)
    imgs = u8_images(c, seed=hw[0] * 7 + len(cfg))
    raw = O.features_u8(cfg, imgs)
    mean, sd = O.gen_scales(raw)
    model = api.RCN(10, layers(api, cfg), [30])
    assert route(cfg, *hw)[0][final] == 1
    for pair in [(100.0, 50.0), (mean * 1.0000001, sd * 0.9999999)]:
        model.scale_set = pair
        got_launches, got = launched(lambda: model.flatten_feature_set(imgs, standardise=True))
        assert got_launches == route(cfg, *hw)[0]
        assert bits_equal(got, O.standardise(raw, *pair)), (cfg, hw, pair)


@gpu
def test_layered_scratch_growth_and_plan_cache(api):
    """One model called in turn with growing and shrinking batches and two image shapes: the layered scratch is grown, the
    plan recomputed, and neither leaks stale geometry into the next call."""
    cfg = [1, 1, 1]
    model = api.RCN(10, layers(api, cfg), [30])
    rng = np.random.default_rng(41)
    for B, hw in [(3, (64, 64)), (128, (64, 64)), (5, (64, 64)), (4, (101, 61)), (6, (64, 64))]:
        imgs = rng.integers(0, 256, size=(B,) + hw, dtype=np.uint8)
        got_launches, got = launched(lambda: model.flatten_feature_set(imgs))
        assert got_launches == route(cfg, *hw)[0]
        assert bits_equal(got, O.features_u8(cfg, imgs)), (B, hw)


@gpu
def test_layered_grid_stride_image_loop(api):
    """More images than gridDim.y (32768): the convert, strip, maps and final kernels walk the batch with a grid-stride loop.
    About 7 GB of layered scratch; the model is released at the end."""
    import torch
    c = GRID_STRIDE
    g = torch.Generator(device="cuda")
    g.manual_seed(43)
    d_imgs = torch.randint(0, 256, (c.B,) + c.hw, dtype=torch.uint8, device="cuda", generator=g)
    d_imgs[0] = 255
    model = api.RCN(10, layers(api, c.cfg), [30])
    try:
        got_launches, whole = launched(lambda: model.flatten_feature_set(d_imgs))
        assert got_launches == route(c.cfg, *c.hw)[0]
        spot = [0, IMAGE_GRID_CAP - 1, IMAGE_GRID_CAP, c.B - 1]
        assert bits_equal(whole[spot].cpu().numpy(), O.features_u8(c.cfg, d_imgs[spot].cpu().numpy()))
        for lo in range(0, c.B, IMAGE_GRID_CAP):
            part = model.flatten_feature_set(d_imgs[lo:lo + IMAGE_GRID_CAP])
            assert dev_bits_equal(part, whole[lo:lo + IMAGE_GRID_CAP]), f"images {lo}.. differ from the same chunk alone"
    finally:
        model.close()
        del d_imgs
        torch.cuda.empty_cache()


# ---- 2. f64 pixels ----------------------------------------------------------------------------------------------------
F64_MIXED = [1, 0, 3, 1]


def f64_images(n, hw, seed, specials):
    rng = np.random.default_rng(seed)
    imgs = rng.standard_normal((n,) + hw) * 37.0
    if specials == "inf-nan":
        flat = imgs.reshape(n, -1)
        for b in range(n):
            at = rng.choice(flat.shape[1], 24, replace=False)
            flat[b, at] = [np.inf, -np.inf, 1e300, -1e300, np.nan, 0.5] * 4
    elif specials == "overflow":
        # -1.5e308 above 1.5e308: the reference's 2 * 1.5e308 is +Inf before the -1.5e308 is added; a fused multiply-add
        # of the same taps would round 1.5e308 instead
        for b in range(n):
            for y, x in zip(rng.integers(1, hw[0] - 2, 6), rng.integers(0, hw[1] - 1, 6)):
                imgs[b, y, x], imgs[b, y + 1, x] = -1.5e308, 1.5e308
    return imgs


@gpu
@pytest.mark.parametrize("cfg,hw", [([1, 1, 1], (64, 64)), (F64_MIXED, (64, 64)), (F64_MIXED, (20, 20))])
@pytest.mark.parametrize("specials", ["none", "inf-nan", "overflow"])
def test_f64_pixels_bit_exact(api, cfg, hw, specials):
    """Non-integer pixels through T = double (layered at 64x64, fused at 20x20); with +-Inf, +-1e300 and NaN pixels the
    reference's zero taps turn Inf into NaN and ReLU maps NaN to 0, so every output is finite or +Inf; and pixels whose
    doubled tap overflows, where only a separately rounded multiply and add reproduce the reference."""
    imgs = f64_images(3, hw, seed=hw[0] + len(cfg), specials=specials)
    want = np.stack([O.flatten_feature_set(cfg, im) for im in imgs])
    model = api.RCN(10, layers(api, cfg), [30])
    got_launches, got = launched(lambda: model.flatten_feature_set(imgs))
    assert got_launches == route(cfg, *hw, u8=False)[0]
    assert bits_equal(got, want), (cfg, hw, specials)
    assert (want >= 0).all()                         # finite or +Inf: no NaN reaches the output


# ---- 3. epoch mode through the stand-alone feature kernels -------------------------------------------------------------
Net = namedtuple("Net", "name cfg hw pixels hidden B N kernels")
EPOCH_NETS = [
    # 40 hidden units: smallnet_eligible allows 32 rows, so the generic dense step runs after features_cp_kernel
    Net("cp-u8-hidden40", [1, 3], (28, 28), "u8", [40], 64, 64 * 4 + 23, {"features_cp_kernel"}),
    # f64 pixels never run a front end inside kernel A
    Net("fused-f64", [1, 3], (28, 28), "f64", [30], 64, 64 * 4 + 23, {"features_fused_kernel", A_FEATS}),
    # the layered path: the front end does not fit kernel A, the head does
    Net("layered-u8-64x64", [1, 1, 1], (64, 64), "u8", [30], 8, 8 * 3 + 5,
        {"convert_images_kernel", "conv_same_maps_kernel", "conv_same_final_kernel", A_FEATS}),
]
ETA = 3.0


def epoch_data(n):
    rng = np.random.default_rng(zlib.crc32(n.name.encode()))
    if n.pixels == "u8":
        imgs = rng.integers(0, 256, size=(n.N,) + n.hw, dtype=np.uint8)
        feats = lambda x: O.features_u8(n.cfg, x)                             # noqa: E731
    else:
        imgs = rng.standard_normal((n.N,) + n.hw) * 37.0
        feats = lambda x: np.stack([O.flatten_feature_set(n.cfg, im) for im in x])  # noqa: E731
    labels = rng.integers(0, 10, n.N).astype(np.int64)
    perm = rng.permutation(n.N).astype(np.int64)
    return imgs, labels, perm, feats


@gpu
@pytest.mark.parametrize("n", EPOCH_NETS, ids=[n.name for n in EPOCH_NETS])
def test_epoch_mode_through_feature_kernels(api, n):
    """epoch_bind with a perm (N not a multiple of B), epoch_step past the wrap, then epoch_run for two more steps ==
    train_batch_images on the perm's chunks, bit for bit (parameters, last_batch_stats, cursor); one step against the
    oracle, with labels of which half are the oracle's predictions so that the hit count sees every label."""
    import torch
    imgs, labels, perm, feats = epoch_data(n)
    chunks = n.N // n.B
    seek = (chunks - 1) * n.B                        # the oracle step: the last full chunk before the wrap
    sel = perm[seek:seek + n.B]
    X_raw = feats(imgs[sel])
    scale = O.gen_scales(X_raw)
    X = O.standardise(X_raw, *scale)
    rows = n.hidden + [10]
    shapes = list(zip(rows, [X_raw.shape[1]] + rows[:-1]))
    net = O.Net(shapes)
    rng = np.random.default_rng(7)
    params = np.concatenate([np.concatenate([rng.standard_normal(r * k) * (2.0 / np.sqrt(k)), rng.standard_normal(r) * 0.5])
                             for r, k in shapes])
    labels[sel[::2]] = O.argmax_last(net.forward(params, X))[::2]

    def fresh():
        m = api.RCN(10, layers(api, n.cfg), n.hidden)
        m.load_weights_and_bias_shapes(shapes)
        m.set_params(params)
        m.scale_set = scale
        return m

    n_steps = chunks + 1 + 2
    ref = fresh()
    for k in range(n_steps):
        idx = perm[(k % chunks) * n.B:(k % chunks + 1) * n.B]
        ref.train_batch_images(imgs[idx], labels[idx], ETA)
    d_imgs, d_labels, d_perm = (torch.from_numpy(a).cuda() for a in (imgs, labels, perm))
    ep = fresh()
    ep.epoch_bind(d_imgs, d_labels, n.B, perm=d_perm)
    names, _ = launched(lambda: ep.epoch_step(ETA))
    assert n.kernels <= set(names), (n.name, names)
    assert A_FUSED not in names, (n.name, names)
    if n.name.startswith("cp"):
        assert not any(k.startswith("smallnet") for k in names), (n.name, names)
    for _ in range(chunks):
        ep.epoch_step(ETA)
    assert ep.epoch_position() == n.B                # wrapped: the remainder of N % B samples is dropped
    ep.epoch_run(ETA, 2)
    assert ep.epoch_position() == (n_steps % chunks) * n.B
    assert np.array_equal(ep.get_params(), ref.get_params()), n.name
    assert ep.last_batch_stats() == ref.last_batch_stats(), n.name

    one = fresh()
    one.epoch_bind(d_imgs, d_labels, n.B, perm=d_perm)
    one.epoch_seek(seek)
    one.epoch_step(ETA)
    want, _ = net.train_batch(params, X, np.eye(10)[labels[sel]], ETA)
    assert_close(one.get_params(), want, what=f"{n.name}: params after one epoch step")
    acts = net.forward(params, X)
    cost, hits = one.last_batch_stats()
    assert hits == O.accuracy(acts, labels[sel]) and hits >= 1, (n.name, hits)
    assert abs(cost - 0.5 * np.sum((acts - np.eye(10)[labels[sel]]) ** 2)) <= 1e-9 * max(1.0, cost)
    assert one.epoch_position() == 0


# ---- 4. gen_scales across blocks ---------------------------------------------------------------------------------------
GRID_CAP_N = SCALE_PER_BLOCK * SCALE_BLOCKS      # 1 212 416: the last size with 8 values per thread


def check_scales(got, want, scale, what, report):
    (gm, gs), (m, sd) = got, want
    report.append(f"{what}: mean rel {abs(gm - m) / max(scale, 1e-300):.2e}, sd rel {abs(gs - sd) / max(sd, 1e-300):.2e}")
    assert abs(gm - m) <= 1e-12 * scale, (what, gm, m)
    assert abs(gs - sd) <= 1e-12 * sd, (what, gs, sd)


@gpu
def test_gen_scales_across_blocks(api):
    """Mean and population sd of raw u8 features (integers: exact sums) at one block, the block boundary, more blocks than
    one final pass of 256 threads covers, the grid cap and one past it; and of a signed non-integer set.  Bar: 1e-12
    relative to the exact values (to sum |v| / n for the signed set's mean).  How the oracle's sequential sums compare is
    printed, not asserted."""
    model = api.RCN(10, layers(api, [1, 3]), [30])
    rng = np.random.default_rng(47)
    report = []
    for n in [1, 2047, 2048, 2049, 2048 * 257, GRID_CAP_N, GRID_CAP_N + 1]:
        k = rng.integers(0, 65281, n) * (rng.random(n) < 0.6)          # ReLU'd: many zeros
        v = k.astype(np.float64).reshape(1, n)
        want = exact_scales(*int_sums(k))
        got_launches, got = launched(lambda: model.gen_scales(v))
        assert got_launches == Counter({"scale_partial_kernel": 2, "scale_final_kernel": 2})
        check_scales(got, want, abs(want[0]), f"n={n}", report)
        om, osd = O.gen_scales(v)
        report.append(f"n={n} oracle sequential: mean rel {abs(om - want[0]) / max(want[0], 1e-300):.2e}, "
                      f"sd rel {abs(osd - want[1]) / max(want[1], 1e-300):.2e}")
    e = 20
    k = rng.integers(-2 ** 40, 2 ** 40, GRID_CAP_N + 1)                # v = k / 2^20: signed, non-integer, exact sums
    v = (k * 2.0 ** -e).reshape(1, -1)
    want = exact_scales(*int_sums(k), Fraction(1, 2 ** e))
    check_scales(model.gen_scales(v), want, float(np.abs(v).mean()), "signed", report)
    print("\n".join(report))


@gpu
def test_gen_scales_c4_batch_on_device(api):
    """The c4 batch, 128 x 2^20 raw features (134 M values) as a device tensor; exact sums in int64 on the device."""
    import torch
    g = torch.Generator(device="cuda")
    g.manual_seed(53)
    k = torch.randint(0, 65281, (128, 1 << 20), dtype=torch.int64, device="cuda", generator=g)
    k = k * (torch.rand(k.shape, device="cuda", generator=g) < 0.6)
    s1, s2 = int(k.sum()), int((k * k).sum())
    assert s2 < 2 ** 62
    v = k.to(torch.float64)
    del k
    model = api.RCN(10, layers(api, [1, 1, 1, 1]), [30])
    want = exact_scales(s1, s2, v.numel())
    report = []
    check_scales(model.gen_scales(v), want, want[0], f"n={v.numel()}", report)
    om, osd = O.gen_scales(v.cpu().numpy())
    report.append(f"oracle sequential: mean rel {abs(om - want[0]) / want[0]:.2e}, sd rel {abs(osd - want[1]) / want[1]:.2e}")
    print("\n".join(report))
    del v
    torch.cuda.empty_cache()
