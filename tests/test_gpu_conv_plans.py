"""The f64 convolution kernels of csrc/conv.cu on every tile, split and direct-kernel plan, with non-finite pixels, and at
dataset-sized batches.

Shapes are chosen with a restatement of the host plan (``use_direct``, ``launch_gemm_tiles``' tile rule, the split rule of
``launch_conv2d_backward_weight`` and ``split_plan``) and every case asserts, with the library's launch profiler, which
kernels ran and how often, so a shape cannot quietly move to another engine.  The profiler names kernels, not tiles: the
tile a case lands on rests on the restatement, which each case prints.

Bars: the shared own-magnitude 1e-9 (``assert_close``) against oracle/ext.py (C++ f64 loops) for every case that fits the
oracle (under ~0.3 GFLOP per op); at dataset sizes the reference is torch in float64 on the same GPU, own-magnitude 1e-9
for forward and backward-data, componentwise 1e-9 (against the same op on absolute values, DESIGN.md section 2) for the
8.4 M-pixel weight gradient.  Cases that move more than 1 GB have ``large`` in their id (``-k "not large"``)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle.ext as E
from conftest import assert_close

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NUM_SMS, KT, DT, MAX_GRID_YZ = 148, 16, 16, 65535
NONE, SAME = 0, 1


# -- the host plan, restated ---------------------------------------------------------------------------------------------
def cdiv(a, b):
    return -(-a // b)


def out_hw(H, W, kh, kw, pad):
    return (H, W) if pad == SAME else (H - kh + 1, W - kw + 1)


def direct_smem(Ci, Co, kh, kw):
    return ((DT + kh - 1) * (DT + kw - 1) * Ci + Co * kh * kw * Ci) * 8


def use_direct(Ci, Co, kh, kw):
    return kh * kw * Ci <= 64 and direct_smem(Ci, Co, kh, kw) <= 96 * 1024


def split_plan(K, splits):
    splits = max(splits, 1)
    kps = max(cdiv(cdiv(K, splits), KT) * KT, KT)
    return (cdiv(K, kps) if K > 0 else 1), kps


def gemm_tile(M, N, splits=1):
    if M <= 32:
        return (32, 128)
    return (128, 128) if cdiv(M, 128) * cdiv(N, 128) * splits >= NUM_SMS * 7 // 8 else (64, 64)


def wgrad_splits(Co, n_k, Kc):
    if Co <= 32:
        tiles = cdiv(n_k, 128)
    else:
        tiles = cdiv(Co, 128) * cdiv(n_k, 128)
        if tiles < NUM_SMS:
            tiles = cdiv(Co, 64) * cdiv(n_k, 64)
    splits = 1
    if tiles < NUM_SMS:
        splits = min(cdiv(2 * NUM_SMS, tiles), max(Kc // 64, 1), 128)
    return split_plan(Kc, splits)[0]


def plan(B, H, W, Ci, Co, kh, kw, pad):
    """Engine, tile and launch count of each pass (the DMMA grid holds at most MAX_GRID_YZ column tiles per launch)."""
    Ho, Wo = out_hw(H, W, kh, kw, pad)
    n_fwd, n_bwd, Kc, n_k = B * Ho * Wo, B * H * W, B * Ho * Wo, kh * kw * Ci
    fwd_tile, bwd_tile = gemm_tile(Co, n_fwd), gemm_tile(Ci, n_bwd)
    splits = wgrad_splits(Co, n_k, Kc)
    return dict(fwd="direct" if use_direct(Ci, Co, kh, kw) else fwd_tile,
                fwd_launches=1 if use_direct(Ci, Co, kh, kw) else cdiv(cdiv(n_fwd, fwd_tile[1]), MAX_GRID_YZ),
                bwd=bwd_tile, bwd_launches=cdiv(cdiv(n_bwd, bwd_tile[1]), MAX_GRID_YZ),
                wgrad=gemm_tile(Co, n_k, splits), wgrad_splits=splits, direct_smem=direct_smem(Ci, Co, kh, kw))


def test_plan_restatement_examples():
    """Hand-worked points of the plan, so an edit of the restatement cannot drift silently."""
    assert split_plan(9000, 128) == (113, 80)
    assert wgrad_splits(8, 72, 9 * 25 * 40) == 113
    assert wgrad_splits(256, 2880, 200) == 1
    assert gemm_tile(129, 9 * 32 * 32) == (128, 128) and gemm_tile(33, 234) == (64, 64) and gemm_tile(32, 10 ** 7) == (32, 128)
    assert plan(8192, 32, 32, 16, 32, 3, 3, SAME)["fwd_launches"] == 2 and plan(8191, 32, 32, 16, 32, 3, 3, SAME)["fwd_launches"] == 1


# -- helpers ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def X(built_library):
    from mercer_research_b200 import ext
    return ext


def _profile(fn):
    """{kernel name: launches} of everything the library launched inside fn."""
    from mercer_research_b200 import _lib
    _lib.profile_enable(True)
    try:
        out = fn()
        rep = _lib.profile_report()
    finally:
        _lib.profile_enable(False)
    return out, {k: v["launches"] for k, v in rep.items()}


def _flops(B, H, W, Ci, Co, kh, kw, pad):
    Ho, Wo = out_hw(H, W, kh, kw, pad)
    return 2 * B * Ho * Wo * kh * kw * Ci * Co


def _assert_nonfinite_match(got, want, what):
    """Non-finite exactly where the oracle is (same sign for the infinities); the finite rest to the 1e-9 bar."""
    got, want = np.asarray(got), np.asarray(want)
    assert np.array_equal(np.isnan(got), np.isnan(want)), f"{what}: NaN positions differ"
    inf = np.isinf(want)
    assert np.array_equal(np.isinf(got), inf), f"{what}: infinity positions differ"
    assert np.array_equal(np.sign(got[inf]), np.sign(want[inf])), f"{what}: infinity signs differ"
    fin = np.isfinite(want)
    assert 0 < fin.sum() < want.size
    assert_close(got[fin], want[fin], what=what + " (finite part)")


def _close_dev(got, want, rtol=1e-9, what="", bound=None, step=512):
    """assert_close on device tensors without host copies, in chunks along dim 0.  With ``bound`` (same shape) the bar is
    componentwise, |got - want| <= rtol * bound, instead of own-magnitude."""
    import torch
    scale = float(want.abs().max())
    n_bad, worst = 0, 0.0
    for i in range(0, want.shape[0], step):
        g, w = got[i:i + step], want[i:i + step]
        lim = rtol * (bound[i:i + step] if bound is not None else w.abs() + 1e-3 * scale)
        err = (g - w).abs()
        bad = (err > lim) | ~torch.isfinite(g)
        n_bad += int(bad.sum())
        worst = max(worst, float((err / lim.clamp_min(1e-300)).max()))
    assert n_bad == 0, f"{what}: {n_bad}/{want.numel()} elements off (worst err/bar {worst:.3e})"


def _free():
    import gc
    import torch
    gc.collect()
    torch.cuda.empty_cache()


# -- A. the DMMA implicit GEMMs on every plan, against the oracle --------------------------------------------------------
IGEMM_CASES = {
    # id: (B, H, W, Ci, Co, kh, kw, pad)
    "tile32x128": (2, 12, 11, 16, 24, 3, 3, SAME),
    "tile64-M33": (2, 9, 13, 33, 33, 3, 3, SAME),
    "tile64-M64": (2, 9, 13, 64, 64, 3, 3, SAME),
    "tile64-M65": (2, 9, 13, 65, 65, 3, 3, SAME),
    "tile64-M128": (2, 9, 13, 128, 128, 3, 3, NONE),
    "tile64-M129": (2, 9, 13, 129, 129, 3, 3, SAME),
    "tile128-forward": (9, 32, 32, 8, 129, 3, 3, SAME),       # 2 x 72 = 144 tiles of 128 x 128
    "tile128-backward-data": (9, 32, 32, 129, 8, 3, 3, SAME),
    "tile128-wgrad": (9, 32, 32, 16, 64, 3, 3, SAME),         # Im2colPixelK with 128 rows: 1 x 2 x 96 splits
    "K75-5x5-Ci3": (2, 14, 19, 3, 40, 5, 5, SAME),
    "K65-1x1-Ci65": (3, 10, 7, 65, 48, 1, 1, NONE),
    "K81-3x3-Ci9": (2, 15, 11, 9, 70, 3, 3, NONE),
    "rect1x7": (2, 11, 17, 16, 40, 1, 7, SAME),
    "rect7x1": (2, 17, 11, 16, 40, 7, 1, SAME),
    "rect5x3": (2, 13, 21, 8, 36, 5, 3, SAME),
    "even2x4-none": (2, 10, 13, 16, 40, 2, 4, NONE),
    "even4x2-none": (2, 13, 10, 16, 24, 4, 2, NONE),
    "kh=H": (3, 5, 19, 8, 40, 5, 3, NONE),
    "kw=W": (3, 19, 6, 8, 40, 3, 6, NONE),
    "wgrad-one-split": (2, 10, 10, 320, 256, 3, 3, SAME),    # 4 x 45 = 180 tiles of 64 x 64 >= 148: no split
    "wgrad-splits-capped-by-Kc": (2, 10, 10, 16, 16, 3, 3, SAME),   # Kc = 200: 200 / 64 = 3 splits
    "wgrad-128-splits-lowered": (9, 25, 40, 8, 8, 3, 3, SAME),      # Kc = 9000: 128 -> split_plan -> 113
}
EXPECTED_SPLITS = {"wgrad-one-split": 1, "wgrad-splits-capped-by-Kc": 3, "wgrad-128-splits-lowered": 113, "tile128-wgrad": 96}


@pytest.mark.parametrize("cid", list(IGEMM_CASES))
def test_igemm_plan_against_oracle(X, cid):
    case = IGEMM_CASES[cid]
    B, H, W, Ci, Co, kh, kw, pad = case
    p = plan(*case)
    print(cid, case, p)
    assert p["fwd"] != "direct" and _flops(*case) < 0.3e9
    if cid in EXPECTED_SPLITS:
        assert p["wgrad_splits"] == EXPECTED_SPLITS[cid]
    if cid.startswith("tile"):
        want_tile = {"tile32x128": (32, 128), "tile64": (64, 64), "tile128": (128, 128)}[cid.split("-")[0]]
        key = {"backward-data": "bwd", "wgrad": "wgrad"}.get(cid.split("-", 1)[-1], "fwd")
        assert p[key] == want_tile, (key, p)
    rng = np.random.default_rng(sum(map(ord, cid)))
    Ho, Wo = out_hw(H, W, kh, kw, pad)
    x = rng.standard_normal((B, H, W, Ci))
    w = rng.standard_normal((Co, kh, kw, Ci)) / np.sqrt(kh * kw * Ci)
    b = rng.standard_normal(Co)
    dz = rng.standard_normal((B, Ho, Wo, Co))
    act = len(cid) % 3

    y, k = _profile(lambda: X.conv2d_forward(x, w, b, pad, act))
    assert k == {"conv2d_forward_igemm": p["fwd_launches"]}, k
    assert_close(y, E.conv2d_forward(x, w, b, pad, act), what=f"{cid} forward")

    dx, k = _profile(lambda: X.conv2d_backward_data(dz, w, (H, W), pad))
    assert k == {"conv_flip_weights_kernel": 1, "conv2d_backward_data_igemm": p["bwd_launches"]}, k
    want_dx = E.conv2d_backward_data(dz, w, (H, W), pad)
    assert_close(dx, want_dx, what=f"{cid} backward-data")
    yprev = 1 / (1 + np.exp(-rng.standard_normal((B, H, W, Ci))))
    assert_close(X.conv2d_backward_data(dz, w, (H, W), pad, y_prev=yprev, activation_prev=2),
                 E.activation_backward(yprev, want_dx, 2), what=f"{cid} backward-data with fused y_prev")

    (dw, db), k = _profile(lambda: X.conv2d_backward_weight(x, dz, kh, kw, pad))
    assert k.get("conv2d_backward_weight_igemm") == 1 and "bias_grad_kernel" in k, k
    assert ("reduce_splits_kernel" in k) == (p["wgrad_splits"] > 1), k
    assert set(k) <= {"conv2d_backward_weight_igemm", "bias_grad_kernel", "reduce_splits_kernel"}, k
    wdw, wdb = E.conv2d_backward_weight(x, dz, kh, kw, pad)
    assert_close(dw, wdw, what=f"{cid} backward-weight")
    assert_close(db, wdb, what=f"{cid} bias gradient")
    if cid.startswith("wgrad"):
        dw2, db2 = X.conv2d_backward_weight(x, dz, kh, kw, pad)
        assert np.array_equal(dw, dw2) and np.array_equal(db, db2), "split-K weight gradient is not run-to-run identical"


# -- B. the direct kernel --------------------------------------------------------------------------------------------------
DIRECT_CASES = {
    "33x47-Ci1-Co5": (3, 33, 47, 1, 5, 3, 3, SAME),
    "33x47-Ci2-Co13-5x5-none": (2, 33, 47, 2, 13, 5, 5, NONE),
    "40x16-Ci3-Co136": (2, 40, 16, 3, 136, 3, 3, SAME),
    "40x16-Ci4-Co8": (3, 40, 16, 4, 8, 3, 3, NONE),
    "40x16-Ci1-Co136-7x7-none-smem-attr": (2, 40, 16, 1, 136, 7, 7, NONE),
    "33x47-Ci1-Co136-7x7-same-smem-attr": (2, 33, 47, 1, 136, 7, 7, SAME),
}


@pytest.mark.parametrize("cid", list(DIRECT_CASES))
def test_direct_kernel_against_oracle(X, cid):
    case = DIRECT_CASES[cid]
    B, H, W, Ci, Co, kh, kw, pad = case
    p = plan(*case)
    print(cid, case, p)
    assert p["fwd"] == "direct"
    assert (p["direct_smem"] > 48 * 1024) == cid.endswith("smem-attr")
    rng = np.random.default_rng(sum(map(ord, cid)))
    x = rng.standard_normal((B, H, W, Ci))
    w = rng.standard_normal((Co, kh, kw, Ci)) / np.sqrt(kh * kw * Ci)
    b = rng.standard_normal(Co)
    for act in (0, 1, 2):
        y, k = _profile(lambda: X.conv2d_forward(x, w, b if act else None, pad, act))
        assert k == {"conv2d_direct_small_kernel": 1}, k
        assert_close(y, E.conv2d_forward(x, w, b if act else None, pad, act), what=f"{cid} act {act}")


def test_direct_u8_kernel_through_convnet():
    """The u8 direct kernel is only reachable through the handle: a one-conv network on 33 x 47 u8 images, Co = 13."""
    import mercer_research_b200 as m
    net = m.ConvNet((33, 47, 1), [m.Conv(13, 3, 3, m.Padding.Same)], [8], 10)
    try:
        rng = np.random.default_rng(21)
        params = net.init_params(rng)
        (name, sl, shp), (_, slb, _) = net.param_slices()[:2]
        images = rng.integers(0, 256, size=(5, 33, 47), dtype=np.uint8)
        _, k = _profile(lambda: net.classify_images(images))
        assert k.get("conv2d_direct_small_u8_kernel") == 1, k
        want = E.conv2d_forward(images.astype(np.float64)[..., None], params[sl].reshape(shp), params[slb], SAME, E.ACT_RELU)
        assert_close(net.layer_output(0), want, what="u8 direct kernel")
    finally:
        net.close()


def test_direct_kernel_equals_igemm_multi_tile(tmp_path):
    """One multi-tile small-channel shape through the direct kernel and, with RCN_CUDA_CONV_DIRECT=0, the implicit GEMM."""
    code = ("import sys, json, numpy as np; sys.path.insert(0, %r); from mercer_research_b200 import ext, _lib;"
            "rng = np.random.default_rng(5); x = rng.standard_normal((3, 33, 47, 3)); w = rng.standard_normal((13, 3, 3, 3));"
            "b = rng.standard_normal(13); _lib.profile_enable(True); y = ext.conv2d_forward(x, w, b, 1, 1);"
            "k = sorted(_lib.profile_report()); np.save(sys.argv[1], y); print(json.dumps(k))") % ROOT
    outs, kernels = [], []
    for flag in ("1", "0"):
        path = str(tmp_path / f"y{flag}.npy")
        r = subprocess.run([sys.executable, "-c", code, path], env=dict(os.environ, RCN_CUDA_CONV_DIRECT=flag),
                           capture_output=True, text=True, check=True)
        kernels.append(json.loads(r.stdout.strip().splitlines()[-1]))
        outs.append(np.load(path))
    assert kernels == [["conv2d_direct_small_kernel"], ["conv2d_forward_igemm"]], kernels
    assert_close(outs[0], outs[1], what="direct vs implicit GEMM")


# -- C. non-finite pixels --------------------------------------------------------------------------------------------------
NONFINITE_CASES = {"direct-same": (2, 20, 37, 2, 5, 3, 3, SAME), "direct-none": (2, 20, 37, 1, 13, 5, 3, NONE),
                   "igemm-same": (2, 20, 37, 16, 24, 3, 3, SAME), "igemm-none": (2, 20, 37, 12, 40, 3, 5, NONE)}


def _poison(a, rng):
    """NaN, +Inf and -Inf at interior, edge and corner pixels of an NHWC array (in place)."""
    B, H, W, C = a.shape
    spots = [(0, H // 2, W // 2, np.nan), (1, H // 3, 2 * W // 3, np.inf), (0, H // 2 + 1, W // 2 + 6, -np.inf),
             (0, 0, W // 3, np.inf), (1, H - 1, W // 4, -np.inf), (1, H // 2, 0, np.nan), (0, 3, W - 1, -np.inf),
             (0, 0, 0, np.nan), (1, H - 1, W - 1, np.inf), (0, H - 1, 0, -np.inf), (1, 0, W - 1, np.inf)]
    for b, y, x, v in spots:
        a[b, y, x, rng.integers(0, C)] = v


@pytest.mark.parametrize("cid", list(NONFINITE_CASES))
def test_nonfinite_pixels(X, cid):
    case = NONFINITE_CASES[cid]
    B, H, W, Ci, Co, kh, kw, pad = case
    p = plan(*case)
    print(cid, case, p)
    assert (p["fwd"] == "direct") == cid.startswith("direct")
    rng = np.random.default_rng(sum(map(ord, cid)))
    Ho, Wo = out_hw(H, W, kh, kw, pad)
    x = rng.standard_normal((B, H, W, Ci))
    w = rng.standard_normal((Co, kh, kw, Ci))
    b = rng.standard_normal(Co)
    dz = rng.standard_normal((B, Ho, Wo, Co))
    _poison(x, rng)
    _poison(dz, rng)
    y, k = _profile(lambda: X.conv2d_forward(x, w, b, pad, 0))
    assert set(k) == {"conv2d_direct_small_kernel" if cid.startswith("direct") else "conv2d_forward_igemm"}, k
    _assert_nonfinite_match(y, E.conv2d_forward(x, w, b, pad, 0), f"{cid} forward")
    dx, k = _profile(lambda: X.conv2d_backward_data(dz, w, (H, W), pad))
    assert set(k) == {"conv_flip_weights_kernel", "conv2d_backward_data_igemm"}, k
    _assert_nonfinite_match(dx, E.conv2d_backward_data(dz, w, (H, W), pad), f"{cid} backward-data")


# -- D. dataset-sized batches on the device, against torch f64 --------------------------------------------------------------
def _dev_randn(shape, seed, scale=1.0):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn(shape, dtype=torch.float64, device="cuda", generator=g) * scale


def _oracle_images(got, idx, fn):
    for i in idx:
        assert_close(got[i:i + 1].cpu().numpy(), fn(i), what=f"image {i} against the oracle")


LARGE_TILE_CASES = [
    pytest.param((8191, 32, 32, 16, 32), id="large-B8191-65528-tile-rows"),
    pytest.param((8192, 32, 32, 16, 32), id="large-B8192-65536-tile-rows"),
    pytest.param((9321, 30, 30, 8, 32), id="large-B9321-partial-last-tile-row"),
]


@pytest.mark.parametrize("case", LARGE_TILE_CASES)
def test_large_forward_backward_data_across_tile_limit(X, case):
    import torch
    import torch.nn.functional as F
    B, H, W, Ci, Co = case
    p = plan(B, H, W, Ci, Co, 3, 3, SAME)
    N = B * H * W
    print(case, p, "pixels", N, "tile rows", cdiv(N, 128))
    assert p["fwd"] == (32, 128) and p["bwd"] == (32, 128) and 9 * Ci < 256   # DMMA, not tcgen05 (K < 256)
    x = _dev_randn((B, H, W, Ci), 1)
    w = _dev_randn((Co, 3, 3, Ci), 2, 1 / np.sqrt(9 * Ci))
    b = _dev_randn((Co,), 3)
    nchw = lambda t: t.permute(0, 3, 1, 2)
    nhwc = lambda t: t.permute(0, 2, 3, 1)

    y, k = _profile(lambda: X.conv2d_forward(x, w, b, SAME, 0))
    assert k == {"conv2d_forward_igemm": p["fwd_launches"]}, k
    _close_dev(y, nhwc(F.conv2d(nchw(x), nchw(w), b, padding=1)), what="forward vs torch f64")
    wn, bn = w.cpu().numpy(), b.cpu().numpy()
    _oracle_images(y, (0, B // 2, B - 1), lambda i: E.conv2d_forward(x[i:i + 1].cpu().numpy(), wn, bn, SAME, 0))
    del y
    _free()

    dz = _dev_randn((B, H, W, Co), 4)
    dx, k = _profile(lambda: X.conv2d_backward_data(dz, w, (H, W), SAME))
    assert k == {"conv_flip_weights_kernel": 1, "conv2d_backward_data_igemm": p["bwd_launches"]}, k
    ref = nhwc(torch.nn.grad.conv2d_input((B, Ci, H, W), nchw(w), nchw(dz), padding=1))
    _close_dev(dx, ref, what="backward-data vs torch f64")
    _oracle_images(dx, (0, B // 2, B - 1), lambda i: E.conv2d_backward_data(dz[i:i + 1].cpu().numpy(), wn, (H, W), SAME))
    del dx, ref, dz, x
    _free()


def test_large_backward_weight_8192_images(X):
    """dW over 8.4 M pixels: 128 splits of the pixel contraction, combined in split order.  Componentwise bar against
    torch on |dz| and |x|; an all-positive input, where the two bars coincide, against assert_close."""
    import torch
    B, H, W, Ci, Co = 8192, 32, 32, 16, 32
    p = plan(B, H, W, Ci, Co, 3, 3, SAME)
    print(p)
    assert p["wgrad_splits"] == 128 and p["wgrad"] == (32, 128)
    nchw = lambda t: t.permute(0, 3, 1, 2)
    x = _dev_randn((B, H, W, Ci), 11)
    dz = _dev_randn((B, H, W, Co), 12)

    def ref(xa, dza):
        dw = torch.nn.grad.conv2d_weight(nchw(xa), (Co, Ci, 3, 3), nchw(dza), padding=1).permute(0, 2, 3, 1)
        return dw.contiguous(), dza.sum(dim=(0, 1, 2))

    (dw, db), k = _profile(lambda: X.conv2d_backward_weight(x, dz, 3, 3, SAME))
    assert k.get("conv2d_backward_weight_igemm") == 1 and k.get("reduce_splits_kernel") == 1 and "bias_grad_kernel" in k, k
    assert not any("tcgen05" in n for n in k), k
    dw2, db2 = X.conv2d_backward_weight(x, dz, 3, 3, SAME)
    assert torch.equal(dw, dw2) and torch.equal(db, db2), "weight gradient is not run-to-run identical"
    want_w, want_b = ref(x, dz)
    bound_w, bound_b = ref(x.abs(), dz.abs())
    _close_dev(dw, want_w, bound=bound_w, what="dW, componentwise")
    _close_dev(db, want_b, bound=bound_b, what="db, componentwise")
    x.abs_()
    dz.abs_()
    dw, db = X.conv2d_backward_weight(x, dz, 3, 3, SAME)
    want_w, want_b = ref(x, dz)
    assert_close(dw.cpu().numpy(), want_w.cpu().numpy(), what="dW, all-positive input")
    assert_close(db.cpu().numpy(), want_b.cpu().numpy(), what="db, all-positive input")
    del x, dz
    _free()


def test_large_direct_kernel_past_65535_images(X):
    """70 000 single-channel 28 x 28 images in one call: each image bit-identical to a call of 1 000 images."""
    import torch
    B, Co = 70000, 8
    assert plan(B, 28, 28, 1, Co, 3, 3, SAME)["fwd"] == "direct"
    x = _dev_randn((B, 28, 28, 1), 21)
    w = _dev_randn((Co, 3, 3, 1), 22)
    b = _dev_randn((Co,), 23)
    y, k = _profile(lambda: X.conv2d_forward(x, w, b, SAME, 1))
    assert k == {"conv2d_direct_small_kernel": 1}, k
    for i in range(0, B, 1000):
        assert torch.equal(y[i:i + 1000], X.conv2d_forward(x[i:i + 1000], w, b, SAME, 1)), f"images {i}..{i + 999} differ"
    wn, bn = w.cpu().numpy(), b.cpu().numpy()
    _oracle_images(y, (0, 35000, 65535, B - 1), lambda i: E.conv2d_forward(x[i:i + 1].cpu().numpy(), wn, bn, SAME, 1))
    del x, y
    _free()


def test_large_skinny_backward_data_past_its_grid_limit():
    """A 512-wide layer in front of a 10-row output at batch 1 048 576 (65 536 chunks of 16 samples): the layer's delta
    against torch f64 on the device."""
    import torch
    import mercer_research_b200 as m
    from mercer_research_b200 import _lib
    B, L = 1 << 20, 8
    model = m.RCN(10, [], [512])
    try:
        model.load_weights_and_bias(L)
        rng = np.random.default_rng(31)
        model.set_params(rng.standard_normal(model.n_params) * 0.1)
        feats = _dev_randn((B, L), 32)
        labels = torch.randint(0, 10, (B,), device="cuda", generator=torch.Generator(device="cuda").manual_seed(33))
        _, k = _profile(lambda: model.accumulate_gradients(feats, labels=labels))
        assert k.get("skinny_backward_data_kernel") == cdiv(cdiv(B, 16), MAX_GRID_YZ) == 2, k
        got = torch.empty((B, 512), dtype=torch.float64, device="cuda")
        _lib.check(_lib.load().rcn_cuda_get_deltas(model._h, 0, got.data_ptr()))
        model.synchronize()
        W0, b0, W1, b1 = (torch.as_tensor(a, device="cuda") for a in
                          (model.get_weights(0), model.get_bias(0), model.get_weights(1), model.get_bias(1)))
        step = 1 << 16
        want = torch.empty_like(got)
        for i in range(0, B, step):
            a0 = torch.sigmoid(feats[i:i + step] @ W0.T + b0)
            a1 = torch.sigmoid(a0 @ W1.T + b1)
            d1 = (a1 - torch.nn.functional.one_hot(labels[i:i + step], 10).double()) * a1 * (1 - a1)
            want[i:i + step] = (d1 @ W1) * a0 * (1 - a0)
        _close_dev(got, want, what="skinny backward-data delta vs torch f64", step=step)
    finally:
        model.close()
        _free()


def test_simt_gemm_past_its_grid_limit(tmp_path):
    """The SIMT cross-check GEMM (RCN_CUDA_GEMM=simt) at batch 600 000 (75 000 rows of 8 columns): a 4-33-2 sigmoid network
    (33 rows: too wide for the fused small-network kernels) - its gradient sums against numpy f64, componentwise, and its
    output activations elementwise."""
    B, L, Hd = 600000, 4, 33
    rng = np.random.default_rng(41)
    feats = rng.standard_normal((B, L))
    labels = rng.integers(0, 2, B).astype(np.int64)
    params = rng.standard_normal(Hd * L + Hd + 2 * Hd + 2) * 0.5
    np.save(tmp_path / "feats.npy", feats)
    np.save(tmp_path / "labels.npy", labels)
    np.save(tmp_path / "params.npy", params)
    code = ("import sys, json, numpy as np; sys.path.insert(0, %r); import mercer_research_b200 as m; from mercer_research_b200 import _lib;"
            "d = sys.argv[1]; f = np.load(d + '/feats.npy'); lab = np.load(d + '/labels.npy');"
            "net = m.RCN(2, [], [%d]); net.load_weights_and_bias(f.shape[1]); net.set_params(np.load(d + '/params.npy'));"
            "_lib.profile_enable(True); net.accumulate_gradients(f, labels=lab); k = _lib.profile_report();"
            "np.save(d + '/grads.npy', net.get_gradients()); np.save(d + '/out.npy', net.activations(1));"
            "print(json.dumps({n: v['launches'] for n, v in k.items()}))") % (ROOT, Hd)
    r = subprocess.run([sys.executable, "-c", code, str(tmp_path)], env=dict(os.environ, RCN_CUDA_GEMM="simt"),
                       capture_output=True, text=True, check=True)
    k = json.loads(r.stdout.strip().splitlines()[-1])
    assert "dense_forward_gemm" in k and not any(n.startswith(("skinny", "smallnet")) or "tcgen05" in n for n in k), k

    # numpy reference; params = [W0 (Hd x L, column-major) | b0 | W1 (2 x Hd, column-major) | b1]
    o = 0
    W0 = params[o:o + Hd * L].reshape(L, Hd).T; o += Hd * L
    b0 = params[o:o + Hd]; o += Hd
    W1 = params[o:o + 2 * Hd].reshape(Hd, 2).T; o += 2 * Hd
    b1 = params[o:o + 2]
    sig = lambda z: 1 / (1 + np.exp(-z))
    a0 = sig(feats @ W0.T + b0)
    a1 = sig(a0 @ W1.T + b1)
    d1 = (a1 - np.eye(2)[labels]) * a1 * (1 - a1)
    d0 = (d1 @ W1) * a0 * (1 - a0)
    want = np.concatenate([(d0.T @ feats).T.ravel(), d0.sum(0), (d1.T @ a0).T.ravel(), d1.sum(0)])
    bound = np.concatenate([(np.abs(d0).T @ np.abs(feats)).T.ravel(), np.abs(d0).sum(0), (np.abs(d1).T @ a0).T.ravel(),
                            np.abs(d1).sum(0)])
    got = np.load(tmp_path / "grads.npy")
    assert np.all(np.abs(got - want) <= 1e-9 * bound), np.max(np.abs(got - want) / bound)
    assert_close(np.load(tmp_path / "out.npy"), a1, what="output activations")


# -- E. the ConvNet handle at dataset sizes -------------------------------------------------------------------------------
def _cifar_net(m):
    P = m.Padding
    return m.ConvNet((32, 32, 3), [m.Conv(16, 3, 3, P.Same), m.Conv(32, 3, 3, P.Same), m.Pool(m.Pooling.Max, P.Same)], [32], 10)


def _layer_out_dev(net, layer):
    import torch
    from mercer_research_b200 import _lib
    out = torch.empty((net._B_out,) + tuple(net.layer_shape(layer)), dtype=torch.float64, device="cuda")
    _lib.check(_lib.load().rcn_cuda_cnn_get_layer_output(net._h, layer, out.data_ptr()))
    net.synchronize()
    return out


def _one_call_equals_chunks(net, images, labels, chunk, conv_layers, kernels):
    import torch
    n = images.shape[0]
    lab_all, k = _profile(lambda: net.classify_images(images))
    for name, launches in kernels.items():
        assert k.get(name) == launches, (name, k)
    assert not any("tcgen05" in name for name in k), k
    outs = [_layer_out_dev(net, i) for i in conv_layers]
    acc_all, cost_all = net.evaluate_images(images, labels)
    acc, cost = 0, 0.0
    for i in range(0, n, chunk):
        lab = net.classify_images(images[i:i + chunk])
        assert torch.equal(lab, lab_all[i:i + chunk]), f"labels of images {i}.. differ"
        for j, o in zip(conv_layers, outs):
            assert torch.equal(_layer_out_dev(net, j), o[i:i + chunk]), f"layer {j} output of images {i}.. differs"
        a, c = net.evaluate_images(images[i:i + chunk], labels[i:i + chunk])
        acc += a
        cost += c
    assert acc_all == acc
    assert abs(cost_all - cost) <= 1e-12 * abs(cost_all), (cost_all, cost)


def test_large_convnet_f64_10000_images_one_call_equals_chunks():
    import torch
    import mercer_research_b200 as m
    net = _cifar_net(m)
    try:
        net.init_params(np.random.default_rng(51))
        images = _dev_randn((10000, 32, 32, 3), 52)
        labels = torch.randint(0, 10, (10000,), device="cuda", generator=torch.Generator(device="cuda").manual_seed(53))
        p1 = plan(10000, 32, 32, 16, 32, 3, 3, SAME)
        print("conv0", plan(10000, 32, 32, 3, 16, 3, 3, SAME)["fwd"], "conv1", p1)
        _one_call_equals_chunks(net, images, labels, 1000, [0, 1],
                                {"conv2d_direct_small_kernel": 1, "conv2d_forward_igemm": p1["fwd_launches"]})
    finally:
        net.close()
        _free()


def test_large_convnet_u8_70000_images_one_call_equals_chunks():
    import torch
    import mercer_research_b200 as m
    P = m.Padding
    net = m.ConvNet((28, 28, 1), [m.Conv(8, 3, 3, P.Same), m.Pool(m.Pooling.Max, P.Same)], [30], 10)
    try:
        net.init_params(np.random.default_rng(61))
        g = torch.Generator(device="cuda").manual_seed(62)
        images = torch.randint(0, 256, (70000, 28, 28), dtype=torch.uint8, device="cuda", generator=g)
        labels = torch.randint(0, 10, (70000,), device="cuda", generator=g)
        _one_call_equals_chunks(net, images, labels, 7000, [0], {"conv2d_direct_small_u8_kernel": 1})
    finally:
        net.close()
        _free()


def test_large_convnet_training_step_8192_images():
    """One accumulate at B = 8 192 made of 1 024 copies of 8 images against the 8-image batch: every copy's layer outputs
    bit-identical, gradient sums 1 024 x the 8-image sums (componentwise 1e-9 against 1 024 x the per-image |gradient|),
    hits 1 024 x."""
    import torch
    import mercer_research_b200 as m
    net = _cifar_net(m)
    try:
        net.init_params(np.random.default_rng(71))
        x8 = _dev_randn((8, 32, 32, 3), 72)
        lab8 = torch.arange(8, device="cuda", dtype=torch.int64) % 10
        net.accumulate_gradients_images(x8, lab8)
        g8 = net.get_gradients()
        _, hits8 = net.last_batch_stats()
        outs8 = [_layer_out_dev(net, i) for i in range(3)]
        abs8 = np.zeros_like(g8)
        for i in range(8):
            net.accumulate_gradients_images(x8[i:i + 1], lab8[i:i + 1])
            abs8 += np.abs(net.get_gradients())

        big, big_lab = x8.repeat(1024, 1, 1, 1), lab8.repeat(1024)
        p0, p1 = plan(8192, 32, 32, 3, 16, 3, 3, SAME), plan(8192, 32, 32, 16, 32, 3, 3, SAME)
        print("conv0", p0, "conv1", p1)
        _, k = _profile(lambda: net.accumulate_gradients_images(big, big_lab))
        assert k.get("conv2d_direct_small_kernel") == 1 and k.get("conv2d_forward_igemm") == p1["fwd_launches"] == 2, k
        assert k.get("conv2d_backward_data_igemm") == p1["bwd_launches"] == 2, k
        assert k.get("conv2d_backward_weight_igemm") == 2 and "reduce_splits_kernel" in k, k
        assert not any("tcgen05" in name for name in k), k
        _, hits = net.last_batch_stats()
        assert hits == 1024 * hits8
        for i in range(3):
            o = _layer_out_dev(net, i)
            assert torch.equal(o.view(1024, 8, -1), outs8[i].view(1, 8, -1).expand(1024, -1, -1)), f"layer {i} output"
        g = net.get_gradients()
        bad = np.abs(g - 1024 * g8) > 1e-9 * 1024 * abs8
        assert not bad.any(), f"{int(bad.sum())} gradient sums off the componentwise bar"
    finally:
        net.close()
        _free()
