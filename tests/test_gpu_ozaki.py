"""The tcgen05 integer-slice GEMMs (csrc/ozaki.cuh, ozaki.cu) element by element, on every operand path: the four dense
layouts of ext.gemm_f64, the TMA-gathered and the per-row-gathered convolution input (forward, backward-data) and the
split-K backward-weight GEMM.

Each GPU result is held against two references:
 (a) an exact numpy emulation of the scheme (below): the slicing into balanced base-256 digits, the scale source of each
     operand path, the diagonal sums, the Horner combine and the split-K plan.  The GPU must match it to a few f64 ulps of
     the unscaled accumulator.  A dropped digit plane, a wrong +128 carry or a lost partial k-block costs ~1e-10 relative,
     under any f64 bar, but not under this one.
 (b) plain f64: |gpu - ref| <= 1e-9 * terms componentwise, terms = (|A|.|B|)[m, n] (for a convolution: the same
     convolution of |x| with |w|).  Each operand's slicing error is relative to the maximum of its scale unit (a row, an
     image, a channel), so the bar that does not depend on how magnitudes vary inside a unit is |gpu - ref| <= 1e-9 *
     unit, unit = amax(A's unit) . sum|B| + sum|A| . amax(B's unit) (DESIGN.md section 2).  Every case is held to it,
     and to the componentwise bar wherever the magnitudes inside each unit are alike.

The emulation's own CPU tests run without a GPU.  RCN_CUDA_GEMM is read once per process, so the convolution cases run
in one subprocess per engine (this file, run as a script) and are checked here.
"""
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

S, D = 5, 4                       # digit planes per operand, highest diagonal kept
BM, BN, BK = 128, 96, 64          # tile of ozaki_gemm_kernel
MAX_K = 16384                     # exact int32 accumulation bound of one split
NUM_SMS = 148                     # kNumSMs (split planning)
BAR = 1e-9                        # componentwise bar (b)
ULPS = 2.0 ** -48                 # bar (a): a few f64 ulps of the unscaled accumulator


# ---- the scheme, emulated -------------------------------------------------------------------------------------------

def amax_rows(x, axis=-1):
    """Row maxima as the slicing kernels fold them: any NaN / Inf makes the maximum NaN."""
    x = np.asarray(x, dtype=np.float64)
    fin = np.isfinite(x)
    m = np.max(np.abs(np.where(fin, x, 0.0)), axis=axis, initial=0.0)
    return np.where(fin.all(axis=axis), m, np.nan)


def row_scale(amax):
    """(inv, scale) of ozaki.cu row_scale: amax = f * 2^e, f in [0.5, 1) -> inv = 2^(6-e), scale = 2^(e-6).  A non-finite
    amax or one >= 1e290 gives all-zero planes (inv 0) and scale NaN; amax <= 1e-290 gives all-zero planes and scale 0."""
    amax = np.asarray(amax, dtype=np.float64)
    inv = np.zeros(amax.shape)
    scale = np.full(amax.shape, np.nan)
    ok = amax < 1e290
    tiny = ok & ~(amax > 1e-290)
    good = ok & ~tiny
    e = np.frexp(amax[good])[1]
    inv[good] = np.ldexp(1.0, 6 - e)
    scale[good] = np.ldexp(1.0, e - 6)
    scale[tiny] = 0.0
    return inv, scale


def slice6(x, inv):
    """ozaki.cu slice6: t = x * inv, q_0 = rint(t) (ties to even), then (t - f) * 256 four times; a digit equal to +128
    becomes -128 and carries 1 into the next more significant digit.  Returns float64 digits [S, *x.shape]."""
    x = np.asarray(x, dtype=np.float64)
    inv = np.broadcast_to(inv, x.shape)
    with np.errstate(invalid="ignore"):
        t = np.where(inv == 0.0, 0.0, x * inv)   # inv 0: the kernel's digits are all 0 (NaN converts to 0 as well)
    d = np.empty((S,) + x.shape)
    for j in range(S):
        f = np.rint(t)
        d[j] = f
        t = (t - f) * 256.0
    for j in range(S - 1, 0, -1):
        c = d[j] == 128.0
        d[j] -= 256.0 * c
        d[j - 1] += c
    return d


def plan_splits(M, N, K):
    """ozaki.cuh ozaki_plan_splits, as launch_gemm_ozaki then rounds it: (splits, k per split)."""
    n_kb = -(-K // BK)
    tiles = -(-M // BM) * -(-N // BN)
    splits = -(-K // MAX_K)
    if tiles < NUM_SMS:
        splits = max(splits, min(-(-2 * NUM_SMS // tiles), n_kb // 8))
    splits = max(splits, 1)
    kbps = -(-n_kb // splits)
    return -(-n_kb // kbps), kbps * BK


def combine(pa, pb, sa, sb):
    """One tile pass: diagonals sum_{i+j=d} planes_i . planes_j^T (float64 matmuls: every sum is an integer < 2^53, so
    BLAS computes it exactly), Horner with weight 2^-8 (== the kernel's fma), times sa * sb.  Returns (value, bound (a))."""
    acc = [sum(pa[i] @ pb[d - i].T for i in range(d + 1)) for d in range(D + 1)]
    v = acc[D]
    for d in range(D - 1, -1, -1):
        v = v * 2.0 ** -8 + acc[d]
    mag = sum(np.abs(acc[d]) * 2.0 ** (-8 * d) for d in range(D + 1))
    with np.errstate(invalid="ignore", over="ignore", under="ignore"):
        return v * sa[:, None] * sb[None, :], ULPS * mag * np.abs(sa)[:, None] * np.abs(sb)[None, :]


def emulate(get_a, amax_a, get_b, amax_b, K, split_k=None):
    """C = A . B^T through the scheme, plus the f64 reference, its terms |A|.|B|^T, which outputs f64 makes non-finite
    and the unit terms amax_a . sum|B| + sum|A| . amax_b.
    get_a(k0, k1) / get_b(k0, k1) return the (rows, k1 - k0) slab of each operand; amax_* are the per-row maxima of the
    path's scale source.  split_k: k per split (partials summed in split order); None = one pass."""
    inv_a, sa = row_scale(amax_a)
    inv_b, sb = row_scale(amax_b)
    step = split_k or max(K, 1)
    out = bnd = ref = terms = bad = unit = None
    for k0 in range(0, max(K, 1), step):
        k1 = min(K, k0 + step)
        a, b = get_a(k0, k1), get_b(k0, k1)
        v, e = combine(slice6(a, inv_a[:, None]), slice6(b, inv_b[:, None]), sa, sb)
        fa, fb = np.isfinite(a), np.isfinite(b)
        a0, b0 = np.where(fa, a, 0.0), np.where(fb, b, 0.0)
        r, t = a0 @ b0.T, np.abs(a0) @ np.abs(b0).T
        nf = (~fa.all(1))[:, None] | (~fb.all(1))[None, :]
        with np.errstate(over="ignore"):   # only where a >= 1e290 element has made the output NaN anyway
            u = amax_a[:, None] * np.abs(b0).sum(1)[None, :] + np.abs(a0).sum(1)[:, None] * amax_b[None, :]
        if out is None:
            out, bnd, ref, terms, bad, unit = v, e, r, t, nf, u
        else:
            out, bnd, ref, terms, bad, unit = out + v, bnd + e, ref + r, terms + t, bad | nf, unit + u
    return out, bnd, ref, terms, bad, unit


def emulate_dense(a, b, k_per_split=None):
    """A (M, K) @ B (K, N): every dense operand path scales each row by its own maximum."""
    bt = np.ascontiguousarray(b.T)
    return emulate(lambda k0, k1: a[:, k0:k1], amax_rows(a), lambda k0, k1: bt[:, k0:k1], amax_rows(bt), a.shape[1],
                   k_per_split)


# ---- CPU tests of the emulation ---------------------------------------------------------------------------------------

def test_slices_digit_ranges_and_reconstruction():
    rng = np.random.default_rng(1)
    x = rng.standard_normal((64, 4096)) * 10.0 ** rng.uniform(-20, 20, size=(64, 1))
    x[:, :64] = rng.integers(-1000, 1001, size=(64, 64)) / 2.0 ** rng.integers(0, 12, size=(64, 1))   # many exact ties
    x[3] *= 1e-250                      # amax ~1e-250: still above the 1e-290 floor, so sliced
    amax = amax_rows(x)
    inv, sc = row_scale(amax)
    d = slice6(x, inv[:, None])
    assert np.abs(d[0]).max() <= 65 and d[1:].min() >= -128 and d[1:].max() <= 127
    assert np.array_equal(d, np.rint(d))
    recon = sum(d[j] * 2.0 ** (-8 * j) for j in range(S)) * sc[:, None]
    # the dropped remainder is at most half a unit of the last digit: 2^-33 * scale <= 2^-38 * amax
    assert (np.abs(recon - x) <= 2.0 ** -33 * sc[:, None]).all()
    assert (2.0 ** -33 * sc <= 2.0 ** -38 * amax).all()


def test_slices_carries_signed_zero_powers_of_two_and_amax():
    amax = 40.0                          # frexp: 0.625 * 2^6 -> inv = 1, every t below is x itself
    inv, sc = row_scale(np.array([amax]))
    assert inv[0] == 1.0 and sc[0] == 1.0
    cases = {
        2.5: (3, -128, 0, 0, 0),         # rint(2.5) = 2 (even), r = +0.5 -> digit 128 -> -128 with a carry
        3.5: (4, -128, 0, 0, 0),         # rint(3.5) = 4, r = -0.5 -> -128, no carry
        -1.5: (-1, -128, 0, 0, 0),       # rint(-1.5) = -2, r = +0.5 -> carry
        -2.5: (-2, -128, 0, 0, 0),
        2 + 2.0 ** -9: (2, 1, -128, 0, 0),               # tie one digit down: rint(0.5) = 0, then 128 -> carry
        2 + 2.0 ** -33: (2, 0, 0, 0, 0),                 # half a unit of the last digit: ties to even 0, dropped
        2 + 3 * 2.0 ** -33: (2, 0, 0, 0, 2),             # 1.5 units of the last digit: ties to even 2
        63.5: (64, -128, 0, 0, 0),
        0.0: (0, 0, 0, 0, 0), -0.0: (0, 0, 0, 0, 0),
        32.0: (32, 0, 0, 0, 0), 2.0 ** -32: (0, 0, 0, 0, 1), -(2.0 ** -20): (0, 0, 0, -16, 0),
        amax: (40, 0, 0, 0, 0), -amax: (-40, 0, 0, 0, 0),
    }
    x = np.array(list(cases))
    d = slice6(x, 1.0)
    for i, (v, want) in enumerate(cases.items()):
        assert tuple(d[:, i].astype(int)) == want, (v, d[:, i])
        assert abs(sum(d[j, i] * 2.0 ** (-8 * j) for j in range(S)) - v) <= 2.0 ** -33
    # powers of two as the row maximum: amax = 2^e exactly gives f = 0.5, so t = 32
    for e in (-900, -7, 0, 6, 7, 900):
        inv, sc = row_scale(np.array([2.0 ** e]))
        assert sc[0] == 2.0 ** (e + 1 - 6) and tuple(slice6(np.array([2.0 ** e, -(2.0 ** e)]), inv[0])[0]) == (32, -32)
    # rows the digits cannot represent
    inv, sc = row_scale(np.array([np.nan, np.inf, 1e290, 1e300, 1e-290, 0.0, 1.1e-290, 9.9e289]))
    assert np.isnan(sc[:4]).all() and (inv[:4] == 0).all() and (sc[4:6] == 0).all() and (inv[4:6] == 0).all()
    assert sc[6] > 0 and sc[7] > 0
    assert np.isnan(amax_rows(np.array([[1.0, np.nan, 2.0], [1.0, -np.inf, 0.0]]))).all()
    assert (slice6(np.array([np.nan, 1e300, 5.0]), 0.0) == 0).all()


def test_emulated_gemm_is_within_1e10_componentwise_of_f64():
    rng = np.random.default_rng(2)
    a = rng.standard_normal((97, 1000)) * 10.0 ** rng.uniform(-50, 50, size=(97, 1))
    b = rng.standard_normal((1000, 129)) * 10.0 ** rng.uniform(-50, 50, size=(1, 129))
    a[5, :500] = -a[5, 500:]
    b[:500, 7] = b[500:, 7]              # cancels to ~0 against row 5
    for k_per_split in (None, 192):
        out, bnd, ref, terms, bad, _ = emulate_dense(a, b, k_per_split)
        assert not bad.any()
        assert (np.abs(out - a @ b) <= 1e-10 * terms).all()
        assert (bnd < 1e-13 * terms).all()


def test_split_plan_mirrors_the_library():
    assert plan_splits(64, 576, 512) == (1, 512)
    assert plan_splits(64, 576, 65536) == (49, 21 * 64)
    assert plan_splits(4096, 4096, 16384) == (1, 16384)
    assert plan_splits(4096, 4096, 16448) == (2, 8256)


# ---- dense GEMM through ext.gemm_f64(impl=1) --------------------------------------------------------------------------

def dense_case(M, N, K, seed):
    """Rows: scales spread 1e+-100, one element 1e8 above the rest (only up to K = 4096: a row whose terms one element
    dominates has a componentwise error growing like sqrt(K) * 2^-39, which nears 1e-9 at K = 16384), 1e-200 values, zero
    rows, rows that cancel against the antisymmetric columns.  Columns: scales spread 1e+-100, zero columns."""
    rng = np.random.default_rng(seed)
    a = rng.standard_normal((M, K))
    kind = np.arange(M) % 6
    a *= np.where(kind == 0, 10.0 ** rng.uniform(-100, 100, size=M), 1.0)[:, None]
    if K <= 4096:
        for m in np.flatnonzero(kind == 1):
            a[m, rng.integers(K)] *= 1e8
    a[kind == 2] *= 1e-200
    a[kind == 3] = 0.0
    half = K // 2
    a[kind == 4, half:2 * half] = a[kind == 4, :half]
    b = rng.choice([-1.0, 1.0], size=(K, N)) * rng.uniform(0.5, 1.5, size=(K, N))
    b *= 10.0 ** rng.uniform(-100, 100, size=N)
    ckind = np.arange(N) % 4
    b[half:2 * half, ckind == 1] = -b[:half, ckind == 1]
    b[2 * half:, ckind == 1] = 0.0
    b[:, ckind == 3] = 0.0
    return a, b


def check(got, emu, ebound, ref, terms, ref_bad, unit, what, componentwise=True):
    """(a) against the emulation, (b) against f64 (see the module docstring), non-finite sets of both.  componentwise
    False: only the unit bar of (b)."""
    got = np.asarray(got, dtype=np.float64).reshape(emu.shape)
    emu_bad, got_bad = ~np.isfinite(emu), ~np.isfinite(got)
    assert np.array_equal(got_bad, emu_bad), (what, "non-finite set differs from the emulation", int(got_bad.sum()),
                                              int(emu_bad.sum()))
    assert got_bad[ref_bad].all(), (what, "finite where f64 is not")
    ok = ~got_bad
    err = np.abs(got - emu)[ok]
    bad = err > ebound[ok]
    assert not bad.any(), (what, "(a) emulation", int(bad.sum()), float(np.max(err / np.maximum(ebound[ok], 1e-300))))
    err = np.abs(got - ref)[ok]
    bad = err > BAR * unit[ok]
    assert not bad.any(), (what, "(b) f64 relative to the scale units", int(bad.sum()),
                           float(np.max(err / np.maximum(unit[ok], 1e-300))))
    if componentwise:
        bad = err > BAR * terms[ok]
        assert not bad.any(), (what, "(b) f64 componentwise", int(bad.sum()),
                               float(np.max(err / np.maximum(terms[ok], 1e-300))))


DENSE_SHAPES = [(1, 1, 1), (127, 97, 63), (129, 129, 65), (97, 127, 511), (129, 97, 513), (129, 97, 16384),
                (1, 1, 16384)]
LAYOUTS = [(True, True), (False, True), (False, False), (True, False)]


@pytest.fixture(scope="module")
def X(built_library):
    from mercer_research_b200 import ext
    return ext


@pytest.mark.gpu
@pytest.mark.parametrize("M,N,K", DENSE_SHAPES)
@pytest.mark.parametrize("layout", LAYOUTS, ids=["kk", "rk", "rr", "kr"])
def test_gemm_matches_emulation_and_f64_componentwise(X, M, N, K, layout):
    from mercer_research_b200 import _lib
    a, b = dense_case(M, N, K, seed=M * 31 + N * 7 + K)
    _lib.profile_enable(True)
    got = X.gemm_f64(a, b, impl=1, a_kcontig=layout[0], b_kcontig=layout[1])
    names = set(_lib.profile_report())
    _lib.profile_enable(False)
    assert "ext_gemm_f64(tcgen05 int8 slices)" in names, names
    for kc in layout:   # each operand's slicer
        assert ("ozaki_slice_kmajor_kernel" if kc else "ozaki_slice_rmajor_kernel") in names, names
    check(got, *emulate_dense(a, b), f"gemm {M}x{N}x{K} {layout}")


@pytest.mark.gpu
def test_gemm_int32_exactness_edge(X):
    """K = 16384 with the digits (63, 127, 127, 127, 127) in every element and equal signs along k: diagonal 4 accumulates
    16384 * 64389 = 1.055e9 of the 2^31 an int32 holds (the bound 5 * 16384 * 128^2 that OZ_MAX_K rests on is 1.34e9),
    and the result is exactly the emulation's.  One more k is refused as an invalid argument."""
    from mercer_research_b200 import _lib
    v = 63 + 127 * sum(2.0 ** (-8 * j) for j in range(1, S))
    assert tuple(slice6(np.array([v]), row_scale(np.array([v]))[0])[:, 0]) == (63, 127, 127, 127, 127)
    M, N, K = 130, 97, 16384
    rng = np.random.default_rng(9)
    a = np.outer(rng.choice([-1.0, 1.0], size=M), np.full(K, v))
    b = np.outer(np.full(K, v), rng.choice([-1.0, 1.0], size=N))
    emu, *_ = emulate_dense(a, b)
    for layout in LAYOUTS:
        got = X.gemm_f64(a, b, impl=1, a_kcontig=layout[0], b_kcontig=layout[1])
        assert np.array_equal(got, emu), layout
    a1 = np.ones((8, K + 1))
    with pytest.raises(_lib.RcnCudaError) as e:
        X.gemm_f64(a1, a1.T, impl=1)
    assert e.value.status == 1 and "exceeds 16384" in e.value.message


# ---- convolutions -----------------------------------------------------------------------------------------------------

SPREAD = [1.0, 1e-2, 1e-4, 1e-8]     # per-image scales of x and dz


def conv_case(name, B, H, W, Ci, Co, kh, kw, pad, ops=("fwd", "bwd", "wgt"), spread=True, bad=None, offset=False,
              intra=None):
    """spread: images scaled by SPREAD; intra: the top half of every image of x and dz scaled by this factor."""
    return dict(name=name, B=B, H=H, W=W, Ci=Ci, Co=Co, kh=kh, kw=kw, pad=pad, ops=list(ops), spread=spread, bad=bad,
                offset=offset, intra=intra)


def tma_ok(Ho, Wo, C, n_k):
    """ozaki.cuh ozaki_conv_tma_ok for an aligned tensor."""
    tiles = (Wo <= BM and BM % Wo == 0 and Ho % (BM // Wo) == 0) or Wo % BM == 0
    return C % BK == 0 and tiles and n_k <= MAX_K


def geometry(c):
    same = c["pad"] == 1
    Ho, Wo = (c["H"], c["W"]) if same else (c["H"] - c["kh"] + 1, c["W"] - c["kw"] + 1)
    ph, pw = (c["kh"] // 2, c["kw"] // 2) if same else (0, 0)
    return Ho, Wo, ph, pw


def conv_inputs(c):
    rng = np.random.default_rng(zlib.crc32(c["name"].encode()))
    B, H, W, Ci, Co, kh, kw = (c[k] for k in ("B", "H", "W", "Ci", "Co", "kh", "kw"))
    Ho, Wo, _, _ = geometry(c)
    x = rng.standard_normal((B, H, W, Ci))
    dz = rng.standard_normal((B, Ho, Wo, Co))
    if c["spread"]:
        s = np.array([SPREAD[b % len(SPREAD)] for b in range(B)])[:, None, None, None]
        x, dz = x * s, dz * s
    if c["intra"] is not None:
        x[:, :H // 2] *= c["intra"]
        dz[:, :Ho // 2] *= c["intra"]
    w = rng.standard_normal((Co, kh, kw, Ci)) / np.sqrt(kh * kw * Ci)
    if c["bad"] is not None:
        x[BAD_X] = c["bad"]
        dz[BAD_DZ] = c["bad"]
    return x, w, dz


def im2col(t, Ho, Wo, kh, kw, ph, pw, p0, p1):
    """Rows = grid pixels p0..p1-1 of [B][Ho][Wo]; k = (ky, kx, c), c fastest; tap (ky, kx) of pixel (oy, ox) reads
    t[b, oy + ky - ph, ox + kx - pw] (zero outside)."""
    B, Hi, Wi, C = t.shape
    b0, b1 = p0 // (Ho * Wo), -(-p1 // (Ho * Wo))
    tp = np.zeros((b1 - b0, Ho + kh - 1, Wo + kw - 1, C))      # row r of tp is row r - ph of t
    ys, xs = slice(ph, min(Ho + kh - 1, Hi + ph)), slice(pw, min(Wo + kw - 1, Wi + pw))
    tp[:, ys, xs] = t[b0:b1, :ys.stop - ph, :xs.stop - pw]
    cols = np.empty((b1 - b0, Ho, Wo, kh, kw, C))
    for ky in range(kh):
        for kx in range(kw):
            cols[:, :, :, ky, kx] = tp[:, ky:ky + Ho, kx:kx + Wo]
    cols = cols.reshape((b1 - b0) * Ho * Wo, kh * kw * C)
    return cols[p0 - b0 * Ho * Wo:p1 - b0 * Ho * Wo]


def conv_expect(c, op, x, w, dz, tma):
    """Emulation and f64 reference of one convolution op as the GEMM the library runs (conv.cu)."""
    B, H, W, Ci, Co, kh, kw = (c[k] for k in ("B", "H", "W", "Ci", "Co", "kh", "kw"))
    Ho, Wo, ph, pw = geometry(c)
    if op in ("fwd", "bwd"):
        if op == "fwd":   # Y(pix, co) = im2col(x)(pix, k) . w(co, k)
            t, grid, pads, wk = x, (Ho, Wo), (ph, pw), w.reshape(Co, -1)
        else:             # dX(pix, ci) = im2col(dz)(pix, k') . w'(ci, k'), complementary padding, flipped weights
            t, grid, pads = dz, (H, W), (kh - 1 - ph, kw - 1 - pw)
            wk = np.ascontiguousarray(w[:, ::-1, ::-1, :].transpose(3, 1, 2, 0)).reshape(Ci, -1)
        rows = im2col(t, *grid, kh, kw, *pads, 0, B * grid[0] * grid[1])
        # scale source of the pixel rows: the whole image (TMA path) or the pixel's own receptive field
        amax_a = np.repeat(amax_rows(t.reshape(B, -1)), grid[0] * grid[1]) if tma else amax_rows(rows)
        return emulate(lambda k0, k1: rows[:, k0:k1], amax_a, lambda k0, k1: wk[:, k0:k1], amax_rows(wk), rows.shape[1])
    # dW(co, k) = sum_pix dz(pix, co) . im2col(x)(pix, k), split over the pixels
    n_pix = B * Ho * Wo
    dzf = dz.reshape(n_pix, Co)
    _, kps = plan_splits(Co, kh * kw * Ci, n_pix)
    amax_b = np.tile(amax_rows(x.reshape(-1, Ci).T), kh * kw)    # one maximum per channel over every pixel of x
    return emulate(lambda k0, k1: dzf[k0:k1].T, amax_rows(dzf.T),
                   lambda k0, k1: im2col(x, Ho, Wo, kh, kw, ph, pw, k0, k1).T, amax_b, n_pix, kps)


def test_conv_reference_matches_torch():
    """The im2col GEMMs that conv_expect emulates are the convolutions themselves (torch f64 on the CPU)."""
    import torch
    F = torch.nn.functional
    for c in (conv_case("ref_same", 2, 5, 7, 3, 4, 3, 3, 1), conv_case("ref_none", 2, 6, 9, 2, 3, 3, 5, 0),
              conv_case("ref_1x3", 1, 4, 8, 3, 2, 1, 3, 1), conv_case("ref_5x5", 3, 6, 6, 2, 3, 5, 5, 1)):
        x, w, dz = conv_inputs(c)
        ph, pw = geometry(c)[2:]
        xt, wt, dzt = (torch.from_numpy(np.ascontiguousarray(v.transpose(0, 3, 1, 2))) for v in (x, w, dz))
        want = {"fwd": F.conv2d(xt, wt, padding=(ph, pw)).permute(0, 2, 3, 1),
                "bwd": torch.nn.grad.conv2d_input(xt.shape, wt, dzt, padding=(ph, pw)).permute(0, 2, 3, 1),
                "wgt": torch.nn.grad.conv2d_weight(xt, wt.shape, dzt, padding=(ph, pw)).permute(0, 2, 3, 1)}
        for op, ref_t in want.items():
            for tma in (False, True):
                out, _, ref, terms, _, _ = conv_expect(c, op, x, w, dz, tma)
                r = ref_t.numpy().reshape(ref.shape)
                assert np.allclose(ref, r, rtol=0, atol=1e-13 * terms.max()), (c["name"], op)
                assert np.abs(out - r).max() <= 1e-10 * terms.max(), (c["name"], op, tma)   # few channels: norm-wise


CONV_CASES = [
    # TMA-gathered input (C % 64 == 0), every tile shape: Wo in {16, 32, 64, 128, 256}; images 1, 1e-2, 1e-4, 1e-8 apart
    conv_case("tma_wo16_3x3", 4, 8, 16, 64, 64, 3, 3, 1),
    conv_case("tma_wo32_3x3_c128", 4, 4, 32, 128, 64, 3, 3, 1),
    conv_case("tma_wo64_1x3", 4, 4, 64, 64, 128, 1, 3, 1),
    conv_case("tma_wo128_3x3", 4, 3, 128, 64, 64, 3, 3, 1),
    conv_case("tma_wo256_3x3", 4, 3, 256, 64, 64, 3, 3, 1),
    conv_case("tma_wo16_5x5", 4, 8, 16, 64, 64, 5, 5, 1),
    conv_case("tma_fwd_none_3x3", 4, 10, 18, 64, 64, 3, 3, 0),     # fwd TMA (8 x 16); bwd-data per-row (10 x 18 grid)
    conv_case("tma_bwd_none_3x3", 4, 4, 32, 64, 64, 3, 3, 0),      # bwd-data TMA from negative coordinates; fwd per-row
    conv_case("tma_fwd_none_5x5", 4, 12, 20, 64, 64, 5, 5, 0),
    # per-row gather (C not a multiple of 64)
    conv_case("row_3x3", 4, 8, 16, 40, 48, 3, 3, 1),
    conv_case("row_none_3x3", 4, 10, 18, 24, 100, 3, 3, 0),
    conv_case("row_1x3", 4, 4, 32, 20, 36, 1, 3, 1),
    conv_case("row_5x5", 4, 8, 16, 24, 40, 5, 5, 1),
    # backward-weight over 65536 pixels: 49 splits
    conv_case("wgt_splits", 16, 64, 64, 64, 64, 3, 3, 1, ops=("wgt",)),
    # pixels 1e4 apart inside every image: on the TMA path only the unit bar holds, the per-row gather keeps the
    # componentwise one
    conv_case("tma_intra_image", 4, 8, 16, 64, 64, 3, 3, 1, intra=1e-4),
    conv_case("row_intra_image", 4, 8, 16, 40, 48, 3, 3, 1, intra=1e-4),
    # a device view 8 bytes off 16-byte alignment
    conv_case("offset", 4, 8, 16, 64, 64, 3, 3, 1, offset=True),
] + [conv_case(f"{path}_{tag}", 4, 8, 16, C, C, 3, 3, 1, spread=False, bad=v)
     for path, C in (("tma", 64), ("row", 40)) for tag, v in (("nan", np.nan), ("inf", np.inf), ("big", 1e300))]
BAD_X, BAD_DZ = (0, 1, 2, 5), (0, 1, 3, 7)      # where conv_inputs puts a case's bad value
NONFINITE_DMMA = [c["name"] for c in CONV_CASES if c["bad"] is not None and c["name"].split("_")[1] in ("nan", "inf")]


def _run_family(engine, out_path):
    """Subprocess body: every case of one engine, results and the kernels that ran into one .npz."""
    import torch
    sys.path.insert(0, ROOT)
    from mercer_research_b200 import _lib, ext
    res = {}
    for c in CONV_CASES:
        if engine == "dmma" and c["name"] not in NONFINITE_DMMA:
            continue
        x, w, dz = conv_inputs(c)
        if c["offset"]:
            def dev(a):
                buf = torch.zeros(a.size + 1, dtype=torch.float64, device="cuda")
                buf[1:] = torch.from_numpy(a.ravel())
                return buf[1:].view(a.shape)
            x, dz, w = dev(x), dev(dz), torch.from_numpy(w).cuda()
        for op in c["ops"]:
            key = f"{c['name']}/{op}"
            _lib.profile_enable(True)
            try:
                if op == "fwd":
                    out = ext.conv2d_forward(x, w, None, c["pad"], 0)
                elif op == "bwd":
                    out = ext.conv2d_backward_data(dz, w, (c["H"], c["W"]), c["pad"])
                else:
                    out, db = ext.conv2d_backward_weight(x, dz, c["kh"], c["kw"], c["pad"])
                    res[key + "/db"] = db.cpu().numpy() if torch.is_tensor(db) else db
                res[key] = out.cpu().numpy() if torch.is_tensor(out) else out
                res[key + "/kernels"] = np.array(sorted(_lib.profile_report()))
            except _lib.RcnCudaError as e:
                res[key + "/error"] = np.array(str(e))
            _lib.profile_enable(False)
    np.savez(out_path, **res)


def _family(engine, tmp_path_factory):
    out = str(tmp_path_factory.mktemp("ozaki") / f"{engine}.npz")
    env = dict(os.environ, RCN_CUDA_GEMM=engine, RCN_CUDA_CONV_DIRECT="0")
    p = subprocess.run([sys.executable, os.path.abspath(__file__), engine, out], env=env, capture_output=True, text=True)
    assert p.returncode == 0, p.stderr[-3000:]
    with np.load(out) as f:
        return {k: f[k] for k in f.files}


@pytest.fixture(scope="module")
def tc_results(built_library, tmp_path_factory):
    return _family("tc", tmp_path_factory)


@pytest.fixture(scope="module")
def dmma_results(built_library, tmp_path_factory):
    return _family("dmma", tmp_path_factory)


def _op_result(res, c, op, tc=True):
    key = f"{c['name']}/{op}"
    assert key + "/error" not in res, (key, str(res[key + "/error"]))
    names = [str(n) for n in res[key + "/kernels"]]
    Ho, Wo, _, _ = geometry(c)
    tag = {"fwd": "conv2d_forward_igemm", "bwd": "conv2d_backward_data_igemm", "wgt": "conv2d_backward_weight_igemm"}[op]
    gemm = [n for n in names if n.startswith(tag)]
    assert len(gemm) == 1, (key, names)
    tma = False
    if tc:
        grid, C = ((Ho, Wo), c["Ci"]) if op == "fwd" else ((c["H"], c["W"]), c["Co"])
        tma = op != "wgt" and not c["offset"] and tma_ok(*grid, C, c["kh"] * c["kw"] * C)
        want = f"{tag}(tcgen05 int8 slices{', TMA im2col' if tma else ''})"
        assert gemm[0] == want, (key, gemm[0], want)
    else:
        assert gemm[0] == tag, (key, names)
    return res[key], tma


CONV_IDS = [c["name"] for c in CONV_CASES if c["bad"] is None]


@pytest.mark.gpu
@pytest.mark.parametrize("name", CONV_IDS)
def test_conv_matches_emulation_and_f64_componentwise(tc_results, name):
    """Forward, backward-data and backward-weight on the path the shape selects; a batch whose images differ in scale by
    up to 1e8 must meet the componentwise bar in every image.  Pixels far apart inside one image meet it on the per-row
    gather; on the TMA path, whose scale unit is the image, they meet the unit bar."""
    c = next(c for c in CONV_CASES if c["name"] == name)
    x, w, dz = conv_inputs(c)
    for op in c["ops"]:
        got, tma = _op_result(tc_results, c, op)
        exp = conv_expect(c, op, x, w, dz, tma)
        componentwise = not (tma and c["intra"] is not None)
        if not componentwise:   # the case lies where the componentwise bar does not hold for the scheme itself
            emu, ref, terms = exp[0], exp[2], exp[3]
            assert np.max(np.abs(emu - ref) / terms) > BAR, (name, op)
        check(got, *exp, f"{name}/{op}", componentwise)
        if op == "wgt":
            db = tc_results[f"{name}/wgt/db"]
            assert (np.abs(db - dz.sum((0, 1, 2))) <= BAR * np.abs(dz).sum((0, 1, 2))).all(), name


@pytest.mark.gpu
@pytest.mark.parametrize("name", [c["name"] for c in CONV_CASES if c["bad"] is not None])
def test_conv_non_finite_values_stay_in_their_unit(tc_results, name):
    """NaN, Inf or 1e300 at one element of image 0 of x and of dz.  The integer-slice paths poison by scale unit: the
    pixel row (per-row gather) or the image (TMA), the input channel (x in backward-weight) or the output channel (dz in
    backward-weight).  Every other output is finite and meets the bar; every output f64 makes non-finite is non-finite."""
    c = next(c for c in CONV_CASES if c["name"] == name)
    x, w, dz = conv_inputs(c)
    Ho, Wo, ph, pw = geometry(c)
    for op in c["ops"]:
        got, tma = _op_result(tc_results, c, op)
        exp = conv_expect(c, op, x, w, dz, tma)
        check(got, *exp, f"{name}/{op}")
        got_bad = ~np.isfinite(got)
        unit = np.zeros(got.shape, bool)
        if op == "wgt":
            unit[:, :, :, BAD_X[3]] = True
            unit[BAD_DZ[3]] = True
        elif tma:
            unit[0] = True
        else:   # the pixels whose receptive field holds the bad element
            ind = np.zeros(x.shape if op == "fwd" else dz.shape)
            ind[BAD_X if op == "fwd" else BAD_DZ] = 1.0
            grid, pads = ((Ho, Wo), (ph, pw)) if op == "fwd" else ((c["H"], c["W"]), (c["kh"] - 1 - ph, c["kw"] - 1 - pw))
            rows = im2col(ind, *grid, c["kh"], c["kw"], *pads, 0, c["B"] * grid[0] * grid[1]).any(1)
            unit.reshape(-1, got.shape[-1])[rows] = True
        assert np.array_equal(got_bad, unit), (name, op, int(got_bad.sum()), int(unit.sum()))


@pytest.mark.gpu
@pytest.mark.parametrize("name", NONFINITE_DMMA)
def test_conv_non_finite_values_on_dmma_match_f64(dmma_results, name):
    """The f64 DMMA implicit GEMMs make non-finite exactly the outputs f64 does."""
    c = next(c for c in CONV_CASES if c["name"] == name)
    x, w, dz = conv_inputs(c)
    for op in c["ops"]:
        got, _ = _op_result(dmma_results, c, op, tc=False)
        _, _, ref, terms, ref_bad, _ = conv_expect(c, op, x, w, dz, False)
        got = got.reshape(ref.shape)
        assert np.array_equal(~np.isfinite(got), ref_bad), (name, op)
        ok = ~ref_bad
        assert (np.abs(got - ref)[ok] <= BAR * terms[ok]).all(), (name, op)


if __name__ == "__main__":
    _run_family(sys.argv[1], sys.argv[2])
