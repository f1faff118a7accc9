"""CPU tests of the drop-in boundary: the C-ABI library loads, exports every symbol include/rcn_cuda.h declares,
fails loudly without a GPU, and the product never routes through the oracle."""
import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "rcn_cuda.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(rcn_cuda_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_exported(built_library):
    syms = declared_symbols()
    assert len(syms) >= 40
    raw = ctypes.CDLL(os.path.join(ROOT, "mercer_research_b200", "librcn_cuda.so"))
    for s in syms:
        assert hasattr(raw, s), f"{s} declared in include/rcn_cuda.h but not exported"


def test_binding_covers_header(built_library):
    from mercer_research_b200 import _lib
    assert set(_lib.SIGNATURES) | {"rcn_cuda_last_error"} == set(declared_symbols())


def test_rust_extern_block_covers_header():
    """rust/src/ffi.rs (the binding a maintainer adds to rcn, INTEGRATION.md section 2) declares every header entry point
    with the header's parameter count; it cannot be compiled here (no rustc), so at least keep it in step textually."""
    header = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "rcn_cuda.h")).read(), flags=re.S)
    rust = re.sub(r"//.*", "", open(os.path.join(ROOT, "rust", "src", "ffi.rs")).read())

    def arity(text, pattern):
        out = {}
        for name, args in re.findall(pattern, text, flags=re.S):
            args = args.strip()
            out[name] = 0 if args in ("", "void") else args.count(",") + 1
        return out

    c = arity(header, r"\b(rcn_cuda_[a-z0-9_]+)\s*\(([^)]*)\)\s*;")
    r = arity(rust, r"pub fn (rcn_cuda_[a-z0-9_]+)\s*\(([^)]*)\)")
    assert set(c) == set(declared_symbols())
    assert set(r) == set(c), (sorted(set(c) - set(r)), sorted(set(r) - set(c)))
    assert {k: v for k, v in r.items() if c[k] != v} == {}


def test_version_and_error_string(built_library):
    assert built_library.rcn_cuda_version() >= 100
    assert isinstance(built_library.rcn_cuda_last_error(), bytes)


NO_DEVICE_SCRIPT = r"""
import sys
import numpy as np
import pytest
sys.path.insert(0, %(root)r)
from mercer_research_b200 import RCN, Padding, Pooling, RCNLayer, RcnCudaError, convolve_2d_separated
with pytest.raises(RcnCudaError) as e:
    RCN(10, [RCNLayer.Convolve2D(Padding.Same), RCNLayer.Pool2D(Pooling.Max)], [30])
assert e.value.status == 4 and "no CPU fallback" in e.value.message, e.value
with pytest.raises(RcnCudaError):
    convolve_2d_separated(np.zeros((5, 5)), 0, Padding.Same)
print("ok")
"""


def test_no_cpu_fallback_without_gpu(built_library):
    """Without a usable device the library refuses to compute. Runs in a process whose devices are hidden, so that a GPU
    machine checks it too."""
    import subprocess
    import sys
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, "-c", NO_DEVICE_SCRIPT % {"root": ROOT}], env=env, capture_output=True, text=True,
                       timeout=300)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr


def test_argument_validation_needs_no_gpu(built_library):
    """Contract violations are reported before any device work (reference panics: kernel.rs:127,133,200,247,284)."""
    from mercer_research_b200 import Padding, Pooling, RcnCudaError, convolve_2d, convolve_2d_separated, pool_2d
    cases = [
        (lambda: convolve_2d_separated(np.zeros((2, 5)), 0, Padding.Same), 2),
        (lambda: pool_2d(np.zeros((1, 5)), Padding.Same, Pooling.Max), 2),
        (lambda: pool_2d(np.zeros((4, 4)), Padding.Same, Pooling.Average), 3),
        (lambda: convolve_2d(np.zeros((4, 4)), np.zeros((2, 2)), Padding.Same), 2),
        (lambda: convolve_2d(np.zeros((2, 2)), np.zeros((3, 3)), Padding.None_), 2),
        (lambda: convolve_2d(np.zeros((8, 8)), np.zeros((5, 5)), Padding.Same), 6),
    ]
    for fn, status in cases:
        with pytest.raises(RcnCudaError) as e:
            fn()
        assert e.value.status == status, e.value


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "mercer_research_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(import|from)\s+oracle", src, flags=re.M), f
                assert "librcn_oracle" not in src, f


def test_layer_codes_and_enums():
    from mercer_research_b200 import Padding, Pooling, RCNLayer, SeparableOperator
    assert RCNLayer.Convolve2D(Padding.None_).code == 0 and RCNLayer.Convolve2D(Padding.Same).code == 1
    assert RCNLayer.Pool2D(Pooling.Average).code == 2 and RCNLayer.Pool2D(Pooling.Max).code == 3
    assert [int(x) for x in SeparableOperator] == [0, 1, 2, 3]  # Top, Bottom, Left, Right (kernel.rs:16-21)


def test_built_library_carries_the_blackwell_instructions(built_library):
    """The shipped library is sm_100a machine code that really uses the units DESIGN.md names (no GPU needed to see it):
    tcgen05 integer MMA + TMEM loads + their mbarrier commits (Ozaki GEMM / conv), TMA tensor loads and the 5-D
    im2col boxes, bulk-async copies (staged feature kernel), FP64 tensor-core DMMA, cp.async rings."""
    import shutil
    import subprocess
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    so = os.path.join(ROOT, "mercer_research_b200", "librcn_cuda.so")
    elf = subprocess.run([cuobjdump, "-lelf", so], capture_output=True, text=True, check=True).stdout
    assert "sm_100a" in elf and not re.search(r"sm_(?!100a)\d+", elf), elf      # one target, no multi-arch fatbin
    sass = subprocess.run([cuobjdump, "-sass", so], capture_output=True, text=True, check=True).stdout
    for mnemonic in ("UTCIMMA", "LDTM", "UTCBAR", "UTMALDG.3D", "UTMALDG.5D", "UBLKCP", "DMMA", "LDGSTS"):
        assert mnemonic in sass, f"{mnemonic} not found in the library's SASS"
