#!/usr/bin/env python
"""bench.py -- training images/sec of rcn's hot path on N B200s (one process per GPU) + roofline + CPU baseline.

  python bench.py --gpus 1 --steps K --warmup W                       # this repo's CUDA path
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
  python bench.py --impl reference --gpus N --steps K --warmup W      # reference CPU algorithm (oracle) on host cores

A "step" is one pass of the hot path over one minibatch: u8 images -> Sobel/ReLU/max-pool features -> standardise
-> sigmoid MLP forward -> backprop -> batch gradient sum -> (all-reduce over ranks) -> SGD update
(rcn/src/rcn.rs:317-356, 407-412, 260-314, 176-223).  Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import gc
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# BASELINE.json configs -> concrete shapes (SURVEY.md 8d). `batch` is PER GPU (weak scaling).
WORKLOADS = {
    # configs[1]: MNIST-shaped CNN (28x28x1, one conv+pool+dense+softmax-position layer), batch 1024
    "c2": dict(desc="rcn MNIST-shaped CNN 28x28 [Conv(Same),Pool(Max)] 784-30-10, batch 1024 per GPU",
               H=28, W=28, cfg=[1, 3], ff=[30], classes=10, batch=1024),
    # configs[0]: the CPU-runnable case (same net, batch 32)
    "c1": dict(desc="rcn MNIST-shaped CNN 28x28 [Conv(Same),Pool(Max)] 784-30-10, batch 32 per GPU",
               H=28, W=28, cfg=[1, 3], ff=[30], classes=10, batch=32),
    # configs[2] in reference semantics: grayscale 32x32, [C,P]x3 -> 64 maps 4x4 = 1024 feats -> 1024-256-10
    "c3": dict(desc="CIFAR-shaped 32x32 gray [C,P]x3 1024-256-10, batch 4096 per GPU",
               H=32, W=32, cfg=[1, 3, 1, 3, 1, 3], ff=[256], classes=10, batch=4096),
    # configs[4]: 64x64 [C,P] -> 4096 feats -> 4096-4096-4096-10
    "c5": dict(desc="dense-heavy head 64x64 [C,P] 4096-4096-4096-10, batch 8192 per GPU",
               H=64, W=64, cfg=[1, 3], ff=[4096, 4096], classes=10, batch=8192),
    # configs[3] in reference semantics: the "wide conv stack" is four stacked Convolve2D(Same) layers on 64x64 inputs -- the
    # reference's convolution has no channel contraction, every layer fans each map out x4: 4 -> 16 -> 64 -> 256 maps of 64x64
    # (SURVEY.md 8d C4).  Feature stage only (flatten_feature_set + standardise): 2 MiB x 4 of f64 features per image make a
    # dense head meaningless; HBM-bound integer/byte work.  (The learned-convolution reading of this config is the (X)
    # extension, profiles/conv_bench.py.)
    "c4": dict(desc="wide conv stack 64x64 [Conv(Same)]x4 -> 256 maps of 64x64 (feature stage only), batch 128 per GPU",
               H=64, W=64, cfg=[1, 1, 1, 1], ff=[30], classes=10, batch=128),
}
_RESULT_FD = 1


def emit_result(line: dict):
    os.write(_RESULT_FD, (json.dumps(line) + "\n").encode())


ETA = 3.0  # main.rs:32
DATA_SEED, PARAM_SEED = 0x5EED, 0xC0FFEE
# --dump-outputs: at most 4 MiB of float64 per array. At most four training workloads (the main one and the extra ones) write
# three arrays that can be that large (params, grads, e2e_params) and the feature-stage workload one: under 55 MB in all
DUMP_MAX_ELEMENTS, DUMP_SEED = 1 << 19, 0xD5


def dump_array(a):
    """float64 numpy copy of ``a`` (numpy array or torch tensor) for --dump-outputs. An array of more than DUMP_MAX_ELEMENTS
    elements is sampled: its flattened elements at a fixed, seeded set of indices, the same for the same size, so that two
    builds are compared element for element."""
    n = int(np.prod(a.shape))
    if n > DUMP_MAX_ELEMENTS:
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(n, DUMP_MAX_ELEMENTS, replace=False))
        if isinstance(a, np.ndarray):
            a = a.reshape(-1)[idx]
        else:
            import torch
            a = a.reshape(-1)[torch.from_numpy(idx).to(a.device)]
    if not isinstance(a, np.ndarray):
        a = a.cpu().numpy()
    return np.array(a, dtype=np.float64)


def feature_len(cfg, H, W):
    maps, h, w = 0, H, W
    for c in cfg:
        if c in (0, 1):
            maps = maps * 4 if maps else 4
            if c == 0:
                h, w = h - 2, w - 2
        elif maps:
            h, w = (h + 1) // 2, (w + 1) // 2
    return maps * h * w


def layer_shapes(wl):
    L = feature_len(wl["cfg"], wl["H"], wl["W"])
    sizes = [L] + wl["ff"] + [wl["classes"]]
    return [(sizes[i + 1], sizes[i]) for i in range(len(sizes) - 1)]


def dense_flops_per_image(shapes):
    fwd = sum(2 * r * c for r, c in shapes)
    bwd_w = fwd
    bwd_d = sum(2 * r * c for r, c in shapes[1:])
    return fwd, bwd_d, bwd_w


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm_gbs=p["hbm_gbs"], bf16_tflops=p.get("bf16_tflops"), source="measured (MEASURED_PEAKS.json)",
                    sm_max_mhz=p.get("sm_max_mhz"))
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, source="fallback (B200_PROFILING.md)", sm_max_mhz=1965.0)


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md clocks line).

    NVML is polled in-process every few ms (a timed region of this workload can be shorter than one `nvidia-smi -lms`
    period); samples carry a host timestamp and only those inside [mark_begin, mark_end] are reported. Falls back to an
    `nvidia-smi -lms 100` subprocess when pynvml is unavailable.

    A timed region expected to be shorter than 50 ms (the driver's K = 20 is half a millisecond, an eighth of the polling
    period) additionally gets one sample immediately before it and one immediately after it, taken from the timing thread (an
    NVML query takes 4-5 us on this pool's boxes; RCN_BENCH_CLOCK_QUIET=1 pauses the poller inside such a region -- measured:
    no difference, 47-49 M images/s either way)."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, gpu_index, period_s=0.004):
        self.gpu, self.period = gpu_index, period_s
        self.samples, self.windows = [], []
        self.stop_flag = False
        self.thread = None
        self.max_mhz = None
        self.mode = None
        self.paused, self.in_call, self.adjacent, self.query_s = False, False, [], []

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            idx = self.gpu
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis:
                ids = [v.strip() for v in vis.split(",") if v.strip()]
                if self.gpu < len(ids) and ids[self.gpu].isdigit():
                    idx = int(ids[self.gpu])
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.nv = pynvml
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.mode = "nvml"
            self.thread = threading.Thread(target=self._poll_nvml, daemon=True)
            self.thread.start()
        except Exception:
            self.mode = "nvidia-smi"
            try:
                q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                     "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
                self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                                              "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
                self.thread = threading.Thread(target=self._poll_smi, daemon=True)
                self.thread.start()
            except Exception:
                self.mode = None

    def _sample_nvml(self):
        nv = self.nv
        t = time.perf_counter()
        try:
            sm = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
            try:
                mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
            except Exception:
                mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
            self.samples.append((t, sm, mask))
            self.query_s.append(time.perf_counter() - t)
        except Exception:
            pass

    def _poll_nvml(self):
        while not self.stop_flag:
            if self.paused:
                time.sleep(0.0005)
                continue
            self.in_call = True
            self._sample_nvml()
            self.in_call = False
            time.sleep(self.period)

    def _poll_smi(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            try:
                sm, mx = float(f[0]), float(f[1])
            except (ValueError, IndexError):
                continue
            self.max_mhz = mx
            mask = 0
            for bit, v in zip([0x8, 0x40, 0x20, 0x4], f[2:6]):
                if v.lower().startswith("active"):
                    mask |= bit
            self.samples.append((time.perf_counter(), sm, mask))

    def mark_begin(self, expected_s=None):
        short = self.mode == "nvml" and expected_s is not None and expected_s < 0.05
        if short:
            if os.environ.get("RCN_BENCH_CLOCK_QUIET", "0") == "1":
                self.paused = True
                while self.in_call:             # a query already in flight finishes first
                    time.sleep(0.0002)
            self._sample_nvml()                 # ... immediately before the region, from this thread
            self.adjacent.append(len(self.samples) - 1)
        self._short = short
        self._t0 = time.perf_counter()

    def mark_end(self):
        self.windows.append((self._t0, time.perf_counter()))
        if getattr(self, "_short", False):
            self._sample_nvml()                 # ... and immediately after it
            self.adjacent.append(len(self.samples) - 1)
            self.paused = False

    def stop(self):
        if self.mode is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock sampling unavailable"], "samples": 0}
        time.sleep(0.02 if self.mode == "nvml" else 0.15)
        self.stop_flag = True
        if self.mode == "nvidia-smi":
            self.proc.terminate()
        inside = [x for x in self.samples if any(a <= x[0] <= b for a, b in self.windows)]
        note = "samples inside the timed regions"
        if self.adjacent:
            inside = inside + [self.samples[i] for i in self.adjacent if i < len(self.samples)]
            note = ("samples inside the timed regions plus, for regions shorter than 50 ms, one immediately before and one immediately "
                    "after each (an NVML query takes %.0f us here)" % (1e6 * float(np.median(self.query_s)) if self.query_s else 0.0))
        if not inside and self.windows:      # region shorter than one sampling period: nearest samples under the same load
            a, b = self.windows[0][0], self.windows[-1][1]
            inside = [x for x in self.samples if a - 0.25 <= x[0] <= b + 0.05]
            note = "timed region shorter than a sampling period: samples within 250 ms before it (warm-up, same load)"
        mask = 0
        for x in inside:
            mask |= x[2]
        sm = [x[1] for x in inside]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(name for bit, name in self.REASONS.items() if mask & bit), "samples": len(sm),
                "source": self.mode, "note": note}


# ---------------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle's threaded train step (C++ restatement of rcn's CPU path -- NOT rustc output)
# ---------------------------------------------------------------------------------------------------------------------
def cpu_sample_batch(wl, cores):
    """Bounded CPU sample: the full minibatch when one CPU step is small, else a sub-batch of the same workload sized
    to ~2e10 flop per step (the per-sample cost of the reference algorithm does not depend on the batch size)."""
    shapes = layer_shapes(wl)
    fwd, bwd_d, bwd_w = dense_flops_per_image(shapes)
    per_image = fwd + bwd_d + bwd_w + 12 * 4 * wl["H"] * wl["W"]
    b = int(2e10 // per_image)
    b = max(4 * cores, b - b % max(1, cores))
    return min(wl["batch"], b)


def cpu_train_steps(wl, steps, warmup, max_seconds=None, batch=None):
    import oracle as O
    B, H, W = batch or wl["batch"], wl["H"], wl["W"]
    shapes = layer_shapes(wl)
    net = O.Net(shapes)
    rng = np.random.default_rng(DATA_SEED)
    n_pool = 4
    images = rng.integers(0, 256, size=(n_pool, B, H, W), dtype=np.uint8)
    labels = (np.arange(B) % wl["classes"]).astype(np.int64)
    params = np.random.default_rng(PARAM_SEED).standard_normal(net.n_params)
    mean, sd = O.gen_scales(O.features_u8(wl["cfg"], images[0][:min(B, 256)]))
    cores = os.cpu_count() or 1
    t_w = time.perf_counter()
    for i in range(warmup):
        net.train_step_u8(wl["cfg"], params, images[i % n_pool], labels, mean, sd, ETA, cores)
        if max_seconds and time.perf_counter() - t_w > max_seconds / 2:
            break
    t0 = time.perf_counter()
    done = 0
    for i in range(steps):
        net.train_step_u8(wl["cfg"], params, images[i % n_pool], labels, mean, sd, ETA, cores)
        done += 1
        if max_seconds and time.perf_counter() - t0 > max_seconds:
            break
    dt = time.perf_counter() - t0
    return done * B / dt, dt / done * 1e3, done, cores, B


def run_reference(args, wl, rank, world):
    if rank != 0:
        return
    # bounded sample: each step is one (sub-)minibatch of the same workload on all host threads; cap the run at ~2 min
    cores = os.cpu_count() or 1
    Bs = cpu_sample_batch(wl, cores)
    ips, ms, done, cores, Bs = cpu_train_steps(wl, args.steps, args.warmup, max_seconds=100.0, batch=Bs)
    sample = (f"{done} steps of batch {Bs} (features+fwd+bwd+SGD) on {cores} host threads" +
              ("" if Bs == wl["batch"] else f"; sub-batch of the {wl['batch']}-image minibatch, per-sample cost is batch-independent"))
    line = {
        "impl": "reference", "metric": "training images/sec", "value": ips, "unit": "images/s", "n_gpus": args.gpus,
        "steps": done, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": wl["desc"], "batch_per_step": Bs, "batch_per_gpu": wl["batch"], "pixels": "u8", "eta": ETA,
                   "note": "C++ restatement of rcn's CPU path (oracle/rcn_oracle.cpp: per-sample matvec backprop, worker threads "
                           "+ mutex-ordered gradient sum as rcn.rs:176-223); the Rust crate cannot be built here (no rustc)"},
        "cpu_baseline": {"value": ips, "unit": "images/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": ips, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit_result(line)


# ---------------------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------------------
_WC_KEEP = []   # write-combined allocations stay alive for the life of the process


def _wc_pinned_copy(a):
    """numpy array -> the same bytes in cudaHostAllocWriteCombined memory (viewed as a numpy array), or None if the CUDA
    runtime cannot be reached from here. CPU reads of such memory are slow; the bench only writes it once."""
    import ctypes
    try:
        import torch
        rt = ctypes.CDLL(os.path.join(os.path.dirname(torch.__file__), "..", "nvidia", "cuda_runtime", "lib", "libcudart.so.12"))
    except OSError:
        try:
            rt = ctypes.CDLL("libcudart.so.12")
        except OSError:
            return None
    p = ctypes.c_void_p()
    rt.cudaHostAlloc.argtypes = [ctypes.POINTER(ctypes.c_void_p), ctypes.c_size_t, ctypes.c_uint]
    if rt.cudaHostAlloc(ctypes.byref(p), a.nbytes, 0x01 | 0x04) != 0 or not p.value:   # portable | write-combined
        return None
    buf = (ctypes.c_uint8 * a.nbytes).from_address(p.value)
    out = np.frombuffer(buf, dtype=a.dtype).reshape(a.shape)
    out[...] = a
    _WC_KEEP.append((rt, p, buf))
    return out


def measure_fp64_peak(torch, dev):
    """cuBLAS DGEMM 8192^3 via torch.matmul -- the f64 denominator MEASURED_PEAKS.json lacks (BASELINE.md section 2)."""
    n = 8192
    a = torch.randn(n, n, dtype=torch.float64, device=dev)
    b = torch.randn(n, n, dtype=torch.float64, device=dev)
    torch.matmul(a, b)
    torch.cuda.synchronize()
    best = 1e9
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); torch.matmul(a, b); e1.record(); torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    del a, b
    return 2 * n ** 3 / (best * 1e-3) / 1e12


def measure_int8_peak(torch, dev):
    """cuBLASLt IGEMM 8192^3 (s8 x s8 -> s32, torch._int_mm): the int8 tensor-pipe denominator of the tcgen05 integer-slice
    GEMMs, MEASURED on this box (round 1 assumed 2 x the bf16 figure). Returns (TOP/s, how) or (None, why)."""
    try:
        n = 8192
        a = torch.randint(-128, 128, (n, n), dtype=torch.int8, device=dev)
        b = torch.randint(-128, 128, (n, n), dtype=torch.int8, device=dev)
        torch._int_mm(a, b)
        torch.cuda.synchronize()
        best = 1e9
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); torch._int_mm(a, b); e1.record(); torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        del a, b
        return 2 * n ** 3 / (best * 1e-3) / 1e12, "torch._int_mm (cuBLASLt IGEMM s8*s8->s32) 8192^3, best of 5, measured in this run"
    except Exception as e:  # noqa: BLE001
        return None, f"int8 IGEMM probe failed ({type(e).__name__}: {e})"


class Ctx:
    pass


def _barrier(ctx):
    ctx.torch.cuda.synchronize()
    if ctx.world > 1:
        ctx.dist.barrier()
    ctx.torch.cuda.synchronize()


def _max_over_ranks(ctx, x):
    if ctx.world == 1:
        return x
    t = ctx.torch.tensor([x], dtype=ctx.torch.float64, device=ctx.dev)
    ctx.dist.all_reduce(t, op=ctx.dist.ReduceOp.MAX)
    return float(t.item())


def on_tc(M, N, K):                                   # mirrors use_tensor_cores() in csrc/dense.cu
    tiles = -(-M // 128) * -(-N // 96)
    return M >= 256 and N >= 256 and K >= 512 and K <= 16384 and tiles >= 74 and float(M) * N * K >= 4.0e9


def kernel_rooflines(wl, B, shapes, prof, prof_steps, pk, fp64_peak, int8_peak):
    """Per-kernel achieved rates from the eager per-launch CUDA-event pass (`prof`: name -> launches, total_ms) against the
    algorithmic work of DESIGN.md section 4. Returns (kernels dict, name of the kernel with the largest share)."""
    H, W = wl["H"], wl["W"]
    L = shapes[0][1]
    n_params = sum(r * c + r for r, c in shapes)
    fwd, bwd_d, bwd_w = dense_flops_per_image(shapes)
    sum_rows = sum(r for r, _ in shapes)
    act_bytes = 2 * sum_rows * 8                      # a_l and delta_l written once per sample
    alg = {
        "features_fused_kernel": ["hbm", B * (H * W * 1 + L * 8), B * 48 * H * W],
        "smallnet_fwd_bwd_kernel(fused features)": ["fp64", B * (H * W * 1 + 8 + L * 8 + act_bytes) + n_params * 8,
                                                    B * (48 * H * W + fwd + bwd_d)],
        "smallnet_fwd_bwd_kernel(fused features, front end ahead of the exchange)": ["fp64", B * (H * W * 1 + 8 + L * 8 + act_bytes) + n_params * 8,
                                                                                      B * (48 * H * W + fwd + bwd_d)],
        "smallnet_fwd_bwd_kernel(fused features, front end ahead of the wait)": ["fp64", B * (H * W * 1 + 8 + L * 8 + act_bytes) + n_params * 8,
                                                                                  B * (48 * H * W + fwd + bwd_d)],
        "smallnet_fwd_bwd_kernel": ["fp64", B * (L * 8 + 8 + act_bytes) + n_params * 8, B * (fwd + bwd_d)],
        "smallnet_wgrad_kernel": ["fp64", B * (L + shapes[0][0]) * 8 + n_params * 8, B * bwd_w],
        "smallnet_wgrad_kernel(+SGD update)": ["fp64", B * (L + shapes[0][0]) * 8 + 3 * n_params * 8, B * bwd_w + 2 * n_params],
        "smallnet_wgrad_kernel(+exchange+SGD update)": ["fp64", B * (L + shapes[0][0]) * 8 + 3 * n_params * 8, B * bwd_w + 2 * n_params],
        "features_cp_kernel": ["hbm", B * (H * W * 1 + L * 8), B * 48 * H * W],
        "sgd_update_kernel": ["hbm", 3 * n_params * 8, 2 * n_params],
        "dp_allreduce_sgd_kernel": ["hbm", 3 * n_params * 8, 2 * n_params],
        "bias_grad_kernel": ["hbm", B * sum_rows * 8, B * sum_rows],
        # skinny output layer (rows <= 16 behind a wide layer): each kernel streams the wide activation matrix once
        "skinny_forward_kernel": ["hbm", B * (shapes[-1][1] + 2 * shapes[-1][0]) * 8, 2 * B * shapes[-1][0] * shapes[-1][1]],
        "skinny_backward_data_kernel": ["hbm", B * (2 * shapes[-1][1] + shapes[-1][0]) * 8, 2 * B * shapes[-1][0] * shapes[-1][1]],
        "skinny_backward_weight_kernel": ["hbm", B * (shapes[-1][1] + shapes[-1][0]) * 8, 2 * B * shapes[-1][0] * shapes[-1][1]],
    }
    for tag in ("forward", "backward_data", "backward_weight"):
        for suffix in ("", "(tcgen05 int8 slices)"):
            alg[f"dense_{tag}_gemm{suffix}"] = ["tensor", 0, 0]
    slice_bytes = 0
    for li, (r, c) in enumerate(shapes):
        f = 2.0 * r * c * B
        tc_f, tc_w = on_tc(r, B, c), on_tc(r, c, B)
        alg["dense_forward_gemm" + ("(tcgen05 int8 slices)" if tc_f else "")][2] += f
        alg["dense_backward_weight_gemm" + ("(tcgen05 int8 slices)" if tc_w else "")][2] += f
        slice_bytes += (13 * (r * c + c * B) if tc_f else 0) + (13 * (r * B + c * B) if tc_w else 0)
        if li >= 1:
            rp = shapes[li - 1][0]                    # backward-data into layer li-1: M = rp, K = r, N = B
            tc_d = on_tc(rp, B, r)
            alg["dense_backward_data_gemm" + ("(tcgen05 int8 slices)" if tc_d else "")][2] += 2.0 * rp * r * B
            slice_bytes += 13 * (rp * r + r * B) if tc_d else 0
    alg["ozaki_slice"] = ["hbm", slice_bytes, 0]      # both slicing kernels together: 8 B read + 5 B written per element
    kernels = {k: {"launches_per_step": v["launches"] / prof_steps, "avg_us": v["total_ms"] / v["launches"] * 1e3,
                   "share": None} for k, v in prof.items()}
    tot = sum(v["total_ms"] for v in prof.values()) or 1.0
    for k, v in prof.items():
        kernels[k]["share"] = round(v["total_ms"] / tot, 4)
        key = "ozaki_slice" if k.startswith("ozaki_slice") or k.startswith("ozaki_amax") else k
        if key in alg:
            d_s = v["total_ms"] / prof_steps * 1e-3          # seconds of this kernel name per step
            if key == "ozaki_slice":
                d_s = sum(x["total_ms"] for n_, x in prof.items() if n_.startswith("ozaki_slice") or n_.startswith("ozaki_amax")) / prof_steps * 1e-3
            bnd, nbytes, nflops = alg[key]
            kernels[k]["bound"] = bnd
            if nbytes:
                kernels[k]["GBps"] = round(nbytes / d_s / 1e9, 1)
                kernels[k]["frac_hbm"] = round(nbytes / d_s / 1e9 / pk["hbm_gbs"], 4)
            if nflops and "tcgen05" in k:
                kernels[k]["f64_equiv_TFLOPs"] = round(nflops / d_s / 1e12, 2)
                kernels[k]["int8_TOPs"] = round(15 * nflops / d_s / 1e12, 1)     # 15 digit-plane products per f64 product
                kernels[k]["frac_int8_tensor"] = round(15 * nflops / d_s / 1e12 / int8_peak, 4)
            elif nflops:
                kernels[k]["TFLOPs_f64"] = round(nflops / d_s / 1e12, 3)
                kernels[k]["frac_fp64"] = round(nflops / d_s / 1e12 / fp64_peak, 4)
    top = max(prof, key=lambda k: prof[k]["total_ms"]) if prof else None
    return kernels, top, alg


def run_leg(ctx, name, wl, B, steps, warmup, exchange, *, main, steps_per_graph=5, no_graph=False, host_alloc="pinned",
            dump=False):
    """One workload on this rank: device-resident `value` leg (epoch mode, CUDA graph), host-buffer `e2e` leg, eager per-kernel
    profile; the main leg (c2) additionally reads the in-graph device timeline. Collective on every rank; returns a dict
    (rank 0's view; timings are max over ranks). ``dump``: rank 0 keeps the outputs of the last timed step in ``_outputs``."""
    torch, dist, dev, rank, world = ctx.torch, ctx.dist, ctx.dev, ctx.rank, ctx.world
    from mercer_research_b200 import RCN, _lib
    from mercer_research_b200.trainer import DataParallelTrainer
    H, W = wl["H"], wl["W"]
    shapes = layer_shapes(wl)
    L = shapes[0][1]
    n_params = sum(r * c + r for r, c in shapes)
    model = RCN(wl["classes"], wl["cfg"], wl["ff"], device=ctx.local_rank)
    assert model.feature_len(H, W) == L
    model.load_weights_and_bias(L)
    assert model.layer_shapes == shapes
    scale = 1.0 if L <= 1024 else 1.0 / 64.0        # the 4096-wide layers: N(0,1)/64 keeps the sigmoids out of saturation
    seeded_params = np.random.default_rng(PARAM_SEED).standard_normal(n_params) * scale
    model.set_params(seeded_params)                 # same replica on every rank
    trainer = DataParallelTrainer(model, eta=ETA, exchange=exchange)

    # synthetic dataset resident in HBM, larger than L2 (126 MB) so that consecutive steps never hit in L2
    pool_bytes = 192 << 20
    n_batches = max(4, -(-pool_bytes // (B * H * W)))
    g = torch.Generator(device=dev); g.manual_seed(DATA_SEED + rank)
    images = torch.randint(0, 256, (n_batches, B, H, W), dtype=torch.uint8, device=dev, generator=g)
    labels = (torch.arange(B, device=dev) % wl["classes"]).to(torch.int64)
    raw = model.flatten_feature_set(images[0][:min(B, 1024)])
    model.gen_scales(raw)                       # (mean, sd) are fixed inputs on the streaming path (SURVEY.md 8a a6)
    if world > 1:                               # every replica must use the same scale_set
        ms = torch.tensor(model.scale_set, dtype=torch.float64, device=dev)
        dist.broadcast(ms, 0)
        model.scale_set = tuple(ms.tolist())
    del raw
    stream = torch.cuda.current_stream(dev)
    model.set_stream(stream.cuda_stream)
    use_timeline = main and not no_graph

    # epoch mode: the resident dataset is walked in chunks_exact(B) steps by a device-side cursor (rcn.rs:144-149),
    # so ONE captured CUDA graph (all kernels + the exchange) replays for every step.
    all_labels = labels.repeat(n_batches)
    trainer.bind_dataset(images.view(n_batches * B, H, W), all_labels, B)
    step_desc = trainer.describe()
    graph_ok = not no_graph and (world == 1 or trainer.p2p)   # the NCCL all-reduce is issued eagerly (a captured NCCL
                                                              # graph blocked destroy_process_group on this stack)
    kernels_per_step = None
    if graph_ok:
        l_before = _lib.kernel_launches()
        # the timed region is a whole number of replays: the largest divisor of K that is <= --steps-per-graph
        # (data-parallel groups take graphs twice as long: a graph boundary is a full dependency, so the first kernel A of a
        # graph cannot run its front end under the previous graph's last exchange kernel -- ~4 us lost per boundary at N = 8)
        spg_cap = steps_per_graph * (2 if world > 1 else 1)
        spg = max(d for d in range(1, max(1, min(spg_cap, steps)) + 1) if steps % d == 0)
        trainer.capture(warmup=3, steps_per_graph=spg)
        kernels_per_step = (_lib.kernel_launches() - l_before) // (3 + spg)   # 3 warm-up steps + spg captured steps
    else:
        spg = 1
        l_before = _lib.kernel_launches()
        for _ in range(2):
            trainer.epoch_step()
        torch.cuda.synchronize()
        kernels_per_step = (_lib.kernel_launches() - l_before) // 2

    clocks = ClockSampler(ctx.local_rank)
    if rank == 0:
        clocks.start()
    # warm-up: at least W steps and at least ~0.3 s of the same load, so clocks have ramped before the timed region
    n_warm = max(warmup, 3)
    t_w = time.perf_counter()
    for i in range(n_warm):
        trainer.epoch_step()
    torch.cuda.synchronize()
    per_step = max((time.perf_counter() - t_w) / n_warm, 1e-6)
    extra = torch.tensor([min(200000, int(0.3 / per_step))], dtype=torch.int64, device=dev)
    if world > 1:
        dist.broadcast(extra, 0)            # every rank must run the same number of (exchanging) steps
    for i in range(int(extra.item())):
        trainer.epoch_step()
    n_warm += int(extra.item())
    # the warm-up ran a timing-dependent number of steps: the timed steps start again from the seeded parameters at the first
    # batch, so that the same arguments give them the same inputs run after run (set_params / epoch_seek copy into the
    # buffers the captured graph already uses)
    model.set_params(seeded_params)
    model.epoch_seek(0)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # no cyclic-GC pass between the graph launches of the timed region (what timeit does: at the driver's K = 20 the region is
    # four launches / 0.4 ms long, and a collection landing between two of them stalls the GPU for longer than a step)
    gc.collect()
    gc.disable()
    _barrier(ctx)
    clocks.mark_begin(expected_s=per_step * steps)
    e0.record(stream)
    trainer.epoch_steps(steps)              # exactly K steps: K / spg replays of the spg-step graph
    e1.record(stream)
    _barrier(ctx)
    clocks.mark_end()
    gc.enable()
    trainer.check()
    outputs = None
    if dump and rank == 0:      # what a caller of the step receives after the last timed step
        outputs = {"params": dump_array(model.get_params()), "grads": dump_array(model.get_gradients()),
                   "batch_stats": dump_array(np.array(model.last_batch_stats(), dtype=np.float64))}
    launches = kernels_per_step * steps
    ms_step = _max_over_ranks(ctx, e0.elapsed_time(e1)) / steps
    value = world * B / (ms_step * 1e-3)

    # ---- in-graph device timeline of the step kernels (durations inside the replayed graph, and the gaps between them) ----
    # A SEPARATE pass after the timed region (the stamps cost atomics and fences inside the kernels): enabling the timeline
    # bumps the allocation generation, so the trainer re-captures its graph with the timeline pointer baked in.
    timeline = None
    if use_timeline and graph_ok:
        model.timeline_enable(True)
        trainer.epoch_steps(-(-64 // spg) * spg)
        torch.cuda.synchronize()
        trainer.check()
    if use_timeline and graph_ok and rank == 0:
        t0, t1, n_l = model.timeline_read()
        tl = {}
        names = {0: "kernel A (features+fwd+bwd-data)", 1: "kernel B (bwd-weight + update / push)", 2: "exchange+update kernel"}
        spans = {}
        for k in (0, 1, 2):
            n = int(n_l[k])
            if n < 8:
                continue
            idx = [(n - 1 - j) % 64 for j in range(min(48, n - 1))]       # the most recent launches (all inside the timed replays)
            d = (t1[k, idx].astype(np.int64) - t0[k, idx].astype(np.int64)) * 1e-3
            spans[k] = (t0[k, idx].astype(np.int64), t1[k, idx].astype(np.int64))
            tl[names[k]] = {"us_mean": float(d.mean()), "us_min": float(d.min()), "us_max": float(d.max()), "launches_seen": n}
        if 0 in spans and 1 in spans:
            a0, a1 = spans[0]; b0, b1 = spans[1]
            gap_ab = (b0 - a1) * 1e-3                                     # same index = same step
            tl["gap A->B us"] = float(np.median(gap_ab))
            last = spans[2][1] if 2 in spans else b1                      # what precedes the next kernel A
            nxt = np.array([a0[j - 1] - last[j] for j in range(1, len(a0))]) * 1e-3   # idx is newest first: a0[j-1] is the later step
            tl["gap (end of step k) -> kernel A(k+1) us"] = float(np.median(nxt))
        timeline = tl
    if use_timeline and graph_ok:
        model.timeline_enable(False)
        _barrier(ctx)

    # ---- e2e: the reference-facing call with HOST buffers (pinned): the chunks_exact loop of rcn.rs:147-149 over a
    # host-resident dataset; every step's H2D copy and the D2H read of its (cost, hits) are inside the timed region -----
    e2e_steps_n = steps
    n_host = max(2, min(e2e_steps_n, (512 << 20) // (B * H * W)))
    hg = torch.Generator(); hg.manual_seed(DATA_SEED + rank)
    h_images = torch.randint(0, 256, (n_host * B, H, W), dtype=torch.uint8, generator=hg).pin_memory()
    h_labels = (torch.arange(n_host * B) % wl["classes"]).to(torch.int64).pin_memory()
    hi, hl = h_images.numpy(), h_labels.numpy()
    if host_alloc == "wc":
        # opt-in experiment: the same dataset in WRITE-COMBINED pinned memory (cudaHostAllocWriteCombined)
        wc = _wc_pinned_copy(hi)
        if wc is not None:
            hi, host_alloc = wc, "pinned, write-combined"

    def e2e_run(n, verify):
        """n steps over the host dataset; returns (cost, hits) of the last step."""
        done = 0
        while done < n:
            m = min(n_host, n - done)
            cost, hits = trainer.train_epoch_host(hi[:m * B], hl[:m * B], B, verify_steps=verify)
            assert len(cost) == m
            done += m
        return cost[-1], hits[-1]

    e2e_run(e2e_steps_n, True)                  # warm-up = the timed call sequence itself: buffers sized, step graphs captured,
                                                # the per-call step counts agreed on across ranks (not repeated in the timed region)
    # ... and, like the device-resident leg, ~0.3 s of the same load: the timed region of a short run (the driver's K = 20 is
    # half a millisecond) must not start on a GPU / PCIe link that idled down while the host buffers were being built
    # (measured: 18-31 M images/s without this, against 39-43 M)
    torch.cuda.synchronize()
    t_w = time.perf_counter()
    e2e_run(e2e_steps_n, False)
    torch.cuda.synchronize()
    per_call = max(time.perf_counter() - t_w, 1e-5)
    reps = torch.tensor([min(2000, int(0.3 / per_call))], dtype=torch.int64, device=dev)
    if world > 1:
        dist.broadcast(reps, 0)
    for _ in range(int(reps.item())):
        e2e_run(e2e_steps_n, False)
    model.set_params(seeded_params)             # as for the device-resident leg: the same inputs run after run
    gc.collect()
    gc.disable()
    _barrier(ctx)
    clocks.mark_begin(expected_s=per_call)
    e0.record(stream)
    e2e_last = e2e_run(e2e_steps_n, False)
    e1.record(stream)
    _barrier(ctx)
    clocks.mark_end()
    gc.enable()
    trainer.check()
    if outputs is not None:
        outputs.update({"e2e_params": dump_array(model.get_params()),
                        "e2e_batch_stats": dump_array(np.array(e2e_last, dtype=np.float64))})
    clk = clocks.stop() if rank == 0 else None
    e2e_ms = _max_over_ranks(ctx, e0.elapsed_time(e1))
    e2e_value = world * B / (e2e_ms / e2e_steps_n * 1e-3)
    h2d = B * H * W + B * 8
    d2h = 16

    # ---- per-kernel durations (CUDA events on the launching stream): separate eager pass that EVERY rank runs ------------
    prof_steps = min(steps, 50)
    _barrier(ctx)
    _lib.profile_enable(True)
    for i in range(prof_steps):
        trainer.step_images(images[i % n_batches], labels)
    torch.cuda.synchronize()
    prof = _lib.profile_report()
    _lib.profile_enable(False)
    trainer.check()
    _barrier(ctx)

    # ---- data-parallel parity self-check (world > 1), through the SAME path the timed region uses: fixed parameters, a fixed
    # 3-chunk dataset bound in epoch mode, 3 steps per captured CUDA graph, two replays back to back (6 SGD steps, the cursor
    # wraps once; kernel B advances the cursor, the exchange kernel runs under the next step's front end).  Rank 0 later
    # repeats the 6 global minibatches on ONE GPU and through the oracle ---------------------------------------------------
    parity = None
    if world > 1 and main:
        p0 = np.random.default_rng(PARAM_SEED + 1).standard_normal(n_params) * 0.05
        model.set_params(p0)
        prng = np.random.default_rng(DATA_SEED + 99)
        pg_images = prng.integers(0, 256, size=(3, world * B, H, W), dtype=np.uint8)
        pg_labels = prng.integers(0, wl["classes"], size=(3, world * B)).astype(np.int64)
        d_pi = torch.from_numpy(np.ascontiguousarray(pg_images[:, rank * B:(rank + 1) * B]).reshape(3 * B, H, W)).to(dev)
        d_pl = torch.from_numpy(np.ascontiguousarray(pg_labels[:, rank * B:(rank + 1) * B]).reshape(3 * B)).to(dev)
        trainer.bind_dataset(d_pi, d_pl, B)
        if graph_ok:
            trainer.capture(warmup=1, steps_per_graph=3)     # restores parameters and cursor after its warm-up step
        trainer.epoch_steps(6)
        torch.cuda.synchronize()
        trainer.check()
        mine = torch.from_numpy(model.get_params()).to(dev)
        gathered = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(gathered, mine)
        if rank == 0:
            allp = [t.cpu().numpy() for t in gathered]
            parity = {"steps": 6, "global_batch": world * B,
                      "replicas_bit_identical": bool(all(np.array_equal(allp[0].view(np.uint64), q.view(np.uint64)) for q in allp[1:])),
                      "path": ("epoch mode, 3 steps per CUDA graph, 2 replays" if graph_ok else "epoch mode, eager steps") +
                              (", NVLink peer-memory exchange" if trainer.p2p else ", NCCL all-reduce"),
                      "_p0": p0, "_images": pg_images, "_labels": pg_labels, "_dp_params": allp[0], "_scale": model.scale_set}

    out = {"name": name, "wl": wl, "B": B, "shapes": shapes, "n_params": n_params, "n_batches": n_batches, "value": value,
           "ms_step": ms_step, "steps": steps, "spg": spg, "graph": graph_ok, "n_warm": n_warm * spg, "launches": int(launches),
           "step_desc": step_desc, "clocks": clk, "e2e_value": e2e_value, "e2e_ms_step": e2e_ms / e2e_steps_n, "h2d": h2d, "d2h": d2h,
           "host_alloc": host_alloc, "prof": prof, "prof_steps": prof_steps, "timeline": timeline, "parity": parity,
           "p2p": trainer.p2p, "scale_set": model.scale_set, "_outputs": outputs}
    # leave the group state clean for the next leg
    if world > 1:
        trainer.graph = None
        torch.cuda.synchronize()
        dist.barrier()
        if trainer.p2p:
            model.dp_shutdown()
            trainer.p2p = False
            dist.barrier()
    model.close()
    del trainer, model, images, h_images, h_labels
    torch.cuda.empty_cache()
    return out


def run_features_leg(ctx, name, wl, B, steps, dump=False):
    """BASELINE configs[3] in reference semantics: throughput of the feature stage alone (rcn_cuda_features) on every rank
    (independent replicas: the stage has no exchange step). Device-resident inputs; the 1 GiB output per call exceeds L2.
    ``dump``: rank 0 keeps (a sample of) the last timed call's features in ``_outputs``."""
    torch, dev, rank, world = ctx.torch, ctx.dev, ctx.rank, ctx.world
    from mercer_research_b200 import RCN, _lib
    H, W = wl["H"], wl["W"]
    model = RCN(wl["classes"], wl["cfg"], wl["ff"], device=ctx.local_rank)
    L = model.feature_len(H, W)
    g = torch.Generator(device=dev); g.manual_seed(DATA_SEED + 7 + rank)
    images = torch.randint(0, 256, (4, B, H, W), dtype=torch.uint8, device=dev, generator=g)
    out = torch.empty((B, L), dtype=torch.float64, device=dev)
    model.scale_set = (100.0, 50.0)
    stream = torch.cuda.current_stream(dev)
    model.set_stream(stream.cuda_stream)
    for i in range(3):
        model.flatten_feature_set(images[i % 4], standardise=True, out=out)
    _barrier(ctx)
    clocks = ClockSampler(ctx.local_rank)
    if rank == 0:
        clocks.start()
    l0 = _lib.kernel_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    clocks.mark_begin()
    e0.record(stream)
    for i in range(steps):
        model.flatten_feature_set(images[i % 4], standardise=True, out=out)
    e1.record(stream)
    _barrier(ctx)
    clocks.mark_end()
    launches = _lib.kernel_launches() - l0
    outputs = {"features": dump_array(out)} if dump and rank == 0 else None
    clk = clocks.stop() if rank == 0 else None
    ms_step = _max_over_ranks(ctx, e0.elapsed_time(e1)) / steps
    _lib.profile_enable(True)
    for i in range(min(steps, 10)):
        model.flatten_feature_set(images[i % 4], standardise=True, out=out)
    torch.cuda.synchronize()
    prof = _lib.profile_report()
    _lib.profile_enable(False)
    model.close()
    del images, out
    torch.cuda.empty_cache()
    nbytes = B * (H * W + L * 8)
    return {"workload": wl["desc"], "value": world * B / (ms_step * 1e-3), "unit": "images/s", "ms_per_step": ms_step, "steps": steps,
            "scaling": "weak (independent replicas: no exchange step)", "batch_per_gpu": B, "feature_len": L, "gpu_launches": int(launches),
            "clocks": clk, "_nbytes": nbytes, "_prof": prof, "_prof_steps": min(steps, 10), "_outputs": outputs}


def leg_roofline(leg, pk, fp64_peak, int8_peak, int8_how, traffic_all, workload_key):
    """Roofline record of one leg (DESIGN.md section 6)."""
    wl, B, shapes = leg["wl"], leg["B"], leg["shapes"]
    H, W = wl["H"], wl["W"]
    n_params = leg["n_params"]
    fwd, bwd_d, bwd_w = dense_flops_per_image(shapes)
    kernels, top, alg = kernel_rooflines(wl, B, shapes, leg["prof"], leg["prof_steps"], pk, fp64_peak, int8_peak)
    ms_step = leg["ms_step"]
    step_bytes = B * (H * W + 8) + 3 * n_params * 8           # compulsory HBM traffic of a whole step (intermediates on chip / in L2)
    # SURVEY.md 8d per-image figures: feature stage 12 MAC/px/op x 4 ops (48 flop/px incl. zero taps) + dense fwd / bwd-data / bwd-weight
    step_flops = B * (48 * H * W + fwd + bwd_d + bwd_w)
    dense_flops = B * (fwd + bwd_d + bwd_w)
    whole = {"ms": ms_step, "compulsory_GBps": step_bytes / (ms_step * 1e-3) / 1e9,
             "frac_hbm_compulsory": step_bytes / (ms_step * 1e-3) / 1e9 / pk["hbm_gbs"],
             "TFLOPs_f64": step_flops / (ms_step * 1e-3) / 1e12, "frac_fp64": step_flops / (ms_step * 1e-3) / 1e12 / fp64_peak,
             "TFLOPs_f64_dense_only": dense_flops / (ms_step * 1e-3) / 1e12,
             "frac_fp64_dense_only": dense_flops / (ms_step * 1e-3) / 1e12 / fp64_peak}
    traffic = (traffic_all.get(workload_key, {}) or {}).get(top) if top else None
    small = top is not None and top.startswith("smallnet")
    if small:   # the fused step = kernel A + kernel B: DRAM bytes of both launches
        tw = traffic_all.get(workload_key, {}) or {}
        parts = [v for k, v in tw.items() if k.startswith("smallnet") and k in leg["prof"] and isinstance(v, (int, float))]   # the kernels this leg ran
        traffic = float(sum(parts)) if parts else None
    if small:
        # the fused narrow-network step: two kernels that are ONE dependent chain; 99 flop per compulsory byte against an FP64
        # ridge of ~5 flop/B => FP64-pipe-bound in the limit. The fraction is the WHOLE step (kernel A + kernel B + the
        # boundaries, timed in the replayed graph) against the DGEMM peak measured in this run; per-kernel durations come
        # from the in-graph device timeline.
        rl = {"kernel": "fused step = " + " + ".join(sorted(k for k in leg["prof"] if k.startswith("smallnet"))),
              "bound": "fp64", "achieved": whole["TFLOPs_f64"], "peak": fp64_peak, "unit": "TFLOP/s", "frac": whole["frac_fp64"],
              "traffic": traffic,
              "peak_source": "torch.matmul f64 8192^3 (cuBLAS DGEMM) measured in this run; MEASURED_PEAKS.json has no f64 figure",
              "achieved_is": "SURVEY 8d algorithmic flops of one step (48 flop/px feature stage + dense fwd/bwd-data/bwd-weight) / "
                             "the step's duration in the timed, graph-replayed region (CUDA events, max over ranks)",
              "hbm": {"achieved_GBps": whole["compulsory_GBps"], "peak_GBps": pk["hbm_gbs"], "frac": whole["frac_hbm_compulsory"],
                      "note": "compulsory bytes of the step (u8 images + labels + 3 x parameters); secondary: the step is not HBM-bound"}}
        if leg["timeline"]:
            tl = leg["timeline"]
            rl["in_graph_timeline"] = tl
            a = tl.get("kernel A (features+fwd+bwd-data)")
            b = tl.get("kernel B (bwd-weight + update / push)")
            if a:
                fa = B * (48 * H * W + fwd + bwd_d)
                # Kernel A starts its front end under the previous step's kernel B / exchange kernel (prewait): its span then
                # begins BEFORE that kernel ends (negative gap).  Its own share of the step is the span minus that overlap.
                overlap = max(0.0, -float(tl.get("gap (end of step k) -> kernel A(k+1) us", 0.0) or 0.0))
                us_a = max(a["us_mean"] - overlap, 1e-3)
                rl["kernel_A"] = {"us": us_a, "span_us": a["us_mean"], "overlap_with_previous_step_us": overlap,
                                  "TFLOPs_f64": fa / (us_a * 1e-6) / 1e12, "frac_fp64": fa / (us_a * 1e-6) / 1e12 / fp64_peak}
            if b:
                fb = B * bwd_w
                rl["kernel_B"] = {"us": b["us_mean"], "TFLOPs_f64": fb / (b["us_mean"] * 1e-6) / 1e12,
                                  "frac_fp64": fb / (b["us_mean"] * 1e-6) / 1e12 / fp64_peak}
    else:
        bound, nbytes, nflops = alg.get(top, ("hbm", 0, 0)) if top else ("hbm", 0, 0)
        dur_s = leg["prof"][top]["total_ms"] / leg["prof_steps"] * 1e-3 if top else 1.0
        peak_source = pk["source"]
        if bound == "hbm":
            achieved, peak, unit = nbytes / dur_s / 1e9, pk["hbm_gbs"], "GB/s"
        elif top and "tcgen05" in top:
            achieved, peak, unit = 15 * nflops / dur_s / 1e12, int8_peak, "TFLOP/s"
            peak_source = "int8 tensor peak: " + int8_how + "; achieved = 15 exact int8 digit-plane products per f64 product, in int8 TOP/s"
        else:
            achieved, peak, unit = nflops / dur_s / 1e12, fp64_peak, "TFLOP/s"
            peak_source = "torch.matmul f64 8192^3 measured in this run (f64 DMMA path; MEASURED_PEAKS.json has no f64 figure)"
        rl = {"kernel": top, "bound": "tensor" if bound == "fp64" else bound, "achieved": achieved, "peak": peak, "unit": unit,
              "frac": achieved / peak if peak else None, "traffic": traffic, "peak_source": peak_source}
    rl.update({"precision": "f64", "fp64_dgemm_tflops_measured": fp64_peak, "int8_tops_measured": int8_peak, "int8_peak_how": int8_how,
               "durations": "per-kernel: CUDA events around every launch on the launching stream, separate eager pass of "
                            f"{leg['prof_steps']} steps (shares); fused c2 step: in-graph device timeline (%globaltimer stamps, "
                            "rcn_cuda_timeline_read) + the timed region itself",
               "whole_step": whole, "kernels": kernels})
    return rl


def _teardown_group(ctx):
    """destroy_process_group() on every rank; it was seen to block on this stack (torch 2.11 / NCCL 2.28) after NCCL work
    had been captured into a CUDA graph, so it runs under a watchdog: if it has not returned after 20 s the process leaves
    without it (every collective has completed at the barrier before)."""
    if ctx.world == 1:
        return
    ctx.torch.cuda.synchronize()
    ctx.dist.barrier()
    done = threading.Event()

    def destroy():
        try:
            ctx.dist.destroy_process_group()
        finally:
            done.set()

    th = threading.Thread(target=destroy, daemon=True)
    th.start()
    if not done.wait(20.0):
        print(f"[bench] rank {ctx.rank}: destroy_process_group() did not return within 20 s; leaving without it", file=sys.stderr, flush=True)
        ctx.hung_teardown = True


def _bind_near_gpu(local_rank):
    """Run this rank's host threads on the CPUs NVML names as closest to its GPU (same socket / NUMA node): launches,
    doorbells and the pinned buffers this process first touches then stay local to the GPU's PCIe root.  Measured need: on
    two-socket boxes the device-resident K = 20 region was bimodal per PROCESS (435 vs 575 us) depending on where the
    scheduler had put it.  Returns (description, original affinity) -- the CPU baseline leg restores the original set."""
    try:
        orig = os.sched_getaffinity(0)
    except (AttributeError, OSError):
        return "unchanged (no sched_getaffinity)", None
    if os.environ.get("RCN_BENCH_AFFINITY", "1") == "0":
        return "unchanged (RCN_BENCH_AFFINITY=0)", orig
    try:
        import pynvml
        pynvml.nvmlInit()
        idx = local_rank
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if local_rank < len(ids) and ids[local_rank].isdigit():
                idx = int(ids[local_rank])
        h = pynvml.nvmlDeviceGetHandleByIndex(idx)
        n_words = (max(orig | {os.cpu_count() or 1}) + 64) // 64
        words = pynvml.nvmlDeviceGetCpuAffinity(h, n_words)
        ideal = {64 * w + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1}
        want = ideal & orig
        if not want or want == orig:
            return f"unchanged ({len(orig)} cpus; NVML ideal set covers them all or none)", orig
        os.sched_setaffinity(0, want)
        return f"NVML ideal CPUs of the GPU ({len(want)} of {len(orig)} cpus)", orig
    except Exception as e:  # noqa: BLE001 -- affinity is an optimisation, never a failure
        return f"unchanged ({type(e).__name__})", orig


def run_gpu(args, wl, rank, world, local_rank):
    affinity, orig_affinity = _bind_near_gpu(local_rank)
    import torch
    import torch.distributed as dist

    torch.cuda.set_device(local_rank)
    ctx = Ctx()
    ctx.torch, ctx.dist, ctx.rank, ctx.world, ctx.local_rank = torch, dist, rank, world, local_rank
    ctx.dev = torch.device("cuda", local_rank)
    ctx.hung_teardown = False
    if world > 1:
        dist.init_process_group("nccl", device_id=ctx.dev)

    # ---- main leg: BASELINE configs[1] (or --workload), per-GPU batch fixed (weak scaling) --------------------------------
    dump = args.dump_outputs is not None
    main = run_leg(ctx, args.workload, wl, wl["batch"], args.steps, args.warmup, args.exchange, main=True,
                   steps_per_graph=args.steps_per_graph, no_graph=args.no_graph, host_alloc=args.host_alloc, dump=dump)
    # ---- extra legs in the same invocation: c3 (STRONG scaling: global batch 4096 split over the ranks, SURVEY 8e) and c5
    # (weak, NCCL all-reduce of the 268.8 MB gradient buffer at N > 1); every leg times --steps steps ---------------------
    legs = {}
    if args.workload == "c2" and not args.no_extra:
        for key in [k for k in args.extra.split(",") if k]:
            w2 = WORKLOADS[key]
            if key == "c4":
                legs[key] = run_features_leg(ctx, key, w2, w2["batch"], args.steps, dump=dump)
                continue
            if key == "c3":
                if w2["batch"] % world:
                    continue
                B2, ex2, scaling = w2["batch"] // world, "auto", "strong"
            else:
                B2, ex2, scaling = w2["batch"], ("nccl" if world > 1 else "auto"), "weak"
            try:
                leg = run_leg(ctx, key, w2, B2, args.steps, min(args.warmup, 3), ex2, main=False, steps_per_graph=4, dump=dump)
                leg["scaling"] = scaling
                legs[key] = leg
            except Exception as e:  # noqa: BLE001  -- an extra leg must never cost the main line
                if world > 1:
                    raise
                legs[key] = {"error": f"{type(e).__name__}: {e}"}
                print(f"[bench] extra leg {key} failed: {e}", file=sys.stderr, flush=True)

    _teardown_group(ctx)
    if rank != 0:
        sys.stdout.flush(); sys.stderr.flush()
        if ctx.hung_teardown:
            os._exit(0)
        return

    print("[bench] rank 0: collective phases done", file=sys.stderr, flush=True)
    if dump:
        os.makedirs(args.dump_outputs, exist_ok=True)
    for key, leg in [(args.workload, main)] + list(legs.items()):
        for name, a in (leg.pop("_outputs", None) or {}).items():
            np.save(os.path.join(args.dump_outputs, f"{key}_{name}.npy"), a)
    pk = peaks()
    fp64_peak = measure_fp64_peak(torch, ctx.dev)
    int8_peak, int8_how = measure_int8_peak(torch, ctx.dev)
    if int8_peak is None:
        int8_how = int8_how + "; FALLBACK: 2 x the measured bf16 cuBLAS figure of MEASURED_PEAKS.json"
        int8_peak = 2.0 * (pk["bf16_tflops"] or 1590.0)
    tpath = os.path.join(ROOT, "profiles", "traffic.json")   # dram bytes per launch from the committed `ncu --set full` capture
    traffic_all = json.load(open(tpath)) if os.path.exists(tpath) else {}
    roofline = leg_roofline(main, pk, fp64_peak, int8_peak, int8_how, traffic_all, args.workload)

    # ---- data-parallel parity: the 3 fixed steps again on ONE GPU and through the oracle ------------------------------------
    parity = None
    if main["parity"]:
        import oracle as O
        from mercer_research_b200 import RCN
        pr = main["parity"]
        single = RCN(wl["classes"], wl["cfg"], wl["ff"], device=local_rank)
        single.load_weights_and_bias(main["shapes"][0][1])
        single.set_params(pr["_p0"])
        single.scale_set = pr["_scale"]
        net = O.Net(main["shapes"])
        p_or = pr["_p0"].copy()
        mean, sd = pr["_scale"]
        for k in (0, 1, 2, 0, 1, 2):                        # the 3-chunk epoch walked twice (chunks_exact + wrap, rcn.rs:144-149)
            single.train_batch_images(pr["_images"][k], pr["_labels"][k], ETA)
            X = O.standardise(O.features_u8(wl["cfg"], pr["_images"][k]), mean, sd)
            p_or, _ = net.train_batch(p_or, X, np.eye(wl["classes"])[pr["_labels"][k]], ETA, n_threads=os.cpu_count() or 1)
        p_single = single.get_params()
        single.close()

        def max_rel(a, b):
            return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300)))
        parity = {"steps": pr["steps"], "global_batch": pr["global_batch"], "path": pr["path"], "replicas_bit_identical": pr["replicas_bit_identical"],
                  "max_rel_vs_single_gpu": max_rel(pr["_dp_params"], p_single), "max_rel_vs_oracle": max_rel(pr["_dp_params"], p_or),
                  "single_gpu_max_rel_vs_oracle": max_rel(p_single, p_or), "tolerance": 1e-9,
                  "what": "parameters after 6 SGD steps from fixed parameters on fixed global batches (rcn.rs:144-149,190-222), "
                          "element-wise relative; oracle = C++ restatement (parity unpinned by the reference's own tests)"}

    print("[bench] rank 0: cpu baseline", file=sys.stderr, flush=True)
    # ---- CPU baseline on this box's host cores (bounded sample, ~10-20 s) ------------------------------------------
    Bs = cpu_sample_batch(wl, os.cpu_count() or 1)
    if orig_affinity:
        try:
            os.sched_setaffinity(0, orig_affinity)   # the CPU baseline gets every host core
        except OSError:
            pass
    cpu_ips, cpu_ms, cpu_done, cores, Bs = cpu_train_steps(wl, steps=10 ** 6, warmup=2, max_seconds=12.0, batch=Bs)
    # BASELINE.json configs[0] (the reference's own CPU-runnable case: the same network at batch 32), ~3 s more
    c1_ips, _, c1_done, _, _ = cpu_train_steps(WORKLOADS["c1"], steps=10 ** 6, warmup=2, max_seconds=3.0)

    B, H, W = main["B"], wl["H"], wl["W"]
    workloads = {}
    for key, leg in legs.items():
        if "error" in leg:
            workloads[key] = leg
            continue
        if "_nbytes" in leg:     # feature-stage-only leg (c4)
            nbytes, prof, psteps = leg.pop("_nbytes"), leg.pop("_prof"), leg.pop("_prof_steps")
            gbs = nbytes / (leg["ms_per_step"] * 1e-3) / 1e9
            tot = sum(v["total_ms"] for v in prof.values()) or 1.0
            tw = traffic_all.get(key, {}) or {}   # dram bytes of one call: per-launch ncu figures x launches per call
            parts = [tw[k] * v["launches"] / psteps for k, v in prof.items() if isinstance(tw.get(k), (int, float))]
            leg["roofline"] = {"kernel": max(prof, key=lambda k: prof[k]["total_ms"]) if prof else None, "bound": "hbm", "achieved": gbs,
                               "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": gbs / pk["hbm_gbs"],
                               "traffic": float(sum(parts)) if parts else None, "peak_source": pk["source"],
                               "achieved_is": "algorithmic bytes (H*W u8 read + L*8 f64 features written per image, SURVEY 8d) / duration of one call",
                               "kernels": {k: {"launches_per_step": v["launches"] / psteps, "avg_us": v["total_ms"] / v["launches"] * 1e3,
                                               "share": round(v["total_ms"] / tot, 4)} for k, v in prof.items()}}
            workloads[key] = leg
            continue
        w2 = leg["wl"]
        rl2 = leg_roofline(leg, pk, fp64_peak, int8_peak, int8_how, traffic_all, key)
        workloads[key] = {
            "workload": w2["desc"], "value": leg["value"], "unit": "images/s", "ms_per_step": leg["ms_step"], "steps": leg["steps"],
            "scaling": leg["scaling"], "batch_per_gpu": leg["B"], "global_batch": leg["B"] * world, "params": leg["n_params"],
            "exchange": ("none (1 GPU)" if world == 1 else ("NVLink peer-memory exchange kernel" if leg["p2p"] else "NCCL all-reduce (eager)")),
            "cuda_graph": leg["graph"], "steps_per_graph": leg["spg"], "gpu_launches": leg["launches"],
            "e2e": {"value": leg["e2e_value"], "unit": "images/s", "ms_per_step": leg["e2e_ms_step"],
                    "h2d_bytes_per_step": leg["h2d"], "d2h_bytes_per_step": leg["d2h"]},
            "clocks": leg["clocks"], "roofline": rl2,
        }

    line = {
        "metric": "training images/sec", "value": main["value"], "unit": "images/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": main["ms_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": wl["desc"], "batch_per_gpu": B, "batch_per_step": B, "global_batch": B * world, "pixels": "u8", "eta": ETA,
                   "params": main["n_params"], "parallelism": f"dp{world}",
                   "l2_policy": f"inputs rotate over {main['n_batches']} resident batches = {main['n_batches'] * B * H * W / 2 ** 20:.0f} MiB > 126 MB L2 "
                                "(each step's kernel A asks L2 for the NEXT step's images ahead of time; every image still comes from HBM once per step)",
                   "step": main["step_desc"], "cuda_graph": main["graph"], "steps_per_graph": main["spg"],
                   "host_cpu_affinity": affinity,
                   # the W requested warm-up steps plus ~0.3 s of the same load so that clocks have ramped
                   "warmup_steps_run": main["n_warm"]},
        "clocks": main["clocks"],
        "e2e": {"value": main["e2e_value"], "unit": "images/s", "h2d_bytes_per_step": main["h2d"], "d2h_bytes_per_step": main["d2h"],
                "ms_per_step": main["e2e_ms_step"], "host_buffers": main["host_alloc"],
                # PCIe bytes per second this rank moved inside the timed region (the link: 43.6-55 GB/s for copy-engine
                # transfers of 0.8-64 MB, profiles/r2_pcie_dma.json; 38 GB/s for SM-issued zero-copy reads)
                "h2d_GBps_per_gpu": main["h2d"] / (main["e2e_ms_step"] * 1e-3) * 1e-9,
                "api": "rcn_cuda_train_epoch_host (chunks_exact loop over a pinned host dataset: the copy engine streams the chunks "
                       "into a device ring ahead of the steps, kernel A waits on an arrival counter, up to 40 steps per CUDA graph launch, "
                       "per-step cost/hits written back to host memory; RCN_CUDA_HOST_COPY=pull = round 1's SM-issued zero-copy loads)"},
        "gpu_launches": int(main["launches"]),
        "roofline": roofline,
        "cpu_baseline": {"value": cpu_ips, "unit": "images/s", "cores": cores, "kind": "port",
                         "sample": f"{cpu_done} steps of batch {Bs} (features+fwd+bwd+SGD) on {cores} host threads, "
                                   "oracle/rcn_oracle.cpp (C++ restatement of rcn's CPU path, not rustc output)",
                         "configs0_batch32": {"value": c1_ips, "unit": "images/s", "cores": cores,
                                              "sample": f"{c1_done} steps of batch 32, same network, same {cores} host threads"}},
        "parity_note": "parity unpinned: the oracle is a C++ restatement of rcn (no Rust toolchain); only kernel.rs:400-441 pin it",
    }
    if parity:
        line["parity"] = parity
    if workloads:
        line["workloads"] = workloads
    emit_result(line)
    sys.stdout.flush(); sys.stderr.flush()
    if ctx.hung_teardown:
        os._exit(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000, help="timed steps of every workload")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--steps-per-graph", type=int, default=5,
                    help="consecutive steps captured into one CUDA graph (the timed region replays it steps/this times). Small graphs on "
                         "purpose: the timed region starts on an idle GPU, a graph's launch latency grows with its node count (measured: "
                         "~38 us for 20 steps, ~12 us for 5) and only the FIRST launch is exposed -- the host enqueues the others while "
                         "the GPU works. (A 2-step head graph followed by 9-step graphs was measured WORSE at K = 20: 22-31 us/step, the "
                         "head is too short to cover the host's launch of the first long graph.)")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel eagerly instead of replaying a CUDA graph")
    ap.add_argument("--host-alloc", default="pinned", choices=["pinned", "wc"],
                    help="e2e leg: ordinary pinned host memory (default) or write-combined pinned memory (experiment)")
    ap.add_argument("--exchange", default="auto", choices=["auto", "p2p", "nccl"],
                    help="multi-GPU gradient exchange: fused NVLink peer-memory kernel, NCCL all-reduce, or by size")
    ap.add_argument("--extra", default="c3,c4,c5", help="extra workloads measured after the main one in the same run (parsed.workloads)")
    ap.add_argument("--no-extra", action="store_true", help="main workload only")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what each workload's timed paths computed in their last step to "
                         "DIR/<workload>_<name>.npy (float64): params, grads and batch_stats ([cost, hits]) of the device-"
                         "resident leg, e2e_params and e2e_batch_stats of the host-buffer leg, features of the feature-stage "
                         "workload; arrays of more than 2^19 elements as a fixed, seeded sample. The same arguments give the "
                         "same inputs, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl b200)")
    # stdout must carry exactly ONE JSON line: route everything else that writes to fd 1 (e.g. NCCL's version banner)
    # to stderr and keep the real stdout for the result line.
    global _RESULT_FD
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, wl, rank, world)
        return
    if world != args.gpus and rank == 0:
        print(f"[bench] note: --gpus {args.gpus} but WORLD_SIZE={world}; using WORLD_SIZE", file=sys.stderr)
    run_gpu(args, wl, rank, world, local_rank)


if __name__ == "__main__":
    main()
