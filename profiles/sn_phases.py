"""Where kernel A (smallnet_fwd_bwd_kernel) spends its time on config c2: per-CTA clock64() stamps at the phase boundaries
(library built by profiles/build_phases.sh with -DRCN_SN_PHASES).  Usage on the GPU box:
    profiles/build_phases.sh && RCN_CUDA_LIB=profiles/_build/librcn_cuda_phases.so python profiles/sn_phases.py [B] [--json PATH]
(--json: also write the per-phase means of the front end and of the whole kernel, in ns, to PATH.)
"""
import json
import ctypes as C
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mercer_research_b200 import RCN, Padding, Pooling, RCNLayer  # noqa: E402

NAMES = ["image loads (bulk) + zero frames", "transpose", "conv+pool stages", "layer-0 DMMA (K split over 16 warps)",
         "partial sums + narrow forward", "output delta + backward chain + writes", "small-parameter partials"]


def main(B=1024, json_path=None):
    dev = torch.device("cuda", 0)
    model = RCN(10, [RCNLayer.Convolve2D(Padding.Same), RCNLayer.Pool2D(Pooling.Max)], [30])
    model.load_weights_and_bias(784)
    model.set_params(np.random.default_rng(1).standard_normal(model.n_params))
    imgs = torch.randint(0, 256, (B, 28, 28), dtype=torch.uint8, device=dev)
    labels = (torch.arange(B, device=dev) % 10).to(torch.int64)
    model.gen_scales(model.flatten_feature_set(imgs))
    for _ in range(5):
        model.train_batch_images(imgs, labels, 3.0)
    torch.cuda.synchronize()
    full = np.zeros((1024, 32), dtype=np.int64)
    rc = model._lib.rcn_cuda_debug_sn_phases(full.ctypes.data_as(C.c_void_p))
    assert rc == 0
    out = full[:, :8]
    n = (B + 7) // 8
    d = np.diff(out[:n], axis=1) / 1.965   # ns at 1965 MHz
    sub = full[:n, [0, 8, 9, 10, 11, 12, 1]]
    ds = np.diff(sub, axis=1) / 1.965
    print("  head of kernel A (thread 0): " + ", ".join(f"{nm} {ds[:, k].mean():.0f}" for k, nm in enumerate(
        ["bulk-load issue + labels", "W fragment loads issued", "small params staged", "zero frames", "barrier", "mbarrier wait"])))
    tail = full[:n, [4, 16, 17, 5, 18, 19, 20, 21, 6, 7]]
    dt = np.diff(tail, axis=1) / 1.965
    print("  tail of kernel A (thread 0): " + ", ".join(f"{nm} {dt[:, k].mean():.0f}" for k, nm in enumerate(
        ["partial-sum tree", "bias + sigmoid", "narrow layers", "activations out", "delta + statistics", "backward chain", "deltas out",
         "block barrier", "gradient partials"])))
    print(f"kernel A, B={B}, {n} CTAs; per-phase ns (mean / min / max over CTAs)")
    for k, name in enumerate(NAMES):
        print(f"  {name:45s} {d[:, k].mean():8.0f} {d[:, k].min():8.0f} {d[:, k].max():8.0f}")
    tot = (out[:n, 7] - out[:n, 0]) / 1.965
    print(f"  {'thread-0 lifetime':45s} {tot.mean():8.0f} {tot.min():8.0f} {tot.max():8.0f}")
    if json_path:
        rec = {"B": B, "ctas": n, "clock_mhz_assumed": 1965,
               "head_ns": {nm: float(ds[:, k].mean()) for k, nm in enumerate(
                   ["bulk-load issue + labels", "W fragment loads issued", "small params staged", "zero frames", "barrier",
                    "mbarrier wait"])},
               "phases_ns": {nm: float(d[:, k].mean()) for k, nm in enumerate(NAMES)},
               "thread0_lifetime_ns": float(tot.mean())}
        with open(json_path, "w") as f:
            json.dump(rec, f, indent=1)


def timeline(B=1024, steps=40):
    """Replays ONE captured CUDA graph of the c2 step (kernel A, kernel B, sgd_update) `steps` times over a device-resident
    dataset and prints, from %globaltimer stamps inside the kernels, each kernel's span and the gaps between them."""
    dev = torch.device("cuda", 0)
    model = RCN(10, [RCNLayer.Convolve2D(Padding.Same), RCNLayer.Pool2D(Pooling.Max)], [30])
    model.load_weights_and_bias(784)
    model.set_params(np.random.default_rng(1).standard_normal(model.n_params) * 0.1)
    N = B * 64
    imgs = torch.randint(0, 256, (N, 28, 28), dtype=torch.uint8, device=dev)
    labels = (torch.arange(N, device=dev) % 10).to(torch.int64)
    model.gen_scales(model.flatten_feature_set(imgs[:4096]))
    model.epoch_bind(imgs, labels, B)
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        model.set_stream(side.cuda_stream)
        for _ in range(3):
            model.epoch_step(3.0)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        model.set_stream(torch.cuda.current_stream().cuda_stream)
        for _ in range(8):      # several steps per graph: the host's launch cost must not be what is measured
            model.epoch_step(3.0)
    for _ in range(5):
        g.replay()
    torch.cuda.synchronize()
    model.timeline_enable(True)          # bumps the allocation generation: capture again with the timeline pointer baked in
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        model.set_stream(torch.cuda.current_stream().cuda_stream)
        for _ in range(8):
            model.epoch_step(3.0)
    for _ in range(max(1, steps // 8)):
        g.replay()
    torch.cuda.synchronize()
    t0, t1, n_l = model.timeline_read()
    n = int(min(n_l[0], n_l[1], 56))
    order = [(int(n_l[0]) - n + j) % 64 for j in range(n)]          # oldest -> newest of the last n launches
    A0, A1 = t0[0, order].astype(np.int64), t1[0, order].astype(np.int64)
    orderb = [(int(n_l[1]) - n + j) % 64 for j in range(n)]
    B0, B1 = t0[1, orderb].astype(np.int64), t1[1, orderb].astype(np.int64)
    rows = [("kernel A  first CTA start -> last CTA end", (A1 - A0)), ("gap A -> B", (B0 - A1)), ("kernel B  span", (B1 - B0)),
            ("gap B(+update) -> next kernel A", (A0[1:] - B1[:-1])), ("step period (A start to A start)", np.diff(A0))]
    print(f"graph-replayed c2 step, B={B}: {n} steps recorded; ns (median / min / max)")
    for name, v in rows:
        print(f"  {name:45s} {np.median(v):8.0f} {v.min():8.0f} {v.max():8.0f}")


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "timeline":
        timeline(int(sys.argv[2]) if len(sys.argv) > 2 else 1024)
        sys.exit(0)

    args = sys.argv[1:]
    jp = None
    if "--json" in args:
        k = args.index("--json")
        jp = args[k + 1]
        del args[k:k + 2]
    main(int(args[0]) if args else 1024, jp)
