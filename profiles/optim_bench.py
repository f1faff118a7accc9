"""Times the optimizer step of the convolutional network handle (ConvNet.set_optimizer: momentum SGD, AdamW) against the
plain SGD update and against torch's own optimizers, on one GPU, with CUDA events only.

  apply     ConvNet.apply_gradients alone on a network whose dense part is far larger than the 126 MB L2: Conv(8)/Pool on
            128x128x1 images -> a 32768-feature x 2048 dense layer -> 10 classes, 67.2 M parameters.  The gradient buffer
            is a bound torch tensor of random values.  Bytes per parameter and step: plain SGD 24 (read p, g; write p),
            momentum SGD 40 (+ read / write v), AdamW 56 (+ read / write m and v).
  torch     torch.optim.SGD (momentum 0 and 0.9) and AdamW on one flat f64 CUDA tensor of the same size, foreach and fused,
            in the same process, charged the same bytes.
  steps     the replayed epoch_step (one captured graph) of the MNIST and config-3 shapes of cnn_bench.py with plain SGD,
            momentum SGD and AdamW, alternated three times (medians), on resident data twice the L2; and the optimizer
            kernel's time per step from the launch profiler in a separate pass of eager steps.

usage: python profiles/optim_bench.py [--out DIR]   -> DIR/optim_bench_b200.json"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from cnn_bench import L2_BYTES, SHAPES, gpu_info, m, timed  # noqa: E402
from mercer_research_b200 import _lib  # noqa: E402

BYTES = {"plain": 24, "momentum": 40, "adamw": 56}
OPTS = {"plain": lambda: m.SGD(), "momentum": lambda: m.SGD(momentum=0.9), "adamw": lambda: m.AdamW()}
ETA = {"plain": 0.05, "momentum": 0.005, "adamw": 1e-4}


def run_apply():
    net = m.ConvNet((128, 128, 1), [m.Conv(8), m.Pool(m.Pooling.Max, m.Padding.Same)], [2048], 10)
    n = net.n_params
    g = torch.randn(n, dtype=torch.float64, device="cuda")
    net.bind_gradient_buffer(g)
    net.set_stream(torch.cuda.current_stream().cuda_stream)
    res = {"n_params": n, "feature_len": net.feature_len, "library": {}, "torch": {}}
    for name in ("plain", "momentum", "adamw"):
        runs = []
        net.set_optimizer(OPTS[name]())
        for _ in range(3):
            runs.append(timed(lambda: net.apply_gradients(ETA[name], 64))[0])
        ms = float(np.median(runs))
        res["library"][name] = dict(median_ms=ms, runs_ms=runs, bytes_per_param=BYTES[name],
                                    bytes_per_s=BYTES[name] * n / (ms * 1e-3))
        _lib.profile_enable(True)
        for _ in range(5):
            net.apply_gradients(ETA[name], 64)
        rep = _lib.profile_report()
        _lib.profile_enable(False)
        res["library"][name]["kernels"] = {k: v["total_ms"] / 5 for k, v in rep.items()}
        print(f"apply {name}: {ms * 1e3:.1f} us, {BYTES[name] * n / (ms * 1e-3) / 1e9:.0f} GB/s", flush=True)
    net.close()
    del g
    torch.cuda.empty_cache()
    p = torch.zeros(n, dtype=torch.float64, device="cuda", requires_grad=True)
    p.grad = torch.randn(n, dtype=torch.float64, device="cuda")
    makers = {
        "plain": lambda **kw: torch.optim.SGD([p], lr=ETA["plain"], **kw),
        "momentum": lambda **kw: torch.optim.SGD([p], lr=ETA["momentum"], momentum=0.9, **kw),
        "adamw": lambda **kw: torch.optim.AdamW([p], lr=ETA["adamw"], **kw),
    }
    for name, make in makers.items():
        for impl in ("foreach", "fused"):
            try:
                opt = make(**{impl: True})
                runs = [timed(opt.step)[0] for _ in range(3)]
            except Exception as e:   # an implementation torch does not offer for f64 is reported, not timed
                res["torch"][f"{name}_{impl}"] = {"error": str(e)}
                continue
            ms = float(np.median(runs))
            res["torch"][f"{name}_{impl}"] = dict(median_ms=ms, runs_ms=runs, bytes_per_s=BYTES[name] * n / (ms * 1e-3))
            print(f"torch {name} {impl}: {ms * 1e3:.1f} us, {BYTES[name] * n / (ms * 1e-3) / 1e9:.0f} GB/s", flush=True)
            del opt
    del p
    torch.cuda.empty_cache()
    return res


def run_steps(shape):
    c = SHAPES[shape]
    B = c["B"]
    per_batch = B * int(np.prod(c["shape"])) * (1 if c["u8"] else 8)
    n_batches = max(2, -(-2 * L2_BYTES // per_batch))
    gen = torch.Generator(device="cuda"); gen.manual_seed(2)
    if c["u8"]:
        data = torch.randint(0, 256, (n_batches * B,) + c["shape"][:2], dtype=torch.uint8, device="cuda", generator=gen)
    else:
        data = torch.randn((n_batches * B,) + c["shape"], dtype=torch.float64, device="cuda", generator=gen)
    labels = torch.randint(0, 10, (n_batches * B,), device="cuda", generator=gen)
    perm = torch.randperm(n_batches * B, device="cuda", generator=gen)
    nets, graphs = {}, {}
    for name in OPTS:
        net = m.ConvNet(c["shape"], c["layers"], c["ff"], 10)
        net.init_params(np.random.default_rng(1))
        net.set_optimizer(OPTS[name]())
        net.epoch_bind(data, labels, B, perm)
        net.epoch_accumulate()
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            net.set_stream(torch.cuda.current_stream().cuda_stream)
            net.epoch_step(ETA[name])
        net.set_stream(torch.cuda.current_stream().cuda_stream)
        nets[name], graphs[name] = net, graph
    g0 = _lib.allocation_generation()
    runs = {name: [] for name in OPTS}
    for _ in range(3):
        for name in OPTS:
            runs[name].append(timed(graphs[name].replay)[0])
    assert _lib.allocation_generation() == g0, "a library buffer moved under a captured step"
    res = {"batch": B, "n_params": nets["plain"].n_params}
    for name, net in nets.items():
        torch.cuda.synchronize()
        _lib.profile_enable(True)
        for _ in range(5):
            net.epoch_step(ETA[name])
        rep = _lib.profile_report()
        _lib.profile_enable(False)
        upd = {k: v["total_ms"] / 5 for k, v in rep.items() if k.startswith(("optim_", "sgd_update_kernel"))}
        total = sum(v["total_ms"] for v in rep.values()) / 5
        v = runs[name]
        res[name] = dict(graph_step_median_ms=float(np.median(v)), runs_ms=v, update_kernels_ms_per_step=upd,
                         update_share_of_kernel_time=sum(upd.values()) / total)
    for name in ("momentum", "adamw"):
        res[name]["over_plain"] = res[name]["graph_step_median_ms"] / res["plain"]["graph_step_median_ms"]
    print(f"{shape}: " + ", ".join(f"{k} {res[k]['graph_step_median_ms']:.3f} ms" for k in OPTS), flush=True)
    for net in nets.values():
        net.close()
    del graphs, data, labels, perm
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=".", help="directory that receives optim_bench_b200.json")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    out = dict(gpu_info(), time=time.strftime("%Y-%m-%d %H:%M:%S"), torch=torch.__version__)
    out["apply"] = run_apply()
    out["steps"] = {s: run_steps(s) for s in ("mnist", "cifar")}
    with open(os.path.join(args.out, "optim_bench_b200.json"), "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
