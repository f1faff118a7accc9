"""Times one training step of the convolutional network handle (mercer_research_b200.ConvNet) on device-resident data
larger than the 126 MB L2, for an MNIST-shaped network and the two shapes of BASELINE.json configs 3 and 4:

  mnist   28x28 u8,    Conv(8)/Pool                                -> 1568-30-10,   B = 1024
  cifar   32x32x3 f64, Conv(32)/Pool/Conv(64)/Pool/Conv(128)/Pool -> 2048-256-10, B = 4096
  wide    64x64 u8,    Conv(64)/Conv(64)/Pool/Conv(128)/Pool       -> 32768-32-10,  B = 256

Two ways to drive the same steps over the same data, alternated three times (median and spread of each): the eager loop,
one train_batch_images call per host-sliced minibatch (step_ms / images_per_s), and the epoch mode, the data bound with a
random perm and one captured epoch_step replayed per step (epoch_graph).  The epoch staging kernel's time per step comes
from the library's launch profiler, its bytes from the shapes (images read and written, the f64 copy of u8 images, perm
and labels); a torch device-to-device copy moving the same number of bytes, rotated through the dataset so it comes from
HBM, is timed in the same call.
Per shape also: per-kernel time shares of the eager step from the library's
launch profiler (a separate pass), the conv engine each layer's forward / backward-data / backward-weight took, and for
the GEMM-shaped kernels the achieved rate against the DGEMM peak (torch.matmul f64) or the int8 tensor-core peak
(torch._int_mm) measured in the same call.  The tcgen05 conv kernels run 15 int8 plane products per f64 product, so their
int8 rate is 15 x 2MNK over the kernel time.
Heads (run_heads, also alone with --heads-only -> cnn_heads_b200.json): per shape the sigmoid / quadratic head and the softmax
cross-entropy head (ConvNet(head=...)) on the same parameters and data, alternated three times in the same process: the eager
step and the replayed epoch step of each; and the per-step time of softmax_xent_head_kernel (and of every other kernel) from
the launch profiler in a separate pass.  usage: python profiles/cnn_bench.py [--out DIR] [--heads-only]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import mercer_research_b200 as m  # noqa: E402
from mercer_research_b200 import _lib, ext  # noqa: E402

P, Q = m.Padding, m.Pooling
SHAPES = {
    "mnist": dict(shape=(28, 28, 1), u8=True, B=1024, ff=[30], layers=[m.Conv(8), m.Pool(Q.Max, P.Same)]),
    "cifar": dict(shape=(32, 32, 3), u8=False, B=4096, ff=[256],
                  layers=[m.Conv(32), m.Pool(Q.Max, P.Same), m.Conv(64), m.Pool(Q.Max, P.Same), m.Conv(128), m.Pool(Q.Max, P.Same)]),
    "wide": dict(shape=(64, 64, 1), u8=True, B=256, ff=[32],
                 layers=[m.Conv(64), m.Conv(64), m.Pool(Q.Max, P.Same), m.Conv(128), m.Pool(Q.Max, P.Same)]),
}
L2_BYTES = 126 << 20


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()
        name, power = [s.strip() for s in out[0].split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as e:
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": "unknown", "error": str(e)}


def timed(fn, min_s=0.3):
    """ms per call of fn, over >= min_s of back-to-back calls between two CUDA events."""
    fn(); torch.cuda.synchronize()
    n = 1
    while True:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record(); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if ms >= min_s * 1e3:
            return ms / n, n
        n = max(n * 2, int(n * min_s * 1e3 / max(ms, 1e-3)) + 1)


def peaks():
    a = torch.randn(8192, 8192, dtype=torch.float64, device="cuda")
    ms, _ = timed(lambda: a @ a)
    dgemm = 2 * 8192 ** 3 / (ms * 1e-3)
    i = torch.randint(-128, 127, (8192, 8192), dtype=torch.int8, device="cuda")
    ms, _ = timed(lambda: torch._int_mm(i, i))
    int8 = 2 * 8192 ** 3 / (ms * 1e-3)
    return {"dgemm_flops": dgemm, "int8_ops": int8}


def layer_geometry(net):
    """per conv layer: (index, B-free GEMM sizes) -- pixels per sample, Co, K = kh*kw*Ci, input map."""
    out, (h, w, c) = [], net.input_shape
    for i, l in enumerate(net.layers):
        if isinstance(l, m.Conv):
            ho, wo, co = net.layer_shape(i)
            out.append(dict(layer=i, in_hwc=(h, w, c), pix=ho * wo, Co=co, K=l.kh * l.kw * c))
        h, w, c = net.layer_shape(i)
    return out


def engines(net, B, geo):
    """The kernels each conv layer's three passes launch (the handle calls the same launch functions; a first layer on u8
    images runs the u8 instantiation of the direct kernel where this f64 op reports the direct kernel)."""
    res = []
    for g in geo:
        l = net.layers[g["layer"]]
        h, w, c = g["in_hwc"]
        x = torch.randn(B, h, w, c, dtype=torch.float64, device="cuda")
        wt = torch.randn(l.out_channels, l.kh, l.kw, c, dtype=torch.float64, device="cuda")
        row = {"layer": g["layer"]}
        for name, fn in (("forward", lambda: ext.conv2d_forward(x, wt, None, l.padding, ext.Activation.ReLU)),
                         ("backward_weight", lambda: ext.conv2d_backward_weight(x, y, l.kh, l.kw, l.padding)),
                         ("backward_data", lambda: ext.conv2d_backward_data(y, wt, (h, w), l.padding))):
            if name == "forward":
                y = fn()
            torch.cuda.synchronize()
            _lib.profile_enable(True)
            fn()
            rep = _lib.profile_report()
            _lib.profile_enable(False)
            row[name] = sorted(k for k in rep if "igemm" in k or "direct" in k)
        res.append(row)
        del x, wt, y
    return res


def run_shape(name, cfg, pk):
    c = cfg
    net = m.ConvNet(c["shape"], c["layers"], c["ff"], 10)
    net.init_params(np.random.default_rng(1))
    B = c["B"]
    per_batch = B * int(np.prod(c["shape"])) * (1 if c["u8"] else 8)
    n_batches = max(2, -(-2 * L2_BYTES // per_batch))
    g = torch.Generator(device="cuda"); g.manual_seed(2)
    if c["u8"]:
        data = torch.randint(0, 256, (n_batches, B) + c["shape"][:2], dtype=torch.uint8, device="cuda", generator=g)
    else:
        data = torch.randn((n_batches, B) + c["shape"], dtype=torch.float64, device="cuda", generator=g)
    labels = torch.randint(0, 10, (n_batches, B), device="cuda", generator=g)
    k = [0]

    def step():
        i = k[0] % n_batches
        k[0] += 1
        net.train_batch_images(data[i], labels[i], 0.05)

    for _ in range(3):
        step()
    torch.cuda.synchronize()
    # the same data bound for epoch mode under a random perm; one captured step replayed per step
    flat, flat_y = data.view((n_batches * B,) + data.shape[2:]), labels.view(-1)
    perm = torch.randperm(n_batches * B, device="cuda", generator=g)
    net.epoch_bind(flat, flat_y, B, perm)
    net.epoch_accumulate()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        net.set_stream(torch.cuda.current_stream().cuda_stream)
        net.epoch_step(0.05)
    net.set_stream(torch.cuda.current_stream().cuda_stream)
    gen = _lib.allocation_generation()
    eager_runs, graph_runs = [], []
    for _ in range(3):
        eager_runs.append(timed(step))
        graph_runs.append(timed(graph.replay))
    assert _lib.allocation_generation() == gen, "a library buffer moved under the captured step"
    ms = float(np.median([r[0] for r in eager_runs]))
    n = int(sum(r[1] for r in eager_runs))
    g_ms = float(np.median([r[0] for r in graph_runs]))

    def spread(runs):
        v = [r[0] for r in runs]
        return dict(median_ms=float(np.median(v)), min_ms=min(v), max_ms=max(v), runs_ms=v,
                    spread=(max(v) - min(v)) / float(np.median(v)), steps=[r[1] for r in runs])

    # staging kernel: time per step (event-bracketed launches, eager epoch steps) and bytes moved per step
    img_bytes = int(np.prod(c["shape"])) * (1 if c["u8"] else 8)
    stage_bytes = B * img_bytes * (2 + (8 if c["u8"] else 0)) + B * 8 * 3   # images in/out (+f64), perm, labels in/out
    torch.cuda.synchronize()
    _lib.profile_enable(True)
    for _ in range(20):
        net.epoch_step(0.05)
    rep = _lib.profile_report()
    _lib.profile_enable(False)
    st = [v for kname, v in rep.items() if kname.startswith("cnn_stage_batch_kernel")]
    stage_ms = sum(v["total_ms"] for v in st) / max(1, sum(v["launches"] for v in st))
    raw = data.view(torch.uint8).view(-1)
    half = stage_bytes // 2                                                  # a copy moves 2x its size
    dst = torch.empty(half, dtype=torch.uint8, device="cuda")
    off = [0]

    def copy():
        o = off[0]
        off[0] = (o + half) % (raw.numel() - half)
        dst.copy_(raw[o:o + half])

    copy_ms, _ = timed(copy)
    epoch = dict(graph_step=spread(graph_runs), eager_step=spread(eager_runs), step_ms=g_ms, images_per_s=B / (g_ms * 1e-3),
                 replay_speedup=ms / g_ms, stage_kernel_ms_per_step=stage_ms, stage_bytes_per_step=stage_bytes,
                 stage_bytes_per_s=stage_bytes / (stage_ms * 1e-3), torch_d2d_copy_ms=copy_ms,
                 torch_d2d_copy_bytes_per_s=2 * half / (copy_ms * 1e-3),
                 stage_launches_per_step=sum(v["launches"] for v in st) / 20)
    # profile pass (separate: the event pairs slow the host)
    torch.cuda.synchronize()
    _lib.profile_enable(True)
    for _ in range(5):
        step()
    rep = _lib.profile_report()
    _lib.profile_enable(False)
    total = sum(v["total_ms"] for v in rep.values())
    shares = {kname: {"ms_per_step": v["total_ms"] / 5, "share": v["total_ms"] / total, "launches_per_step": v["launches"] / 5}
              for kname, v in sorted(rep.items(), key=lambda kv: -kv[1]["total_ms"])}
    geo = layer_geometry(net)
    eng = engines(net, B, geo)
    # GEMM-shaped work per step: each layer's pass is charged to the engine its kernel names (the direct kernel is no GEMM)
    first = geo[0]["layer"]
    rates = {}
    for pas in ("forward", "backward_weight", "backward_data"):
        for tc in (False, True):
            f = sum(2 * B * x["pix"] * x["Co"] * x["K"] for x, e in zip(geo, eng)
                    if not (pas == "backward_data" and x["layer"] == first)
                    and any("igemm" in k and ("tcgen05" in k) == tc for k in e[pas]))
            ks = [kn for kn in shares if kn.startswith("conv2d_" + pas) and ("tcgen05" in kn) == tc and "igemm" in kn]
            if not ks or not f:
                continue
            t = sum(shares[kn]["ms_per_step"] for kn in ks) * 1e-3
            r = {"kernels": ks, "ms_per_step": t * 1e3, "f64_flops_per_s": f / t}
            if tc:   # 15 exact int8 plane products per f64 product
                r["int8_ops_per_s"] = 15 * f / t
                r["fraction_of_measured_int8_peak"] = 15 * f / t / pk["int8_ops"]
            else:
                r["fraction_of_measured_dgemm_peak"] = f / t / pk["dgemm_flops"]
            rates[f"conv2d_{pas} ({'tcgen05' if tc else 'DMMA'})"] = r
    res = dict(batch=B, n_batches_resident=n_batches, resident_bytes=n_batches * per_batch, step_ms=ms, timed_steps=n,
               images_per_s=B / (ms * 1e-3), kernel_shares=shares, conv_engines=eng, gemm_rates=rates,
               n_params=net.n_params, feature_len=net.feature_len, epoch_graph=epoch)
    del graph, data, labels, flat, flat_y, perm, raw, dst
    net.close()
    torch.cuda.empty_cache()
    return res


def run_heads(name, cfg):
    """Both heads on the same parameters and resident data: eager and replayed epoch step times, alternated three times."""
    c = cfg
    B = c["B"]
    per_batch = B * int(np.prod(c["shape"])) * (1 if c["u8"] else 8)
    n_batches = max(2, -(-2 * L2_BYTES // per_batch))
    g = torch.Generator(device="cuda"); g.manual_seed(2)
    if c["u8"]:
        data = torch.randint(0, 256, (n_batches, B) + c["shape"][:2], dtype=torch.uint8, device="cuda", generator=g)
    else:
        data = torch.randn((n_batches, B) + c["shape"], dtype=torch.float64, device="cuda", generator=g)
    labels = torch.randint(0, 10, (n_batches, B), device="cuda", generator=g)
    flat, flat_y = data.view((n_batches * B,) + data.shape[2:]), labels.view(-1)
    perm = torch.randperm(n_batches * B, device="cuda", generator=g)
    nets, steps, graphs = {}, {}, {}
    for head in (m.Head.SigmoidQuadratic, m.Head.SoftmaxCrossEntropy):
        net = m.ConvNet(c["shape"], c["layers"], c["ff"], 10, head=head)
        net.init_params(np.random.default_rng(1))
        k = [0]

        def step(net=net, k=k):
            i = k[0] % n_batches
            k[0] += 1
            net.train_batch_images(data[i], labels[i], 0.05)

        for _ in range(3):
            step()
        net.epoch_bind(flat, flat_y, B, perm)
        net.epoch_accumulate()
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            net.set_stream(torch.cuda.current_stream().cuda_stream)
            net.epoch_step(0.05)
        net.set_stream(torch.cuda.current_stream().cuda_stream)
        nets[head.name], steps[head.name], graphs[head.name] = net, step, graph
    gen = _lib.allocation_generation()
    runs = {h: {"eager": [], "graph": []} for h in nets}
    for _ in range(3):
        for h in nets:
            runs[h]["eager"].append(timed(steps[h])[0])
            runs[h]["graph"].append(timed(graphs[h].replay)[0])
    assert _lib.allocation_generation() == gen, "a library buffer moved under a captured step"
    res = {"batch": B}
    for h in nets:
        torch.cuda.synchronize()
        _lib.profile_enable(True)
        for _ in range(5):
            steps[h]()
        rep = _lib.profile_report()
        _lib.profile_enable(False)
        kern = {kn: {"ms_per_step": v["total_ms"] / 5, "launches_per_step": v["launches"] / 5}
                for kn, v in sorted(rep.items(), key=lambda kv: -kv[1]["total_ms"])}
        r = {mode: dict(median_ms=float(np.median(v)), min_ms=min(v), max_ms=max(v), runs_ms=v) for mode, v in runs[h].items()}
        r["kernels"] = kern
        res[h] = r
    s, x = res["SigmoidQuadratic"], res["SoftmaxCrossEntropy"]
    res["softmax_over_sigmoid"] = {mode: x[mode]["median_ms"] / s[mode]["median_ms"] for mode in ("eager", "graph")}
    res["head_kernel_ms_per_step"] = x["kernels"].get("softmax_xent_head_kernel", {}).get("ms_per_step")
    for net in nets.values():
        net.close()
    del graphs, data, labels, flat, flat_y, perm
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=".", help="directory that receives cnn_bench_b200.json")
    ap.add_argument("--heads-only", action="store_true", help="only run_heads, into cnn_heads_b200.json")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    info = gpu_info()
    if args.heads_only:
        out = dict(info, time=time.strftime("%Y-%m-%d %H:%M:%S"), shapes={})
        for name, cfg in SHAPES.items():
            r = out["shapes"][name] = run_heads(name, cfg)
            print(f"{name}: sigmoid eager {r['SigmoidQuadratic']['eager']['median_ms']:.3f} graph "
                  f"{r['SigmoidQuadratic']['graph']['median_ms']:.3f} ms; softmax eager {r['SoftmaxCrossEntropy']['eager']['median_ms']:.3f} "
                  f"graph {r['SoftmaxCrossEntropy']['graph']['median_ms']:.3f} ms; head kernel {r['head_kernel_ms_per_step']} ms",
                  flush=True)
        with open(os.path.join(args.out, "cnn_heads_b200.json"), "w") as f:
            json.dump(out, f, indent=1)
        return
    pk = peaks()
    out = dict(info, measured_peaks=pk, time=time.strftime("%Y-%m-%d %H:%M:%S"), shapes={})
    for name, cfg in SHAPES.items():
        out["shapes"][name] = run_shape(name, cfg, pk)
        r = out["shapes"][name]
        r["heads"] = run_heads(name, cfg)
        e = r["epoch_graph"]
        print(f"{name}: {r['images_per_s']:.0f} images/s ({r['step_ms']:.3f} ms/step, B={r['batch']}); epoch graph "
              f"{e['step_ms']:.3f} ms/step (x{e['replay_speedup']:.2f}); staging {e['stage_kernel_ms_per_step'] * 1e3:.1f} us "
              f"{e['stage_bytes_per_s'] / 1e9:.0f} GB/s, torch copy {e['torch_d2d_copy_bytes_per_s'] / 1e9:.0f} GB/s", flush=True)
    with open(os.path.join(args.out, "cnn_bench_b200.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: v for k, v in out.items() if k != "shapes"}))


if __name__ == "__main__":
    main()
