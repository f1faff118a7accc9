"""Test-set evaluation throughput on the canonical network ([Conv Same, Pool Max], 28x28 u8 images, 784-30-10).

Times, per batch size, with CUDA events after a warm-up of every shape, the median and range over repeats of:
  evaluate_images   RCN.evaluate_images (rcn_cuda_evaluate_images, device-resident cost / accept outputs)
  features+evaluate flatten_feature_set(standardise=True) + evaluate in 16 384-image chunks, as RCN.train_arrays evaluated
                    before evaluate_images existed (one host synchronise per chunk)
  classify_images   RCN.classify_images into a device tensor

Each library runs in its own process (RCN_CUDA_LIB is read at import), the libraries alternating round by round: the in-tree
build ("new") and every --lib NAME=PATH (e.g. the parent commit's build, which lacks evaluate_images and is timed on the other
two).  Images are seeded and device-resident; at 1 048 576 the set is 822 MB, larger than the 126 MB L2.

The other route for u8 images -- the feature kernel, then the inference kernel on the features (smallnet_infer_kernel<0>) --
lost at every size and is not in the library.  profiles/eval_split_route.patch restores it in place of the one-launch route:
apply it to a copy of the tree, build that copy, and pass its library as --lib split=COPY/mercer_research_b200/librcn_cuda.so.

  python profiles/eval_bench.py --out OUT_DIR [--lib parent=/path/librcn_cuda.so] [--rounds 3]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIZES = [1, 64, 1024, 10000, 1 << 20]
CHUNK = 16384


def worker(sizes, repeats):
    """One library (RCN_CUDA_LIB): {method: {B: [ms per call, one per repeat]}}."""
    sys.path.insert(0, ROOT)
    import ctypes
    import numpy as np
    import torch
    from mercer_research_b200 import _lib
    has_eval = hasattr(ctypes.CDLL(_lib.SO_PATH), "rcn_cuda_evaluate_images")
    if not has_eval:                               # a build from before the entry point existed
        del _lib.SIGNATURES["rcn_cuda_evaluate_images"]
    import mercer_research_b200 as api
    dev = torch.device("cuda", 0)
    model = api.RCN(10, [api.RCNLayer.Convolve2D(api.Padding.Same), api.RCNLayer.Pool2D(api.Pooling.Max)], [30], device=0)
    model.load_weights_and_bias(784)
    model.set_params(np.random.default_rng(0xC0FFEE).standard_normal(model.n_params) * 0.1)
    model.scale_set = (40.0, 60.0)
    g = torch.Generator(device=dev).manual_seed(1234)
    n_max = max(sizes)
    images = torch.randint(0, 256, (n_max, 28, 28), dtype=torch.uint8, device=dev, generator=g)
    labels = torch.randint(0, 10, (n_max,), dtype=torch.int64, device=dev, generator=g)
    stream = torch.cuda.current_stream(dev)
    model.set_stream(stream.cuda_stream)
    cost = torch.zeros(1, dtype=torch.float64, device=dev)
    acc = torch.zeros(1, dtype=torch.int64, device=dev)
    lib = _lib.load()

    def m_evaluate_images(x, y):
        _lib.check(lib.rcn_cuda_evaluate_images(model._h, x.data_ptr(), _lib.PIXELS_U8_ROWMAJOR, y.data_ptr(), x.shape[0], 28, 28,
                                                cost.data_ptr(), acc.data_ptr(), None))

    def m_features_evaluate(x, y):
        a = 0
        for i in range(0, x.shape[0], CHUNK):
            a += model.evaluate(model.flatten_feature_set(x[i:i + CHUNK], standardise=True), y[i:i + CHUNK])
        return a

    def m_classify(x, y):
        model.classify_images(x)

    methods = {"features+evaluate": m_features_evaluate, "classify_images": m_classify}
    if has_eval:
        methods["evaluate_images"] = m_evaluate_images
    res, outputs = {}, {}
    for B in sizes:
        x, y = images[:B], labels[:B]
        for name, fn in methods.items():          # warm-up of every shape (allocations, attributes, module loads)
            fn(x, y)
        torch.cuda.synchronize()
        if has_eval:
            m_evaluate_images(x, y)
            torch.cuda.synchronize()
            outputs[str(B)] = {"accept": int(acc.item()), "cost": float(cost.item()),
                               "accept_features_evaluate": int(m_features_evaluate(x, y))}
        iters = max(3, min(500, 4_000_000 // B))
        for name, fn in methods.items():
            times = []
            for _ in range(repeats):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                for _ in range(iters):
                    fn(x, y)
                e1.record(stream)
                e1.synchronize()
                times.append(e0.elapsed_time(e1) / iters)
            res.setdefault(name, {})[str(B)] = times
    print("RESULT " + json.dumps({"times_ms": res, "outputs": outputs}))


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()
        name, power = [s.strip() for s in out[0].split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as e:   # the measurement itself needs the GPU, not nvidia-smi
        return {"gpu": "unknown", "power_limit": "unknown", "error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--lib", action="append", default=[], help="NAME=PATH of another librcn_cuda.so")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--sizes", default=",".join(str(s) for s in SIZES))
    ap.add_argument("--worker", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    sizes = [int(s) for s in args.sizes.split(",")]
    if args.worker:
        worker(sizes, args.repeats)
        return
    import statistics
    os.makedirs(args.out, exist_ok=True)
    sys.path.insert(0, ROOT)
    from mercer_research_b200 import _lib
    libs = {"new": _lib.SO_PATH}
    for spec in args.lib:
        name, path = spec.split("=", 1)
        libs[name] = os.path.abspath(path)
    runs = {name: [] for name in libs}
    for r in range(args.rounds):
        for name, path in libs.items():
            env = dict(os.environ, RCN_CUDA_LIB=path)
            p = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", "--out", args.out, "--sizes", args.sizes,
                                "--repeats", str(args.repeats)], env=env, capture_output=True, text=True, cwd=ROOT)
            line = [l for l in p.stdout.splitlines() if l.startswith("RESULT ")]
            if p.returncode != 0 or not line:
                raise SystemExit(f"worker {name} failed:\n{p.stdout}\n{p.stderr}")
            runs[name].append(json.loads(line[0][7:]))
            print(f"round {r} {name} done", flush=True)
    summary = {}
    for name, rs in runs.items():
        for method in rs[0]["times_ms"]:
            for B in rs[0]["times_ms"][method]:
                meds = [statistics.median(x["times_ms"][method][B]) for x in rs]
                allt = [t for x in rs for t in x["times_ms"][method][B]]
                med = statistics.median(meds)
                summary.setdefault(name, {}).setdefault(method, {})[B] = {
                    "ms_median": med, "ms_min": min(allt), "ms_max": max(allt),
                    "round_medians_ms": meds, "images_per_s": int(B) / (med * 1e-3)}
    result = dict(gpu_info(), rounds=args.rounds, repeats=args.repeats, sizes=sizes, summary=summary,
                  outputs={name: rs[0]["outputs"] for name, rs in runs.items()})
    with open(os.path.join(args.out, "eval_bench.json"), "w") as f:
        json.dump(result, f, indent=1)
    for name in summary:
        for method, per in summary[name].items():
            print(name, method, " ".join(f"B={B}: {v['images_per_s'] / 1e6:.3f} M/s ({v['ms_median']:.4f} ms, {v['ms_min']:.4f}-{v['ms_max']:.4f})"
                                   for B, v in per.items()))


if __name__ == "__main__":
    main()
