"""Kernel A's staged front end on image pairs in packed fp16 lanes, against the int32 front end of an earlier build, in one
GPU session: the card's name and power limit, `bench.py --gpus 1` alternated between the two libraries (`rounds` runs each,
default 2000 steps), the phase clocks of both `-DRCN_SN_PHASES` builds (profiles/build_phases.sh, profiles/sn_phases.py), and
`bench.py --dump-outputs` of both builds compared array for array, bit for bit.

    python profiles/front_pairs_ab.py --base-lib OLD.so --base-phases-lib OLD_PHASES.so --phases-lib NEW_PHASES.so --out DIR \
        [--parts dumps,phases,timing]

The library under test is the tree's own (mercer_research_b200/librcn_cuda.so).  Writes DIR/front_pairs_ab.json after every
measurement, adding to what an earlier call with other --parts wrote there.
"""
import argparse
import glob
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW_LIB = os.path.join(ROOT, "mercer_research_b200", "librcn_cuda.so")


def run(cmd, lib, log):
    env = dict(os.environ, RCN_CUDA_LIB=lib)
    p = subprocess.run(cmd, cwd=ROOT, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    with open(log, "w") as f:
        f.write(p.stderr)
    if p.returncode != 0:
        raise RuntimeError(f"{' '.join(cmd)} failed ({p.returncode}), see {log}")
    return p.stdout


def bench(lib, log, extra=()):
    out = run([sys.executable, "bench.py", "--gpus", "1", *extra], lib, log)
    line = [l for l in out.splitlines() if l.startswith("{")][-1]
    return json.loads(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base-lib", required=True)
    ap.add_argument("--base-phases-lib", required=True)
    ap.add_argument("--phases-lib", required=True)
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--parts", default="dumps,phases,timing")
    args = ap.parse_args()
    parts = set(args.parts.split(","))
    os.makedirs(args.out, exist_ok=True)
    libs = {"base": os.path.abspath(args.base_lib), "pairs": NEW_LIB}
    path = os.path.join(args.out, "front_pairs_ab.json")
    rec = json.load(open(path)) if os.path.exists(path) else {}
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         stdout=subprocess.PIPE, text=True).stdout.strip().splitlines()
    rec.setdefault("gpu", []).append({"parts": args.parts, "card": gpu})   # one entry per call

    def save():
        with open(path, "w") as f:
            json.dump(rec, f, indent=1)

    if "dumps" in parts:
        dump_outputs(libs, args.out, rec)
        save()
    if "phases" in parts:
        kernel_a_phases(args, rec)
        save()
    if "timing" in parts:
        timing(libs, args, rec, save)
    print(json.dumps({k: rec[k] for k in ("gpu", "dump_outputs_bit_identical", "summary_us_per_step") if k in rec}))


def dump_outputs(libs, out, rec):
    """Same seeded inputs through both builds: every array bench.py --dump-outputs writes must be equal bit for bit."""
    dumps = {}
    for name, lib in libs.items():
        d = os.path.join(out, "dump_" + name)
        bench(lib, os.path.join(out, f"dump_{name}.log"), ["--steps", "50", "--dump-outputs", d])
        dumps[name] = d
    files = sorted(os.path.basename(f) for f in glob.glob(os.path.join(dumps["base"], "*.npy")))
    same = {}
    for f in files:
        a, b = np.load(os.path.join(dumps["base"], f)), np.load(os.path.join(dumps["pairs"], f))
        same[f] = bool(a.shape == b.shape and np.array_equal(a.view(np.uint64), b.view(np.uint64)))
    rec["dump_outputs_bit_identical"] = same


def timing(libs, args, rec, save):
    """bench.py --gpus 1 alternated between the builds, `rounds` more runs each; saved after every run."""
    runs = rec.setdefault("bench_us_per_step", {name: [] for name in libs})   # earlier calls' runs are kept
    for _ in range(args.rounds):
        for name, lib in libs.items():
            r = len(runs[name])
            res = bench(lib, os.path.join(args.out, f"bench_{name}_{r}.log"))
            row = {"c2": res["ms_per_step"] * 1e3}
            for w, v in res.get("workloads", {}).items():
                row[w] = v["ms_per_step"] * 1e3
            row["c2_clocks"] = res.get("clocks")
            runs[name].append(row)
            print(name, r, {k: round(v, 3) for k, v in row.items() if isinstance(v, float)}, flush=True)
            summary = {}
            for w in ("c2", "c3", "c4", "c5"):
                s = {}
                for n in libs:
                    v = [row[w] for row in runs[n] if w in row]
                    if v:
                        s[n] = {"median": statistics.median(v), "min": min(v), "max": max(v), "spread": max(v) - min(v)}
                summary[w] = s
            rec["summary_us_per_step"] = summary
            save()


def kernel_a_phases(args, rec):
    """Where the time went: kernel A's phase clocks (-DRCN_SN_PHASES builds of both trees) on the c2 step."""
    phases = {}
    for name, lib in (("base", os.path.abspath(args.base_phases_lib)), ("pairs", os.path.abspath(args.phases_lib))):
        jp = os.path.join(args.out, f"phases_{name}.json")
        print(run([sys.executable, "profiles/sn_phases.py", "1024", "--json", jp], lib, jp + ".log"), flush=True)
        phases[name] = json.load(open(jp))
    rec["kernel_a_phases"] = phases


if __name__ == "__main__":
    main()
