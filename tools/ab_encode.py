#!/usr/bin/env python
"""A/B measurement of two or more builds of the library on the flagship zstd encode, in one process tree on one GPU.

usage: ab_encode.py OUTDIR [--rounds R] [--steps K] [--warmup W] [--lib NAME=PATH ...]

Each round runs `bench.py --no-secondary --no-cpu-baseline --dump-outputs OUTDIR/<NAME>_<round>` once per build, the
builds alternating within the round, with B2C_LIB selecting the library.  Then it prints every run's GB/s and per-kernel
ms, the median and spread per build, and checks that every dump (sizes.npy, frames.npy, frame_index.npy) is identical
across all runs of all builds.  It also runs tools/enc_times.py at levels 1 and 2 (1 GiB) for every build and records
the GPU's name, power limit and clocks.  Default builds: base = ab_libs/base.so (the parent commit's library, built
beforehand and never committed), new = the library build() made.  Everything it writes goes under OUTDIR."""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(cmd, env=None, log=None):
    r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True)
    if log:
        with open(log, "w") as f:
            f.write(r.stdout + r.stderr)
    if r.returncode != 0:
        sys.stderr.write(r.stdout[-4000:] + r.stderr[-4000:])
        raise SystemExit("failed (%d): %s" % (r.returncode, " ".join(cmd)))
    return r.stdout


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("outdir")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--lib", action="append", default=[], metavar="NAME=PATH")
    ap.add_argument("--no-enc-times", action="store_true")
    a = ap.parse_args()
    libs = [tuple(x.split("=", 1)) for x in a.lib] or [
        ("base", os.path.join(ROOT, "ab_libs", "base.so")),
        ("new", os.path.join(ROOT, "compress_b200", "_lib", "libb200comp.so"))]
    libs = [(n, os.path.abspath(p)) for n, p in libs]
    for n, p in libs:
        if not os.path.exists(p):
            raise SystemExit("%s: %s is missing" % (n, p))
    os.makedirs(a.outdir, exist_ok=True)
    out = open(os.path.join(a.outdir, "ab_summary.txt"), "w")

    def say(s=""):
        print(s)
        out.write(s + "\n")
        out.flush()

    say(run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv"]).strip())
    env0 = dict(os.environ, PYTHONDONTWRITEBYTECODE="1")
    res = {n: [] for n, _ in libs}
    for r in range(a.rounds):
        for n, p in libs:
            d = os.path.join(a.outdir, "%s_%d" % (n, r))
            line = run([sys.executable, "bench.py", "--gpus", "1", "--steps", str(a.steps), "--warmup", str(a.warmup),
                        "--no-secondary", "--no-cpu-baseline", "--dump-outputs", d], env=dict(env0, B2C_LIB=p),
                       log=os.path.join(a.outdir, "%s_%d.log" % (n, r)))
            j = json.loads([x for x in line.splitlines() if x.startswith("{")][-1])
            res[n].append((d, j))
            kms = j["roofline"]["kernel_ms_per_step"]
            say("round %d %-6s %.2f GB/s  ratio %.6f  launches %d  kernels ms/step: %s" % (
                r, n, j["value"], j["ratio"], j["gpu_launches"],
                "  ".join("%s %.3f" % (k.replace("b2c_zstd_", "").replace("b2c_", "").replace("_kernel", ""), v)
                          for k, v in kms.items())))
    say()
    med = {}
    for n, _ in libs:
        v = sorted(j["value"] for _, j in res[n])
        med[n] = statistics.median(v)
        say("%-6s median %.2f GB/s  min %.2f  max %.2f  spread %.2f %%" % (n, med[n], v[0], v[-1], 100 * (v[-1] - v[0]) / med[n]))
        kms = {}
        for _, j in res[n]:
            for k, x in j["roofline"]["kernel_ms_per_step"].items():
                kms.setdefault(k, []).append(x)
        say("       median kernel ms/step: " + "  ".join("%s %.3f" % (k, statistics.median(x)) for k, x in kms.items()))
    n0 = libs[0][0]
    for n, _ in libs[1:]:
        say("%s / %s = %.4f (medians); slowest %s %.2f vs fastest %s %.2f" % (
            n, n0, med[n] / med[n0], n, min(j["value"] for _, j in res[n]), n0, max(j["value"] for _, j in res[n0])))
    # every dump must equal the first one
    ref_dir = res[n0][0][0]
    same = True
    for n, _ in libs:
        for d, j in res[n]:
            for f in ("sizes.npy", "frames.npy", "frame_index.npy"):
                if not np.array_equal(np.load(os.path.join(ref_dir, f)), np.load(os.path.join(d, f))):
                    same = False
                    say("DIFFERENT: %s/%s" % (d, f))
            if j["ratio"] != res[n0][0][1]["ratio"]:
                same = False
                say("DIFFERENT ratio: %s %r" % (d, j["ratio"]))
    say("dumps and ratio identical across all runs: %s" % same)
    if not a.no_enc_times:
        for lv in (1, 2):
            for n, p in libs:
                say("--- enc_times level %d, %s" % (lv, n))
                say(run([sys.executable, os.path.join("tools", "enc_times.py"), str(lv), "1"], env=dict(env0, B2C_LIB=p)).strip())
    say(run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv"]).strip())
    if not same:
        raise SystemExit(1)


if __name__ == "__main__":
    main()
