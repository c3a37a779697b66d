"""Throughput of graphs with cardinalities above 255 (2-byte device values): one JSON line.

The shape is synth.wide_categorical: mentions of cardinality K over their candidates, with
EQUAL_CAT_CONST priors, AND_CAT features on Boolean evidence variables and AND_CAT couplings
between mentions.  The default (100 k mentions, K = 1000, 32 candidates x 4 features) has about
30 M incidences, so the streams do not fit the 126 MB L2.  Host memory: a dataType-1 variable
carries K vmap records of 24 B, i.e. 2.4 GB for the default.

Usage: python tools/bench_wide_card.py [--mentions N] [--card K] [--sweeps S] [--epochs E] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_name_and_power(index=0):
    out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=60)
    if out.returncode != 0:
        raise RuntimeError("nvidia-smi failed: " + out.stderr)
    name, power = [x.strip() for x in out.stdout.strip().split(",")]
    return name, power


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--mentions", type=int, default=100000)
    ap.add_argument("--card", type=int, default=1000)
    ap.add_argument("--cands", type=int, default=32)
    ap.add_argument("--feats", type=int, default=4)
    ap.add_argument("--sweeps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--epochs", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import numbskull_b200 as nb
    from numbskull_b200 import synth
    if nb._lib.device_count() < 1:
        raise SystemExit("no CUDA device: this measurement needs the GPU")
    name, power = gpu_name_and_power()
    g = synth.wide_categorical(args.mentions, card=args.card, cands=args.cands, feats=args.feats,
                               rng=np.random.default_rng(2024))
    ns = nb.NumbSkull(quiet=True)
    t0 = time.perf_counter()
    ns.loadFactorGraph(*g)
    fg = ns.factorGraphs[0]
    fg.seed = 7
    info = fg.device_info()
    load_s = time.perf_counter() - t0
    if info["value_bytes"] != 2:
        raise SystemExit("expected a 2-byte graph")

    fg.inference(0, args.warmup, sample_evidence=False)              # warm-up: module load, first touch
    t0 = time.perf_counter()
    fg.inference(0, args.sweeps, sample_evidence=False)              # returns after a device synchronise
    ms_sweep = 1e3 * (time.perf_counter() - t0) / args.sweeps
    assert np.isfinite(fg.marginals).all()

    fg.learn(0, 1, 0.001, 0.99, 2, 0.01, 1)                          # warm-up epoch
    t0 = time.perf_counter()
    fg.learn(0, args.epochs, 0.001, 0.99, 2, 0.01, 1)
    ms_epoch = 1e3 * (time.perf_counter() - t0) / args.epochs

    stream_bytes = 4 * info["stream_words"]
    line = {
        "workload": "wide_categorical",
        "mentions": args.mentions, "card": args.card, "cands": args.cands, "feats": args.feats,
        "variables": info["n_variable"], "factors": info["n_factor"], "edges": info["n_edges"],
        "value_bytes": info["value_bytes"],
        "row_classes": {"pair": info["n_pair_rows"], "fast": info["n_fast_rows"], "cat": info["n_cat_rows"],
                        "thread": info["n_thread_rows"], "warp": info["n_warp_rows"]},
        "n_colors": info["n_colors"],
        "ms_per_sweep": round(ms_sweep, 4),
        "edge_evals_per_s": info["n_edges"] / (ms_sweep * 1e-3),
        "ms_per_learning_epoch": round(ms_epoch, 3),
        "stream_bytes_per_sweep_from_shapes": stream_bytes,
        "device_bytes": info["device_bytes"],
        "sweeps": args.sweeps, "warmup": args.warmup, "learn_epochs": args.epochs,
        "load_and_build_s": round(load_s, 2),
        "gpu": name, "power_limit": power,
    }
    s = json.dumps(line)
    print(s)
    if args.out:
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
