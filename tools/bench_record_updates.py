"""Cost of in-place record edits against a rebuild: one JSON line.

On C2 (4096^2 Ising grid) and C4 (KBC-style Boolean graph, 200 M variables) it times
FactorGraph.update_variables for k random evidence flips (with new initial values), the same
edit through the C entry point alone (ids sorted, no Python validation), update_weights flipping
isFixed of 1 and 10^4 weights (one pass over the record streams), a full invalidate() plus
rebuild including its first sweep, and one sweep before and after the edits (same layout: the
time should not move).  Every timed call ends in a device synchronise.

Usage: python tools/bench_record_updates.py [--configs c2,c4] [--c4-vars N] [--out FILE]
"""
import argparse
import ctypes as C
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


def sweep_ms(fg, n=10):
    """Mean time of one sweep (CUDA events on the graph's stream), sample_evidence on: every
    variable is sampled, so the work does not depend on the evidence flags."""
    from numbskull_b200 import _lib
    L, g = _lib.lib(), fg._g
    _lib.check(L.nb_gibbs_sweeps(g, 2, 1, 1, fg.seed))
    _lib.check(L.nb_timer_start(g))
    _lib.check(L.nb_gibbs_sweeps(g, n, 1, 1, fg.seed))
    ms = C.c_float(0)
    _lib.check(L.nb_timer_stop(g, C.byref(ms)))
    return ms.value / n


def random_ids(rng, n, k):
    ids = np.unique(rng.integers(0, n, int(k * 1.2) + 16))
    return rng.permutation(ids)[:k]


def run_config(name, g, rng):
    import numbskull_b200 as nb
    from numbskull_b200 import _lib
    L = _lib.lib()
    ns = nb.NumbSkull(quiet=True)
    t0 = time.perf_counter()
    ns.loadFactorGraph(*g)
    fg = ns.factorGraphs[0]
    fg.seed = 12345
    fg._device_graph()
    build_s = time.perf_counter() - t0
    info = fg.device_info()
    V, W = info["n_variable"], info["n_weight"]
    out = {"variables": V, "weights": W, "edges": info["n_edges"], "stream_bytes": 4 * info["stream_words"],
           "tt_quads": info["tt_quads"], "tt2_quads": info["tt2_quads"], "load_and_build_s": round(build_s, 2)}
    fg._sync_device(0, 0)
    out["sweep_ms_before"] = round(sweep_ms(fg), 4)

    evid = fg.variable["isEvidence"]
    var = {}
    for k in (10 ** 3, 10 ** 5, 10 ** 7):
        if k > V:
            continue
        ids = random_ids(rng, V, k)
        flip = (1 - evid[ids]).astype(np.int8)
        init = rng.integers(0, 2, len(ids))
        t0 = time.perf_counter()
        fg.update_variables(ids, isEvidence=flip, initialValue=init)
        py_ms = 1e3 * (time.perf_counter() - t0)
        # the same edit again (flipped back), through the C entry point alone
        s = np.sort(ids)
        back = np.ascontiguousarray((1 - fg.variable["isEvidence"][s]).astype(np.int8))
        init_s = np.ascontiguousarray(fg.variable["initialValue"][s].astype(np.int64))
        t0 = time.perf_counter()
        _lib.check(L.nb_update_variables(fg._g, _lib.ptr(s), len(s), _lib.ptr(back), _lib.ptr(init_s), None))
        c_ms = 1e3 * (time.perf_counter() - t0)
        fg.variable["isEvidence"][s] = back      # keep the records in step with the device
        var[str(k)] = {"update_variables_ms": round(py_ms, 3), "nb_update_variables_ms": round(c_ms, 3)}
    out["evidence_flips"] = var

    wts = {}
    fixed = fg.weight["isFixed"]
    for k in (1, 10 ** 4):
        k = min(k, W)
        ids = random_ids(rng, W, k)
        t0 = time.perf_counter()
        fg.update_weights(ids, 1 - fixed[ids])
        ms = 1e3 * (time.perf_counter() - t0)
        wts[str(k)] = {"update_weights_ms": round(ms, 3)}
    out["isFixed_flips"] = wts
    out["sweep_ms_after"] = round(sweep_ms(fg), 4)

    d = fg.device_digest()
    t0 = time.perf_counter()
    fg.invalidate()
    fg._sync_device(0, 0)
    _lib.check(L.nb_gibbs_sweeps(fg._g, 1, 1, 1, fg.seed))
    out["invalidate_rebuild_first_sweep_s"] = round(time.perf_counter() - t0, 3)
    out["rebuild_digest_equal"] = fg.device_digest() == d
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--configs", default="c2,c4")
    ap.add_argument("--grid", type=int, default=4096)
    ap.add_argument("--c4-vars", type=int, default=200_000_000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import numbskull_b200 as nb
    from numbskull_b200 import synth
    if nb._lib.device_count() < 1:
        raise SystemExit("no CUDA device: this measurement needs the GPU")
    name, power = gpu_name_and_power()
    line = {"workload": "record_updates", "gpu": name, "power_limit": power}
    rng = np.random.default_rng(2026)
    for cfg in args.configs.split(","):
        if cfg == "c2":
            line["c2_ising_%d" % args.grid] = run_config(cfg, synth.ising_grid(args.grid, args.grid), rng)
        elif cfg == "c4":
            line["c4_kbc_%d" % args.c4_vars] = run_config(cfg, synth.kbc_fast(args.c4_vars, seed=1004), rng)
        else:
            raise SystemExit("unknown config " + cfg)
    s = json.dumps(line)
    print(s)
    if args.out:
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
