#!/usr/bin/env python
"""Benchmark of the Gibbs-sweep / weight-learning hot path (BASELINE.json metric:
factor-edge evaluations / s and variable samples / s per sweep).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workloads c2,c4,c3] [--dump-outputs DIR]

Headline workload (``value``, ``e2e``, ``roofline``): BASELINE config 2, the
4096 x 4096 Boolean Ising grid with EQUAL pairwise factors, inference only; a
"step" is one full chromatic Gibbs sweep (every colour once).  After W warm-up
steps the K timed steps run back to back in one call of the library, bracketed
by CUDA events on its stream (barrier + synchronize on both sides).  Every
workload times exactly K of its steps; the ``e2e`` calls through the public API
that follow are timed separately, min(max(K, 3), 10) of them.

``--dump-outputs DIR`` writes what the timed steps computed, as a caller of
that path receives it, to ``DIR/<name>.npy`` (float32 / float64): the sampled
values and the marginals of the K timed sweeps (``c2_*``, ``c4_*``) and the
learned weights (``learn_weights``).  Per-variable arrays hold a fixed, seeded
sample of DUMP_SAMPLE variables.  The inputs depend on the arguments alone, so
two builds run with the same arguments can be compared output for output.

With N = 1 two more blocks ride in the same JSON line:
  ``c4``     BASELINE config 4 at full size (200 M Boolean variables / 1 B edges,
             mixed ISTRUE / IMPLY / AND / OR factors): the configuration the
             north-star target (>= 1e10 edge evals/s at >= 60 % of the HBM
             roofline) is stated on, with its own ``roofline``;
  ``learn``  BASELINE config 3 shape (1 M candidates x 100 labelling functions):
             weight-learning epochs with the B_learn roofline.
With N > 1 every rank owns a 4096-row strip of a (4096*N) x 4096 grid (weak
scaling) and exchanges its boundary rows after every colour; before timing the
ranks prove on a small strip problem that the partitioned run reproduces the
single-GPU tallies bit for bit (``p2p_bit_identical``).

``roofline.frac`` follows SURVEY.md 8(d) (algorithmic bytes / time / measured
copy peak) and can exceed 1 for the Ising kernel, whose 4-byte records move far
fewer bytes than the formula's 30 per edge; ``roofline.frac_dram`` is the same
ratio on the DRAM bytes ncu measured for the kernel (profiles/traffic.json).

``--impl reference`` times the UNMODIFIED numba reference (baseline/_ref, see
baseline/install_ref.sh) on this box's host cores; its inputs are built with
numpy and its own compute_var_map -- no library of this repo is loaded.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))

GRID = int(os.environ.get("NB_BENCH_GRID", 4096))          # rows per GPU and columns
CPU_GRID = int(os.environ.get("NB_BENCH_CPU_GRID", 1024))   # bounded sample for the cpu_baseline leg
C4_VARS = int(os.environ.get("NB_BENCH_C4_VARS", 200_000_000))
C3_COPIES = int(os.environ.get("NB_BENCH_C3_COPIES", 1_000_000))
DUMP_SAMPLE = 1 << 20                                       # variables per dumped array (<= 8 MB each)
METRIC = "factor_edge_evals_per_sec"
UNIT = "factor-edge evals/s"
SEED = 20261017


# --------------------------------------------------------------------------- helpers
def ising_algorithmic_bytes(rows, cols):
    """SURVEY.md section 8(d): B_inf = N_v*16 + sum over edge evals (20 + 5*arity)."""
    nvar = rows * cols
    edge_evals = 2 * (rows * (cols - 1) + (rows - 1) * cols)   # every factor is seen from both ends
    return 16.0 * nvar + edge_evals * (20 + 5 * 2), nvar, edge_evals


def measured_peak():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(key):
    """DRAM bytes per sweep of a kernel from the committed ncu capture (or None)."""
    p = os.path.join(REPO, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get(key)
        except Exception:
            pass
    return None


def roofline(bytes_per_step, ms_per_step, kernel, traffic_key):
    peak, peak_src = measured_peak()
    achieved = bytes_per_step / (ms_per_step * 1e-3) / 1e9
    traffic = ncu_traffic(traffic_key)
    out = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
           "traffic": traffic, "peak_source": peak_src, "algorithmic_bytes_per_step": bytes_per_step,
           "kernel": kernel,
           "frac_note": "frac = SURVEY 8(d) algorithmic bytes / time / peak (may exceed 1 when the record layout moves "
                        "fewer bytes than the formula); frac_dram = ncu dram bytes of the same kernel / time / peak"}
    if traffic:
        out["frac_dram"] = traffic / (ms_per_step * 1e-3) / 1e9 / peak
    return out


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.stop = [], False
        self.index = index
        self.t = threading.Thread(target=self._run, daemon=True)
        self.first = threading.Event()

    def _run(self):
        while not self.stop:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], stdout=subprocess.PIPE,
                                     stderr=subprocess.DEVNULL, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.first.set()
            time.sleep(0.1)

    def __enter__(self):
        # the first query's Python start-up holds the GIL: waiting for it keeps the main thread from
        # stalling between the timer's start event and the launches that follow
        self.t.start()
        self.first.wait(timeout=10)
        return self

    def __exit__(self, *a):
        self.stop = True
        self.t.join(timeout=6)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows for i in range(4)
                          if len(r) >= 7 and r[3 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm)}


# --------------------------------------------------------------------------- reference arm (numba, CPU)
def _ref_ising_arrays(n, m, types, coupling=0.1):
    """The config-2 grid in the REFERENCE's record dtypes (same construction as numbskull_b200/synth.py
    ising_grid; restated here so that this arm imports nothing of the repo's package)."""
    Weight, Variable, Factor, FactorToVar = types
    weight = np.zeros(1, Weight)
    weight["isFixed"] = True
    weight["initialValue"] = coupling
    variable = np.zeros(n * m, Variable)
    variable["cardinality"] = 2
    ii, jj = np.divmod(np.arange(n * m, dtype=np.int64), m)
    has_up, has_left = ii != 0, jj != 0
    nf = has_up.astype(np.int64) + has_left
    first = np.zeros(n * m, np.int64)
    np.cumsum(nf[:-1], out=first[1:])
    nfac = int(nf.sum())
    vid = np.arange(n * m, dtype=np.int64)
    self_id, other = np.empty(nfac, np.int64), np.empty(nfac, np.int64)
    self_id[first[has_up]] = vid[has_up]
    other[first[has_up]] = vid[has_up] - m
    ls = first[has_left] + has_up[has_left]
    self_id[ls] = vid[has_left]
    other[ls] = vid[has_left] - 1
    factor = np.zeros(nfac, Factor)
    factor["factorFunction"] = 3
    factor["featureValue"] = 1.0
    factor["arity"] = 2
    factor["ftv_offset"] = 2 * np.arange(nfac, dtype=np.int64)
    fmap = np.zeros(2 * nfac, FactorToVar)
    fmap["vid"][0::2] = self_id
    fmap["vid"][1::2] = other
    return weight, variable, factor, fmap, np.zeros(n * m, np.bool_), int(2 * nfac)


def _import_reference():
    ref = os.path.join(REPO, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref, "numbskull")):
        raise RuntimeError("baseline/_ref is missing: run baseline/install_ref.sh <numbskull source checkout>")
    sys.path[:0] = [ref, os.path.join(REPO, "baseline", "shims")]
    import numbskull
    assert os.path.abspath(numbskull.__file__).startswith(ref), numbskull.__file__
    from numbskull.numbskulltypes import Weight, Variable, Factor, FactorToVar
    return numbskull, (Weight, Variable, Factor, FactorToVar)


def _ref_graph(numbskull, types, grid, threads):
    ns = numbskull.NumbSkull(nthreads=threads, quiet=True)
    ns.loadFactorGraph(*_ref_ising_arrays(grid, grid, types))       # the reference's public loader
    return ns.factorGraphs[0]


def reference_throughput(steps, warmup, grid=None, threads=None, budget_s=150.0):
    """Times fg.inference() of the unmodified numba reference with nthreads = all host cores and
    reads the reference's own accumulator fg.inference_total_time (factorgraph.py:156-168).  The grid
    is the 4096^2 config when warm-up + K sweeps fit the time budget, else the largest power-of-two
    fraction of it that does (stated in the line)."""
    numbskull, types = _import_reference()
    threads = threads or os.cpu_count() or 1
    if grid is None:
        probe = _ref_graph(numbskull, types, 256, threads)
        probe.inference(0, 1, sample_evidence=True)                 # JIT compilation happens here
        t0 = probe.inference_total_time
        probe.inference(0, 2, sample_evidence=True)
        per_var = (probe.inference_total_time - t0) / 2 / (256 * 256)
        per_var_load = 8e-6                                         # loadFactorGraph's Python loop (numbskull.py:222-227)
        grid = GRID
        while grid > 256 and grid * grid * (per_var * (steps + warmup) + per_var_load) > budget_s:
            grid //= 2
    fg = _ref_graph(numbskull, types, grid, threads)
    fg.inference(0, max(1, warmup), sample_evidence=True)
    t0 = fg.inference_total_time
    fg.inference(0, steps, sample_evidence=True)
    dt = fg.inference_total_time - t0
    _, nvar, edges = ising_algorithmic_bytes(grid, grid)
    return {"value": edges * steps / dt, "unit": UNIT, "cores": threads, "kind": "reference",
            "sample": "%dx%d Ising grid, %d sweeps of the unmodified numba reference (baseline/_ref, numba gibbsthread), "
                      "nthreads=%d, time = fg.inference_total_time" % (grid, grid, steps, threads),
            "grid": grid, "var_samples_per_sec": nvar * steps / dt, "ms_per_step": 1e3 * dt / steps}


def reference_learning_throughput(copies=5000, n_lf=100, epochs=2, threads=None):
    """fg.learn() of the unmodified numba reference on the labelling-function model (BASELINE config 3
    shape, options of test_lf_learning.py:129-137), nthreads = all host cores, time = the reference's own
    fg.learning_total_time (factorgraph.py:196-205).  A bounded sample: loadFactorGraph's Python loops
    alone need ~8 us per variable."""
    numbskull, types = _import_reference()
    Weight, Variable, Factor, FactorToVar = types
    threads = threads or os.cpu_count() or 1
    sys.path.insert(0, REPO)
    from numbskull_b200 import synth
    w, v, f, fm, dm, e = synth.lf_model(copies, n_lf, np.random.default_rng(1003))
    conv = lambda a, t: np.ascontiguousarray(a).view(t) if a.dtype.itemsize == np.dtype(t).itemsize else a.astype(t)  # noqa: E731
    ns = numbskull.NumbSkull(nthreads=threads, quiet=True, learn_non_evidence=True)
    ns.loadFactorGraph(conv(w, Weight), conv(v, Variable), conv(f, Factor), conv(fm, FactorToVar), dm, e)
    fg = ns.factorGraphs[0]

    def learn(n):
        fg.learn(0, n, 1e-4, 1.0, 1, 0.01, 1.0, learn_non_evidence=True)
    learn(1)                                                            # JIT compilation happens here
    t0 = fg.learning_total_time
    learn(epochs)
    dt = (fg.learning_total_time - t0) / epochs
    edges = copies * (1 + 2 * n_lf)
    return {"value": edges / dt, "unit": UNIT, "cores": threads, "kind": "reference", "ms_per_epoch": 1e3 * dt,
            "sample": "lf_model %d x %d (%d variables), %d learning epochs of the unmodified numba reference "
                      "(baseline/_ref, numba learnthread), nthreads=%d, time = fg.learning_total_time"
                      % (copies, n_lf, copies * (1 + n_lf), epochs, threads)}


def run_reference(args):
    if int(os.environ.get("RANK", 0)) != 0:
        return
    if args.ref_mode == "learn":
        try:
            OUT.emit(json.dumps(dict(reference_learning_throughput(), impl="reference")))
        except Exception as exc:  # noqa: BLE001
            OUT.emit(json.dumps({"impl": "reference", "unavailable": "%s: %s" % (type(exc).__name__, exc)}))
        return
    if args.ref_mode == "single":
        try:
            r = reference_throughput(3, 1, grid=512, threads=1)
            OUT.emit(json.dumps(dict({k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}, impl="reference")))
        except Exception as exc:  # noqa: BLE001
            OUT.emit(json.dumps({"impl": "reference", "unavailable": "%s: %s" % (type(exc).__name__, exc)}))
        return
    steps, warmup = max(1, args.steps), max(1, args.warmup)
    try:
        r = reference_throughput(steps, warmup, grid=args.ref_grid or None)
    except Exception as exc:  # noqa: BLE001
        # no baseline/_ref here (baseline/install_ref.sh installs it from a numbskull checkout): the oracle
        # port always exists -- the C restatement of gibbsthread, all host threads
        try:
            grid = args.ref_grid or 2048
            r = cpu_port_throughput(steps, warmup, grid=grid)
            _, nvar, edges = ising_algorithmic_bytes(grid, grid)
            r.update(grid=grid, ms_per_step=1e3 * edges / r["value"], var_samples_per_sec=r["value"] * nvar / edges,
                     sample=r["sample"] + " (numba reference unavailable: %s)" % exc)
        except Exception as exc2:  # noqa: BLE001
            OUT.emit(json.dumps({"impl": "reference", "unavailable": "%s: %s; oracle port: %s" % (type(exc).__name__, exc, exc2)}))
            return
    g = r["grid"]
    line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT,
            "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": r["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": "ising_%dx%d_equal_inference" % (g, g) +
                                   ("" if g == GRID else " (bounded sample of the %dx%d config: the full grid does not "
                                                         "finish %d sweeps within the time budget on %d cores)"
                                                         % (GRID, GRID, steps + warmup, r["cores"]))},
            "var_samples_per_sec": r["var_samples_per_sec"],
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    OUT.emit(json.dumps(line))


def reference_child(mode):
    """One bounded run of the numba reference in a child process (--ref-mode single | learn)."""
    try:
        res = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--ref-mode", mode],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=600)
        line = json.loads(res.stdout.strip().splitlines()[-1])
        line.pop("impl", None)
        return line
    except Exception as exc:  # noqa: BLE001
        return {"unavailable": "numba reference: %s" % exc}


def cpu_baselines(no_port=False):
    """cpu_baseline leg of our arm: the numba reference in a child process (it must not share a
    process with this repo's `numbskull` alias package) on a bounded 1024^2 grid, plus the C port."""
    out = {}
    try:
        res = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "3",
                              "--warmup", "1", "--ref-grid", str(CPU_GRID)], stdout=subprocess.PIPE,
                             stderr=subprocess.DEVNULL, text=True, timeout=600)
        line = json.loads(res.stdout.strip().splitlines()[-1])
        out = dict(line.get("cpu_baseline") or {"unavailable": line.get("unavailable")})
    except Exception as exc:  # noqa: BLE001
        out = {"unavailable": "numba reference: %s" % exc}
    out["single_thread"] = reference_child("single")
    if not no_port:
        try:
            out["port"] = cpu_port_throughput(steps=3, warmup=1)
        except Exception as exc:  # noqa: BLE001
            out["port"] = {"unavailable": str(exc)}
    return out


def cpu_port_throughput(steps, warmup, grid=CPU_GRID, threads=None):
    """The CPU oracle (C port of the reference's gibbsthread sweep, Hogwild over contiguous variable
    ranges like run_pool) on a bounded grid -- second cpu_baseline entry, kind "port"."""
    import oracle
    from numbskull_b200 import synth
    threads = threads or os.cpu_count() or 1
    from numbskull_b200.numbskulltypes import VarToFactor
    w, v, f, fm, dm, e = synth.ising_grid(grid, grid)
    v["vtf_offset"] = np.arange(len(v))                  # Boolean variables: one bucket each (numbskull.py:222-227)
    vm, fi = np.zeros(len(v), VarToFactor), np.zeros(len(fm), np.int64)
    oracle.compute_var_map(v, f, fm, vm, fi, dm)
    og = oracle.OracleGraph(w, v, f, fm, vm, fi, nthreads=threads, seed=1)
    _, nvar, edges = ising_algorithmic_bytes(grid, grid)
    og.inference(0, warmup, sample_evidence=True)
    t0 = time.perf_counter()
    og.inference(0, steps, sample_evidence=True)
    dt = time.perf_counter() - t0
    return {"value": edges * steps / dt, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": "%dx%d Ising grid, %d sweeps, C port of gibbsthread (oracle/nb_oracle.c), %d Hogwild threads"
                      % (grid, grid, steps, threads)}


# --------------------------------------------------------------------------- GPU arm
class Dev(object):
    """Timing helpers on the library's stream."""

    def __init__(self, fg, world):
        import torch
        from numbskull_b200 import _lib
        self.torch, self.lib, self.L = torch, _lib, _lib.lib()
        self.fg, self.g, self.world = fg, fg._device_graph(), world

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        self.torch.cuda.synchronize()
        self.lib.check(self.L.nb_synchronize(self.g))

    def max_over_ranks(self, x):
        if self.world == 1:
            return float(x)
        import torch.distributed as dist
        t = self.torch.tensor([float(x)], device="cuda", dtype=self.torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def launches(self):
        n = C.c_int64(0)
        self.L.nb_launch_count(self.g, C.byref(n))
        return n.value

    def timed(self, fn, steps):
        """fn(steps) between CUDA events on the launching stream, barrier + sync on both sides;
        milliseconds, max over ranks."""
        self.barrier()
        self.lib.check(self.L.nb_timer_start(self.g))
        fn(steps)
        ms = C.c_float(0)
        self.lib.check(self.L.nb_timer_stop(self.g, C.byref(ms)))
        self.barrier()
        return self.max_over_ranks(ms.value)

    def state(self, prefix, n_vars, epochs, seed):
        """The chain-0 values and the marginals (tallies / epochs) of a seeded sample of the first
        n_vars variables, as a caller of FactorGraph.inference receives them (Boolean variables:
        one tally each)."""
        fg = self.fg
        vals = np.empty(len(fg.variable), np.int64)
        self.lib.check(self.L.nb_get_var_values(self.g, 0, self.lib.ptr(vals)))
        marg = np.empty(int(fg.cstart[-1]), np.float64)
        self.lib.check(self.L.nb_get_marginals(self.g, self.lib.ptr(marg), float(epochs)))
        if n_vars > DUMP_SAMPLE:
            ids = np.sort(np.random.default_rng(seed).choice(n_vars, DUMP_SAMPLE, replace=False))
        else:
            ids = np.arange(n_vars)
        return {prefix + "var_value": vals[ids].astype(np.float32), prefix + "marginals": marg[fg.cstart[ids]]}


def write_dump(out_dir, arrays):
    """DIR/<name>.npy for every array (float32 / float64, 64 MB at most in all)."""
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def block_c4(args, local_rank, dump):
    """BASELINE config 4 at full size on one GPU; its outputs go into `dump` unless it is None."""
    import numbskull_b200 as nb
    from numbskull_b200 import _lib, synth
    t0 = time.perf_counter()
    g = synth.kbc_fast(C4_VARS, seed=1004)
    t1 = time.perf_counter()
    ns = nb.NumbSkull(quiet=True)
    ns.loadFactorGraph(*g)
    del g
    fg = ns.factorGraphs[0]
    fg.device, fg.seed = local_rank, SEED
    t2 = time.perf_counter()
    dev = Dev(fg, 1)
    t3 = time.perf_counter()
    info = fg.device_info()
    ar = fg.factor["arity"].astype(np.int64)
    nvar, edges = len(fg.variable), int(info["n_edges"])
    # every variable is sampled (sample_evidence) and no hub repeats inside a factor often enough to matter:
    # B_inf = 16 N_v + sum_f arity_f (20 + 5 arity_f)
    bytes_sweep = 16.0 * nvar + float((ar * (20 + 5 * ar)).sum())
    del ar
    L = dev.L
    steps = args.steps

    def sweeps(n):
        _lib.check(L.nb_gibbs_sweeps(dev.g, n, 0, 1, fg.seed))
    sweeps(3)
    _lib.check(L.nb_reset_counts(dev.g))        # the marginals of the timed sweeps alone
    import torch
    rt = torch.cuda.cudart()
    l0 = dev.launches()
    rt.cudaProfilerStart()
    ms = dev.timed(sweeps, steps)
    rt.cudaProfilerStop()
    l1 = dev.launches()
    if dump is not None:
        dump.update(dev.state("c4_", nvar, steps, 4))
    per_step = ms / steps
    bad = C.c_int64(-1)
    _lib.check(L.nb_graph_check_coloring(dev.g, C.byref(bad)))
    _lib.check(L.nb_reset_counts(dev.g))
    t4 = time.perf_counter()
    fg.inference(0, 1, sample_evidence=True)
    m = fg.marginals
    e2e_ms = 1e3 * (time.perf_counter() - t4)
    out = {"workload": "kbc_%d_vars_%d_edges_mixed_istrue_imply_and_or_inference (BASELINE config 4%s)"
                       % (nvar, edges, "" if C4_VARS == 200_000_000 else ", scaled"),
           "metric": METRIC, "value": edges / (per_step * 1e-3), "unit": UNIT, "ms_per_step": per_step,
           "var_samples_per_sec": nvar / (per_step * 1e-3), "steps": steps, "timed_ms": ms,
           "variables": nvar, "factor_edge_evals_per_sweep": edges, "colors": int(info["n_colors"]),
           "color_conflicts": int(bad.value), "device_GB": round(info["device_bytes"] / 1e9, 2),
           "gpu_launches": int(l1 - l0),
           "rows": {"pair": int(info["n_pair_rows"]), "fast": int(info["n_fast_rows"]), "warp": int(info["n_warp_rows"])},
           "roofline": roofline(bytes_sweep, per_step, "k_gibbs_tt (FAST rows: 16-byte truth-table quads with the weight "
                                "inlined, member gathers from the bit-packed value mirror; one launch per colour; "
                                "traffic = all launches of one sweep)", "k_gibbs_tt_c4_bytes_per_sweep"),
           "e2e_first_call_ms": e2e_ms, "mean_marginal": float(m.mean()),
           "build_s": {"generate": round(t1 - t0, 1), "host_index": round(t2 - t1, 1), "device": round(t3 - t2, 1)}}
    fg.clear()
    del fg, ns, dev
    return out


def block_learn(args, local_rank, dump):
    """BASELINE config 3 shape: weight learning on the labelling-function model (L1, learn_non_evidence,
    step 1e-4 as test_lf_learning.py:129-137); the learned weights go into `dump` unless it is None."""
    import numbskull_b200 as nb
    from numbskull_b200 import _lib, synth
    n_lf = 100
    g = synth.lf_model(C3_COPIES, n_lf, np.random.default_rng(1003))
    ns = nb.NumbSkull(quiet=True)
    ns.loadFactorGraph(*g)
    del g
    fg = ns.factorGraphs[0]
    fg.device, fg.seed = local_rank, SEED
    dev = Dev(fg, 1)
    L = dev.L
    copies = C3_COPIES
    # B_learn (SURVEY 8d) = B_inf(free chain, all variables) + B_inf(evid chain, non-evidence variables, no count
    # term) + 12 per gradient visit.  Per candidate: y (Boolean, 1 + n_lf incidences) and n_lf evidence LFs.
    edges = copies * (1 + 2 * n_lf)
    per_edge_y = 25.0 + n_lf * 30.0                       # y's incidences: arity 1 prior + n_lf arity-2 factors
    b_free = copies * (16.0 * (1 + n_lf) + per_edge_y + n_lf * 30.0)
    b_evid = copies * (8.0 + per_edge_y)                   # only y is non-evidence
    b_learn = b_free + b_evid + 12.0 * edges
    fg._sync_device(0, 0)

    def epochs(n):
        s = C.c_double(1e-4)
        _lib.check(L.nb_learn_sweeps(dev.g, n, C.byref(s), 1.0, 1, 0.01, 1.0, 1, fg.seed, 0))
    epochs(1)
    import torch
    rt = torch.cuda.cudart()
    l0 = dev.launches()
    rt.cudaProfilerStart()
    ms = dev.timed(epochs, args.steps)
    rt.cudaProfilerStop()
    l1 = dev.launches()
    per_step = ms / args.steps
    fg._stale.add("weight_value")
    w = fg.weight_value[0]
    if dump is not None:
        dump["learn_weights"] = w.copy()
    out = {"workload": "lf_model_%dx%d_learning_L1_learn_non_evidence_step1e-4 (BASELINE config 3 shape, %s of its size)"
                       % (copies, n_lf, "%.0f%%" % (100.0 * copies / 1e7)),
           "metric": METRIC, "value": edges / (per_step * 1e-3), "unit": UNIT, "ms_per_step": per_step, "step": "one learning epoch",
           "steps": args.steps, "timed_ms": ms, "variables": int(len(fg.variable)),
           "factor_edge_evals_per_epoch": int(edges), "gpu_launches_per_epoch": (l1 - l0) / args.steps,
           "roofline": roofline(b_learn, per_step, "learning epoch (both chains + gradient reduction by weight id)",
                                "learn_c3_bytes_per_epoch"),
           "weights_head": [round(float(x), 4) for x in w[:6]], "weights_finite": bool(np.isfinite(w).all())}
    fg.clear()
    return out


def block_c4_strong(args, rank, world, local_rank):
    """BASELINE config 4 (the 200 M-variable / 1 B-edge KBC graph) partitioned over the ranks: STRONG
    scaling -- the same graph whatever N.  Every rank generates its owner block on its own
    (synth.kbc_block: the global graph is never materialised), ghosts are refreshed after every
    colour.  Returns the block on rank 0, None elsewhere."""
    import torch
    import torch.distributed as dist
    from numbskull_b200 import _lib, partition, synth
    t0 = time.perf_counter()
    bounds = partition.block_bounds(C4_VARS, world)
    local = synth.kbc_block(C4_VARS, int(bounds[rank]), int(bounds[rank + 1]), seed=1004)
    n_ghost = len(local["variable"]) - local["n_owned"]
    t1 = time.perf_counter()
    run = partition.PartitionedGibbs(local, C4_VARS, rank, world, local_rank, seed=SEED)
    del local
    t2 = time.perf_counter()
    fg = run.fg
    dev = Dev(fg, world)
    fg._sync_device(0, 0, evid=False)
    run.sweeps(2, True, True)
    steps = args.steps
    ms = dev.timed(lambda n: run.sweeps(n, False, True), steps)
    if run.p2p:
        _lib.check(dev.L.nb_p2p_check(dev.g))
    per_step = ms / steps
    tot = torch.tensor([float(fg.color_edges().sum()), float(run.n_owned), float(n_ghost), float(run.halo_bytes_per_sweep),
                        t1 - t0, t2 - t1], device="cuda", dtype=torch.float64)
    mx = tot.clone()
    dist.all_reduce(tot)
    dist.all_reduce(mx, op=dist.ReduceOp.MAX)
    out = None
    if rank == 0:
        edges = tot[0].item()
        out = {"workload": "kbc_%d_vars_%d_edges_block_partitioned_over_%d_gpus (BASELINE config 4, strong scaling)"
                           % (C4_VARS, int(edges), world),
               "metric": METRIC, "value": edges / (per_step * 1e-3), "unit": UNIT, "ms_per_step": per_step, "scaling": "strong",
               "steps": steps, "timed_ms": ms, "colors": run.n_colors, "phases_per_sweep": run.n_phases,
               "ghost_copies_total": int(tot[2].item()), "ghost_copies_per_owned_variable": tot[2].item() / max(tot[1].item(), 1),
               "halo_values_per_sweep_total": int(tot[3].item()), "halo_values_per_sweep_max_rank": int(mx[3].item()),
               "transport": "NVLink peer stores + in-kernel flag barrier" if run.p2p else "NCCL point-to-point",
               "boundary_interior_split": bool(run.split), "jp_rounds": run.jp_rounds,
               "build_s": {"generate_block_max": round(mx[4].item(), 1), "partitioned_build_max": round(mx[5].item(), 1)},
               "limiting_phase": "per colour: boundary kernel + halo push (%d values per rank and sweep at most) + interior "
                                 "kernel; %d phases of launch + flag latency per sweep" % (int(mx[3].item()), run.n_phases)}
    run.close()
    return out


def p2p_identity_check(rank, world, local_rank):
    """Before timing: a (256*world) x 256 strip problem sampled partitioned (this launch, the same
    transport the timed sweeps use) and unpartitioned (every rank, its own GPU) must give the same
    tallies bit for bit."""
    import torch
    import torch.distributed as dist
    import numbskull_b200 as nb
    from numbskull_b200 import _lib, partition, synth
    rows, cols, epochs = 256, 256, 20
    run = partition.ising_strip_runner(rows, cols, rank, world, local_rank, seed=77)
    marg = run.inference(2, epochs, sample_evidence=True)
    if run.p2p:
        _lib.check(_lib.lib().nb_p2p_check(run.fg._g))
    ns = nb.NumbSkull(quiet=True)
    ns.loadFactorGraph(*synth.ising_grid(rows * world, cols))
    fg = ns.factorGraphs[0]
    fg.device, fg.seed = local_rank, 77
    fg.inference(2, epochs, sample_evidence=True)
    want = fg.marginals[rank * rows * cols:(rank + 1) * rows * cols]
    same = bool(np.array_equal(np.asarray(marg), want))
    t = torch.tensor([1 if same else 0], device="cuda", dtype=torch.int64)
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    fg.clear()
    p2p, split = bool(run.p2p), bool(run.split)
    run.close()
    return bool(int(t.item())), p2p, split


def run_ours(args):
    sys.path.insert(0, REPO)
    import torch
    from numbskull_b200 import _lib, synth
    import numbskull_b200 as nb

    world = int(os.environ.get("WORLD_SIZE", 1))
    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        # stdout carries ONE JSON line: keep NCCL's banner out of it
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        import datetime
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank),
                                timeout=datetime.timedelta(seconds=300))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    L = _lib.lib()
    steps, warmup = args.steps, max(3, args.warmup)
    workloads = [w for w in args.workloads.split(",") if w]
    dump = None if args.dump_outputs is None else {}

    identical = None
    if world > 1:
        identical = p2p_identity_check(rank, world, local_rank)
        if not identical[0]:
            raise RuntimeError("partitioned run does not reproduce the single-GPU tallies")

    rows, cols = GRID, GRID
    if world == 1:
        ns = nb.NumbSkull(quiet=True)
        ns.loadFactorGraph(*synth.ising_grid(rows, cols))
        fg = ns.factorGraphs[0]
        fg.device, fg.seed = local_rank, SEED
        runner = None
    else:
        from numbskull_b200 import partition
        runner = partition.ising_strip_runner(rows, cols, rank, world, local_rank, seed=SEED)
        fg = runner.fg
    dev = Dev(fg, world)
    g = dev.g
    info = fg.device_info()
    bytes_sweep, nvar, edges = ising_algorithmic_bytes(rows, cols)
    if world == 1:
        assert edges == info["n_edges"], (edges, info["n_edges"])

    def sweeps(n, burnin=False):
        if runner is None:
            _lib.check(L.nb_gibbs_sweeps(g, n, int(burnin), 1, fg.seed))
        else:
            runner.sweeps(n, burnin=burnin, sample_evidence=True)

    fg._sync_device(0, 0)
    _lib.check(L.nb_reset_counts(g))
    # `ncu --profile-from-start off` then lists exactly the launches of the timed region and of the
    # end-to-end steps (no-ops without a profiler)
    cudart = torch.cuda.cudart()
    with ClockSampler(local_rank) as clocks:
        # warm-up right before the timed sweeps, as burn-in: the marginals are those of the timed sweeps
        sweeps(warmup, burnin=True)
        dev.barrier()
        l0 = dev.launches()
        cudart.cudaProfilerStart()
        t0 = time.perf_counter()
        dev_ms = dev.timed(sweeps, steps)
        wall = time.perf_counter() - t0
        cudart.cudaProfilerStop()
        l1 = dev.launches()
        if dump is not None and rank == 0:     # rank 0's own strip when partitioned
            dump.update(dev.state("c2_", len(fg.variable) if runner is None else runner.n_owned, steps, 2))
        # keep the GPUs busy a little longer so that the sampler sees clocks under load
        # (same count on every rank: it is derived from the rank-agreed dev_ms)
        if dev_ms < 1500:
            sweeps(max(1, int(steps * 1500 / max(dev_ms, 1e-3)) // 4))
            dev.barrier()

    # ---- end to end through the public API with host buffers ----
    # step = new weights in (host float64 array, uploaded because it changed) -> FactorGraph.inference(0, 1)
    # -> the step's result out: the float64 marginals the reference API returns (device tallies cross PCIe
    # as 1 byte each, widened by host threads).  var_value stays resident in HBM: nobody touched the host array.
    e2e_steps = max(3, min(steps, 10))
    target = fg if runner is None else runner

    def e2e_step(i):
        if runner is None:
            fg.weight_value[0][0] = 0.1 + 1e-9 * (i & 1)
            fg.inference(0, 1, sample_evidence=True)
            return fg.marginals
        return runner.inference_e2e(1)

    _lib.check(L.nb_reset_counts(g))            # the timed sweeps tallied too; start the calls from zero
    e2e_step(0)
    e2e_step(1)
    dev.barrier()
    cudart.cudaProfilerStart()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        m = e2e_step(i)
    dev.barrier()
    e2e_dt = dev.max_over_ranks((time.perf_counter() - t0) / e2e_steps)
    cudart.cudaProfilerStop()
    e2e_extra = {}
    if runner is None:
        # the scalable read: compact tallies DMA-ed into pinned host memory, no host conversion
        fg.counts_compact()
        t0 = time.perf_counter()
        for i in range(e2e_steps):
            fg.weight_value[0][0] = 0.1 + 1e-9 * (i & 1)
            fg.inference(0, 1, sample_evidence=True)
            cc = fg.counts_compact()
        e2e_extra["compact_tallies_ms_per_step"] = 1e3 * (time.perf_counter() - t0) / e2e_steps
        e2e_extra["compact_tally_bytes"] = int(cc.nbytes)
        # the reference's round trip: the caller holds var_value / count (edits possible), so both are
        # uploaded on entry and refreshed on exit, as int64
        _ = fg.var_value, fg.count
        fg.inference(0, 1, sample_evidence=True)
        t0 = time.perf_counter()
        for i in range(e2e_steps):
            fg.inference(0, 1, sample_evidence=True)
            m = fg.marginals
        e2e_extra["state_roundtrip_ms_per_step"] = 1e3 * (time.perf_counter() - t0) / e2e_steps
    V, Wn = len(fg.variable), len(fg.weight)
    h2d = Wn * 8                                  # the float64 weights (changed every step)
    d2h = len(fg._count) * 1                      # cumulative tallies <= 255: 1 byte each (2 up to 65535 sweeps)

    c4 = learn = None
    if world == 1 and rank == 0:
        fg.clear()
        del dev
        if "c4" in workloads:
            try:
                c4 = block_c4(args, local_rank, dump)
            except Exception as exc:  # noqa: BLE001
                c4 = {"unavailable": "%s: %s" % (type(exc).__name__, exc)}
        if "c3" in workloads:
            try:
                learn = block_learn(args, local_rank, dump)
            except Exception as exc:  # noqa: BLE001
                learn = {"unavailable": "%s: %s" % (type(exc).__name__, exc)}

    c4s = None
    if world > 1 and "c4" in workloads:
        runner.close()
        try:
            c4s = block_c4_strong(args, rank, world, local_rank)
        except Exception as exc:  # noqa: BLE001
            c4s = {"unavailable": "%s: %s" % (type(exc).__name__, exc)}
            import traceback
            traceback.print_exc()

    if rank != 0:
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
            dist.destroy_process_group()
        return

    ms_per_step = dev_ms / steps
    total_edges, total_vars = edges * world, nvar * world
    value = total_edges * steps / (dev_ms * 1e-3)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64 energy accumulation (f32 weights in the 16-byte quads, f32 exp for the draw)", "data": "synthetic",
        "config": {"workload": "ising_%dx%d_equal_inference%s" % (rows * world, cols,
                                                                 "" if world == 1 else "_strips_of_%d_rows" % rows),
                   "variables": total_vars, "factor_edge_evals_per_sweep": total_edges,
                   "colors": info["n_colors"] if runner is None else runner.n_colors,
                   "l2_policy": "inputs larger than L2 (record stream + per-variable state %.0f MB vs 126 MB)"
                                % ((info["tt2_quads"] * 16 + nvar * 17) / 1e6),
                   "partition": "single GPU" if world == 1 else
                   ("row strips; per colour a boundary phase + NVLink halo push on a side stream, concurrent with "
                    "the interior phase" if runner.p2p and runner.split else "row strips, per-colour halo exchange")},
        "timed_ms": dev_ms,
        "var_samples_per_sec": total_vars * steps / (dev_ms * 1e-3),
        "roofline": roofline(bytes_sweep, ms_per_step, "k_gibbs_tt2 (PAIR rows, uniform slices: 4-byte records; one launch "
                             "per colour; duration = CUDA-event time of the timed sweeps / sweeps)",
                             "k_gibbs_tt2_bytes_per_sweep"),
        "gpu_launches": int(l1 - l0),
        "clocks": clocks.summary(),
        "e2e": dict({"value": total_edges / e2e_dt, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                     "d2h_bytes_per_step": int(d2h), "ms_per_step": 1e3 * e2e_dt,
                     "api": "weight_value[0][:] = w; FactorGraph.inference(0, 1); FactorGraph.marginals (float64) -- "
                            "var_value is HBM-resident (host array untouched since the last call)"}, **e2e_extra),
        "wall_ms_timed_region": 1e3 * wall,
    }
    if identical is not None:
        line["p2p_bit_identical"] = identical[0]
        line["p2p_transport"] = {"peer_stores": identical[1], "boundary_interior_split": identical[2]}
    if c4s is not None:
        line["c4_strong"] = c4s
    if c4 is not None:
        line["c4"] = c4
    if learn is not None:
        line["learn"] = learn
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baselines()
        if learn is not None and "unavailable" not in learn:
            learn["cpu_baseline"] = reference_child("learn")       # the reference's learnthread on the same model shape
    missing = []
    if dump is not None:
        write_dump(args.dump_outputs, dump)
        # a workload that failed wrote nothing: say so, rather than leave a comparison of fewer outputs
        missing = [name for name, blk in (("c4", c4), ("learn", learn)) if blk is not None and "unavailable" in blk]
        line["dump_outputs"] = {"dir": args.dump_outputs, "arrays": sorted(dump), "missing_workloads": missing}
    OUT.emit(json.dumps(line))
    if missing:
        sys.exit("--dump-outputs: no outputs of %s (the workload failed, see the JSON line)" % ", ".join(missing))
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


class _QuietStdout(object):
    """stdout carries exactly ONE JSON line: everything libraries print there while the benchmark
    runs (e.g. the "NCCL version ..." banner at communicator creation) is routed to stderr."""

    def __init__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)

    def emit(self, line):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        print(line)
        sys.stdout.flush()
        os.dup2(2, 1)


OUT = None


def main():
    global OUT
    OUT = _QuietStdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps of every workload")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workloads", default=os.environ.get("NB_BENCH_WORKLOADS", "c2,c4,c3"),
                    help="N = 1 only: extra blocks next to the c2 headline")
    ap.add_argument("--ref-grid", type=int, default=0, help="reference arm: force the grid size")
    ap.add_argument("--ref-mode", default="inference", choices=["inference", "single", "learn"],
                    help="reference arm: the headline inference line, or a bounded single-thread / learning sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the timed steps to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
