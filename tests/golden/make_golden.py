#!/usr/bin/env python
"""Generate the golden fixtures in this directory from the REAL reference.

Needs a source checkout of HazyResearch/numbskull and numba:

    python tests/golden/make_golden.py <numbskull checkout>

The reference package is copied to a temp dir (its ``@jit(cache=True)``
functions write next to their sources, and the checkout may be read-only), the
missing ``past.builtins`` module is shimmed, and the unmodified numba functions
are called.  Nothing from the reference is stored in the repo -- only the
arrays it computes.  ``nthreads=1`` plus a jitted ``np.random.seed /
random.seed`` makes the reference bit-reproducible (SURVEY.md section 8c).

Fixtures (``*.npz``):
  truth_tables   eval_factor over every assignment, all 26 factor functions
  varmap_*       compute_var_map outputs (vmap, factor_index, vtf_offset)
  coin           reference test/ graph: raw file bytes, loaded arrays, results
  run_*          seeded learning + inference trajectories (count, values, weights)
  potentials_*   potential() for every (var, value) on a random state
"""
import os
import random
import shutil
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, REPO)

if len(sys.argv) != 2 or not os.path.isdir(os.path.join(sys.argv[1], "numbskull")):
    sys.exit("usage: python tests/golden/make_golden.py <numbskull checkout>")
REF = sys.argv[1]
tmp = tempfile.mkdtemp(prefix="nbref_")
shutil.copytree(os.path.join(REF, "numbskull"), os.path.join(tmp, "numbskull"))
os.makedirs(os.path.join(tmp, "past"))
open(os.path.join(tmp, "past", "__init__.py"), "w").close()
with open(os.path.join(tmp, "past", "builtins.py"), "w") as f:
    f.write("long = int\n")
sys.path.insert(0, tmp)

import numba  # noqa: E402
import numbskull  # noqa: E402  (the reference)
from numbskull import inference as ref_inf  # noqa: E402
from numbskull.dataloading import compute_var_map as ref_cvm  # noqa: E402
from numbskull.numbskulltypes import VarToFactor  # noqa: E402

from numbskull_b200 import synth  # noqa: E402


@numba.jit(nopython=True)
def seed_numba(s):
    np.random.seed(s)
    random.seed(s)


def save(name, **arrays):
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **arrays)
    print("wrote", path, {k: getattr(v, "shape", None) for k, v in arrays.items()})


def graph_arrays(fg):
    return dict(weight=fg.weight, variable=fg.variable, factor=fg.factor, fmap=fg.fmap,
                vmap=fg.vmap, factor_index=fg.factor_index)


def load(g, **opts):
    ns = numbskull.NumbSkull(quiet=True, nthreads=1, **opts)
    w, v, f, fm, dm, e = g
    ns.loadFactorGraph(w.copy(), v.copy(), f.copy(), fm.copy(), dm.copy(), e)
    return ns


# ---------------------------------------------------------------- truth tables
def truth_tables():
    out = {}
    for name, func in sorted(ref_inf.FACTORS.items(), key=lambda kv: kv[1]):
        for arity in (1, 2, 3):
            if func in (23, 24) and arity != 3:
                continue
            if func in (21, 22, 25, 26) and arity != 2:
                continue
            if func in (18, 19, 20) and arity != 1:
                continue
            for card in (2, 3):
                if func == 30 and card == 3:
                    continue  # UFO indexes members by value; keep it in range
                g = list(synth.random_graph(arity, 1, np.random.default_rng(1), funcs=(func,),
                                            max_arity=arity))
                w, v, f, fm, dm, e = g
                v["cardinality"] = card
                v["isEvidence"] = 0
                v["initialValue"] = 0
                f["arity"] = arity
                fm = np.zeros(arity, fm.dtype)
                fm["vid"] = np.arange(arity)
                fm["dense_equal_to"] = (np.arange(arity) + 1) % card
                ns = load((w, v, f, fm, np.zeros(arity, np.bool_), arity))
                fg = ns.factorGraphs[0]
                rows = []
                for state in np.ndindex(*([card] * arity)):
                    fg.var_value[0][:] = state
                    val = ref_inf.eval_factor(0, -1, 0, 0, fg.variable, fg.factor, fg.fmap,
                                              fg.var_value)
                    # and with each member as the sampled variable, forced to every value
                    forced = [ref_inf.eval_factor(0, m, k, 0, fg.variable, fg.factor, fg.fmap,
                                                  fg.var_value)
                              for m in range(arity) for k in range(card)]
                    rows.append(list(state) + [val] + forced)
                out["f%d_a%d_c%d" % (func, arity, card)] = np.array(rows, np.float64)
    save("truth_tables", **out)


# ------------------------------------------------------------ compute_var_map
def varmaps():
    rng = np.random.default_rng(7)
    cases = {
        "bool": synth.random_graph(40, 90, rng, allow_repeats=True),
        "cat": synth.random_graph(30, 80, rng, funcs=(12, 14, 15), card=4, categorical_frac=0.6,
                                  allow_repeats=True),
        "lf": synth.lf_model(6, 3, rng),
        "ising": synth.ising_grid(5, 7),
    }
    for name, g in cases.items():
        ns = load(g)
        fg = ns.factorGraphs[0]
        save("varmap_" + name, **graph_arrays(fg), domain_mask=g[4])
    # NOTE: the factors_to_skip path (numbskull.py:192-243) is not pinned: the
    # reference sizes factor_index without the skipped factors but
    # compute_var_map counts bucket lengths from ALL fmap entries
    # (dataloading.py:34-38), so its scatter writes out of bounds (observed
    # here: glibc "malloc(): invalid next size").


# ------------------------------------------------------------------ coin graph
def coin():
    _loadtxt = np.loadtxt

    def loadtxt4(*a, **k):  # graph.meta has 8 columns; numpy >= 1.23 wants usecols
        k.setdefault("usecols", (0, 1, 2, 3))
        return _loadtxt(*a, **k)

    np.loadtxt = loadtxt4
    try:
        ns = numbskull.numbskull.load([os.path.join(REF, "test"), "-l", "10", "-i", "10",
                                       "--quiet"])
    finally:
        np.loadtxt = _loadtxt
    fg = ns.factorGraphs[0]
    raw = {n: np.fromfile(os.path.join(REF, "test", "graph." + n), np.uint8)
           for n in ("meta", "weights", "variables", "factors")}
    arrays = {k: v.copy() for k, v in graph_arrays(fg).items()}
    seed_numba(1234)
    ns.learning(out=False)
    ns.inference(out=False)
    save("coin", **{"raw_" + k: v for k, v in raw.items()}, **arrays,
         weight_value=fg.weight_value.copy(), count=fg.count.copy(),
         var_value=fg.var_value.copy(), var_value_evid=fg.var_value_evid.copy(),
         marginals=fg.marginals.copy(), seed=np.int64(1234))


# ----------------------------------------------------------------- seeded runs
def runs():
    rng = np.random.default_rng(11)
    cases = {
        "bool_l2": (synth.random_graph(60, 120, rng, feature_values=True),
                    dict(n_learning_epoch=5, n_inference_epoch=20, stepsize=0.01, decay=0.95,
                         regularization=2, reg_param=0.01, burn_in=2, learn_non_evidence=False)),
        "bool_l1": (synth.random_graph(50, 100, rng),
                    dict(n_learning_epoch=6, n_inference_epoch=15, stepsize=0.02, decay=0.9,
                         regularization=1, reg_param=0.05, truncation=2, burn_in=0,
                         learn_non_evidence=True)),
        "cat": (synth.random_graph(40, 100, rng, funcs=(12, 14, 15), card=4,
                                   categorical_frac=0.7),
                dict(n_learning_epoch=4, n_inference_epoch=20, stepsize=0.01, decay=0.95,
                     regularization=2, reg_param=0.01, burn_in=1, learn_non_evidence=True)),
        "lf": (synth.lf_model(30, 4, rng),
               dict(n_learning_epoch=8, n_inference_epoch=10, stepsize=0.001, decay=0.9,
                    regularization=1, reg_param=0.01, burn_in=3, learn_non_evidence=True)),
        "ising": (synth.ising_grid(8, 8),
                  dict(n_learning_epoch=0, n_inference_epoch=50, burn_in=5)),
        "pairs": (synth.ising_pairs(100, rng=rng),
                  dict(n_learning_epoch=30, n_inference_epoch=5, stepsize=0.01, decay=0.95,
                       regularization=2, reg_param=0.01, burn_in=0)),
        "allfuncs": (synth.random_graph(30, 120, rng, max_arity=3,
                                        funcs=(-1, 0, 1, 2, 3, 4, 7, 8, 9, 18, 19, 20, 21, 22, 23,
                                               24, 25, 26), card=3),
                     dict(n_learning_epoch=3, n_inference_epoch=10, stepsize=0.01, decay=0.95,
                          regularization=2, reg_param=0.01, burn_in=0, learn_non_evidence=True)),
    }
    for name, (g, opts) in cases.items():
        seed = 4242
        ns = load(g, **opts)
        fg = ns.factorGraphs[0]
        arrays = {k: v.copy() for k, v in graph_arrays(fg).items()}
        pot = np.array([ref_inf.potential(v, k, 0, 0, fg.weight, fg.variable, fg.factor, fg.fmap,
                                          fg.vmap, fg.factor_index, fg.var_value, fg.weight_value)
                        for v in range(len(fg.variable))
                        for k in range(int(fg.variable[v]["cardinality"]))])
        seed_numba(seed)
        ns.learning(out=False)
        w_after_learn = fg.weight_value.copy()
        vv_after_learn = fg.var_value.copy()
        ve_after_learn = fg.var_value_evid.copy()
        ns.inference(out=False)
        save("run_" + name, **arrays, domain_mask=g[4], seed=np.int64(seed),
             opts=np.array(sorted(opts.items()), dtype=object).astype(str),
             potentials_initial=pot,
             weight_after_learn=w_after_learn, var_value_after_learn=vv_after_learn,
             var_value_evid_after_learn=ve_after_learn,
             count=fg.count.copy(), var_value=fg.var_value.copy(),
             marginals=fg.marginals.copy())


# --------------------------------------------------------------- RNG stream pin
def rng_stream():
    @numba.jit(nopython=True)
    def draw(s, n):
        np.random.seed(s)
        random.seed(s)
        a = np.empty(n)
        b = np.empty(n)
        for i in range(n):
            a[i] = np.random.rand()
            b[i] = random.random()
        return a, b

    a, b = draw(4242, 1500)
    save("rng_stream", np_rand=a, py_random=b, seed=np.int64(4242))


if __name__ == "__main__":
    rng_stream()
    truth_tables()
    varmaps()
    coin()
    runs()
    shutil.rmtree(tmp, ignore_errors=True)
