"""Graphs with cardinalities above 255: 2-byte device values.

A graph whose cardinalities are all <= 255 keeps 1-byte values; any cardinality above that
(up to 65535) makes the build store 2-byte values, keep the real cardinalities in ``d_vcard``
and run the 16-bit instantiations of the kernels.  Checked against the oracle (a C port of
numbskull's inference.py / learning.py): energies bit for bit, marginals against exact
conditionals and the oracle's sampler, learned weights within 3 sigma, the host mirrors, the
CLI, and the single-GPU restriction of the partitioner.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import REPO, golden

PAIR, FAST, CAT, GEN = 0, 1, 2, 3
CAT_FUNCS = (12, 14, 15, 16, 17)            # AND_CAT, OR_CAT, EQUAL_CAT_CONST, IMPLY_NATURAL_CAT, IMPLY_MLN_CAT
VALUE_FUNCS = (0, 1, 2, 3, 4, 7, 8, 9, 13)   # functions that compare or test member values


def _types():
    from numbskull_b200.numbskulltypes import Weight, Variable, Factor, FactorToVar
    return Weight, Variable, Factor, FactorToVar


def _fg(g, seed=1, **attrs):
    import numbskull_b200 as nb
    ns = nb.NumbSkull(quiet=True)
    ns.loadFactorGraph(*g)
    fg = ns.factorGraphs[0]
    fg.seed = seed
    for k, v in attrs.items():
        setattr(fg, k, v)
    return fg


def _oracle_of(oracle, fg, seed=0):
    return oracle.OracleGraph(fg.weight.copy(), fg.variable.copy(), fg.factor.copy(), fg.fmap.copy(),
                              fg.vmap.copy(), fg.factor_index.copy(), nthreads=1, seed=seed)


def _graph(variable, factors, n_weights, weights=None, fixed=True):
    """factors: list of (function, weight id, [(vid, dense_equal_to), ...])"""
    Weight, _, Factor, FactorToVar = _types()
    w = np.zeros(n_weights, Weight)
    w["isFixed"] = fixed
    w["initialValue"] = 0.0 if weights is None else weights
    f = np.zeros(len(factors), Factor)
    fm = np.zeros(sum(len(m) for _, _, m in factors), FactorToVar)
    pos = 0
    for i, (func, wid, members) in enumerate(factors):
        f[i] = (func, wid, 1.0, len(members), pos)
        for vid, eq in members:
            fm[pos] = (vid, eq)
            pos += 1
    return w, variable, f, fm, np.zeros(len(variable), np.bool_), len(fm)


def _variables(cards, dtypes, evid=None, init=None):
    _, Variable, _, _ = _types()
    v = np.zeros(len(cards), Variable)
    v["cardinality"] = cards
    v["dataType"] = dtypes
    if evid is not None:
        v["isEvidence"] = evid
    if init is not None:
        v["initialValue"] = init
    return v


def _mixed_random(rng, nvar=60, nfac=160, wide=300, small=7):
    """Boolean, small and wide variables of both data types; every function that takes
    categorical members, and value-comparing Boolean functions whose members may be wide."""
    from numbskull_b200 import synth
    g = synth.random_graph(nvar, nfac, rng, funcs=CAT_FUNCS + VALUE_FUNCS, max_arity=3, evidence_frac=0.3,
                           feature_values=True)
    w, v, f, fm, dm, e = g
    kind = rng.integers(0, 5, nvar)           # 0, 1: Boolean; 2: small cat; 3: wide cat; 4: wide dataType 0
    v["dataType"] = np.where((kind == 2) | (kind == 3), 1, 0)
    v["cardinality"] = np.select([kind == 2, kind >= 3], [small, wide], 2)
    v["initialValue"] = rng.integers(0, 1 << 30, nvar) % v["cardinality"]
    fm["dense_equal_to"] = rng.integers(0, 1 << 30, len(fm)) % v["cardinality"][fm["vid"]]
    # a share of the equal_to values of wide members lands high (>= 256)
    hi = (v["cardinality"][fm["vid"]] == wide) & (rng.random(len(fm)) < 0.5)
    fm["dense_equal_to"][hi] = 256 + rng.integers(0, wide - 256, int(hi.sum()))
    return w, v, f, fm, dm, e


def _random_state(rng, fg):
    card = fg.variable["cardinality"]
    s = rng.integers(0, 1 << 30, len(card)) % card
    hi = (card > 256) & (rng.random(len(card)) < 0.5)
    s[hi] = 256 + rng.integers(0, 1 << 30, int(hi.sum())) % (card[hi] - 256)
    return s


# --------------------------------------------------------------------------- build and limits
@pytest.mark.gpu
@pytest.mark.parametrize("card", [256, 300, 4097, 65535])
def test_wide_cardinalities_build_with_two_byte_values(card):
    v = _variables([2, card, card], [0, 1, 0], evid=[1, 0, 0], init=[1, 0, card - 1])
    fac = [(12, 0, [(1, card - 1), (0, 1)]), (15, 1, [(2, card - 2)]), (3, 2, [(1, 0), (2, 0)])]
    fg = _fg(_graph(v, fac, 3, weights=[0.5, -0.25, 1.0]))
    info = fg.device_info()
    assert info["value_bytes"] == 2
    assert info["count_entries"] == 2 * card + 1
    assert np.array_equal(fg.var_value[0], [1, 0, card - 1])


@pytest.mark.gpu
def test_cardinality_65536_is_rejected():
    v = _variables([2, 65536], [0, 0])
    fg = _fg(_graph(v, [(3, 0, [(0, 0), (1, 0)])], 1))
    with pytest.raises(ValueError, match=r"variable cardinality outside \[1, 65535\]"):
        fg.device_info()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["coin", "run_pairs", "run_cat", "run_allfuncs", "run_lf", "run_ising",
                                  "run_bool_l1", "run_bool_l2", "varmap_bool", "varmap_cat", "varmap_ising",
                                  "varmap_lf"])
def test_golden_graphs_keep_one_byte_values(name):
    from numbskull_b200.factorgraph import FactorGraph
    z = golden(name)
    fg = FactorGraph(z["weight"].copy(), z["variable"].copy(), z["factor"].copy(), z["fmap"].copy(),
                     z["vmap"].copy(), z["factor_index"].copy(), 1, 1, 0, 1, device=0, seed=1)
    assert fg.device_info()["value_bytes"] == 1


@pytest.mark.gpu
def test_tally_bound_fails_cleanly_on_wide_graphs():
    """65537 dataType-0 variables of cardinality 65535 need 65537 x 65535 > 2^32 tally slots: the
    build must refuse (the int64 host count array alone would be 34 GB, so this goes through the C ABI)."""
    import ctypes as C
    from numbskull_b200 import _lib
    from numbskull_b200.dataloading import assign_vtf_offsets
    from numbskull_b200.numbskulltypes import VarToFactor
    Weight, _, Factor, FactorToVar = _types()
    n = 65537
    variable = _variables(np.full(n, 65535), np.zeros(n))
    vmap = np.zeros(assign_vtf_offsets(variable), VarToFactor)
    weight, factor, fmap = np.zeros(1, Weight), np.zeros(0, Factor), np.zeros(0, FactorToVar)
    fi = np.zeros(0, np.int64)
    desc = _lib.GraphDesc(_lib.ptr(weight), 1, _lib.ptr(variable), n, _lib.ptr(factor), 0, _lib.ptr(fmap), 0,
                          _lib.ptr(vmap), len(vmap), _lib.ptr(fi), 0, 0, 0x5EED, None, 0, 0, None, 0)
    g = C.c_void_p()
    with pytest.raises(NotImplementedError, match="count array of .* entries unsupported"):
        _lib.check(_lib.lib().nb_graph_create(C.byref(desc), C.byref(g)))
    assert not g.value


# --------------------------------------------------------------------------- energies
@pytest.mark.gpu
@pytest.mark.parametrize("warp", [False, True])
def test_potentials_match_oracle_on_mixed_wide_graphs(oracle, warp):
    rng = np.random.default_rng(11 + warp)
    for trial in range(3):
        g = _mixed_random(rng)
        fg = _fg(g, warp_row_words=3 if warp else 0)
        info = fg.device_info()
        assert info["value_bytes"] == 2
        assert (info["n_warp_rows"] > 0) == warp
        og = _oracle_of(oracle, fg)
        for _ in range(2):
            s = _random_state(rng, fg)
            fg.var_value[0][:] = s
            fg.var_value_evid[0][:] = s[::-1] % fg.variable["cardinality"]
            og.var_value[:] = fg.var_value[0]
            og.var_value_evid[:] = fg.var_value_evid[0]
            assert (og.var_value >= 256).any()
            for evid in (False, True):
                got, want = fg.potentials(evid_chain=evid), og.potentials(evid)
                if warp:
                    assert np.allclose(got, want, rtol=1e-12, atol=1e-12), np.abs(got - want).max()
                else:     # thread rows walked in bucket order: the reference's sums bit for bit
                    assert np.array_equal(got, want), np.abs(got - want).max()


@pytest.mark.gpu
def test_record_rows_with_wide_members(oracle):
    """PAIR / FAST rows whose constant-compare factors have a wide member, a CAT row with a wide
    member whose dense_equal_to is < 256, and a CAT-shaped row whose wide member's dense_equal_to
    is >= 256 (8-bit records would truncate it to a value the member takes): classed GEN, exact."""
    W = 300
    # 0, 1: Boolean; 2: wide dataType 1; 3: wide dataType 0; 4, 5: categorical card 5
    v = _variables([2, 2, W, W, 5, 5], [0, 0, 1, 0, 1, 1], init=[1, 0, 261, 5, 2, 3])
    fac = [(2, 0, [(0, 0), (3, 0)]),                 # AND(Boolean, wide): PAIR row of 0
           (1, 1, [(0, 0), (2, 0)]), (4, 2, [(1, 0)]),
           (0, 3, [(1, 0), (2, 0), (3, 0)]),         # IMPLY_NATURAL: FAST row of 1 (two other members)
           (12, 4, [(4, 1), (2, 5)]),                # AND_CAT with the wide member at 5: CAT row of 4
           (15, 5, [(4, 3)]),
           (12, 6, [(5, 2), (3, 261)]),              # wide member at 261 = 5 + 256: row of 5 is GEN
           (12, 7, [(5, 0), (2, 261)])]
    g = _graph(v, fac, 8, weights=[0.5, -1.25, 0.75, 2.0, 1.5, -0.5, 3.0, 0.25])
    fg = _fg(g)
    og = _oracle_of(oracle, fg)
    ids = np.arange(6, dtype=np.int64)
    for state in ([1, 0, 261, 5, 2, 0], [0, 1, 5, 261, 1, 2], [1, 1, 299, 261, 2, 2]):
        fg.var_value[0][:] = state
        og.var_value[:] = state
        got, cls = fg.potentials_records(ids)
        cards = fg.variable["cardinality"]
        offs = np.concatenate(([0], np.cumsum(cards)[:-1]))
        assert list(cls) == [PAIR, FAST, GEN, GEN, CAT, GEN]
        for i in (0, 1):
            e0, e1 = og.potential(i, 0), og.potential(i, 1)
            assert abs(got[offs[i] + 1] - (e1 - e0)) <= 1e-6 * max(1.0, abs(e0), abs(e1))
        want4 = np.array([og.potential(4, k) for k in range(5)])
        assert np.allclose(got[offs[4]:offs[4] + 5], want4, rtol=1e-6, atol=1e-6)
        assert np.array_equal(fg.potentials(ids), og.potentials()), state


# --------------------------------------------------------------------------- marginals
def _one_wide_variable(card, dtype, seed):
    """A wide variable X next to a Boolean evidence variable E = 1: AND_CAT(X == c, E == 1) with
    weight w_c for 20 values c; every other value has energy 0 (empty buckets of a dataType-1 X)."""
    rng = np.random.default_rng(seed)
    vals = np.sort(rng.choice(card, 20, replace=False))
    w = rng.uniform(1.0, 4.0, 20)
    v = _variables([card, 2], [dtype, 0], evid=[0, 1], init=[0, 1])
    fac = [(12, i, [(0, int(c)), (1, 1)]) for i, c in enumerate(vals)]
    p = np.ones(card)
    p[vals] = np.exp(w)
    return _graph(v, fac, 20, weights=w), p / p.sum()


@pytest.mark.gpu
@pytest.mark.parametrize("card,dtype", [(1000, 1), (300, 0)])
@pytest.mark.parametrize("warp", [False, True])
def test_marginals_of_a_wide_variable_are_exact(card, dtype, warp):
    g, p = _one_wide_variable(card, dtype, seed=card + dtype)
    fg = _fg(g, seed=4, warp_row_words=3 if warp else 0)
    assert fg.device_info()["n_warp_rows"] == (2 if warp else 0)
    fg.inference(10, 50000, sample_evidence=False)
    m = fg.marginals[fg.cstart[0]:fg.cstart[0] + card]
    assert np.abs(m - p).max() < 0.01, (np.abs(m - p).max(), np.argmax(np.abs(m - p)))
    assert fg.var_value[0][1] == 1


@pytest.mark.gpu
@pytest.mark.parametrize("warp", [False, True])
def test_marginals_match_oracle_sampler(oracle, warp):
    from numbskull_b200 import synth
    g = synth.wide_categorical(4, card=260, cands=4, feats=1, couplings=1, rng=np.random.default_rng(7),
                               n_weights=8, evidence_frac=0.0)
    fg = _fg(g, seed=3, warp_row_words=3 if warp else 0)
    og = _oracle_of(oracle, fg, seed=5)
    epochs = 100000
    fg.inference(100, epochs, sample_evidence=False)
    og.inference(100, epochs, sample_evidence=False)
    d = np.abs(fg.marginals - og.marginals)
    assert d.max() < 0.01, (d.max(), np.argmax(d))


# --------------------------------------------------------------------------- learning
def _wide_learning_graph():
    from numbskull_b200 import synth
    return synth.wide_categorical(6, card=270, cands=4, feats=2, couplings=1, rng=np.random.default_rng(9),
                                  n_weights=12, evidence_frac=0.5)


@pytest.mark.gpu
@pytest.mark.parametrize("warp", [False, True])
def test_learned_weights_within_3_sigma_of_oracle(oracle, warp):
    g = _wide_learning_graph()
    args = (0, 200, 0.01, 0.99, 2, 0.01, 1)

    def run(x):
        x.learn(*args)
        return np.asarray(x.weight_value, np.float64).reshape(-1).copy()

    wg = np.array([run(_fg(g, seed=s, warp_row_words=3 if warp else 0)) for s in (1, 2, 3, 4, 5)])
    ref = _fg(g)
    wc = np.array([run(_oracle_of(oracle, ref, seed=s)) for s in (11, 12, 13, 14, 15)])
    mu, sd = wc.mean(0), wc.std(0, ddof=1)
    tol = 3.0 * np.sqrt(sd ** 2 + wg.std(0, ddof=1) ** 2 / 5 + sd ** 2 / 5) + 0.02
    assert (np.abs(wg.mean(0) - mu) <= tol).all(), (wg.mean(0), mu, tol)
    assert np.abs(wg[0] - g[0]["initialValue"]).max() > 0.01        # the weights did move


@pytest.mark.gpu
@pytest.mark.parametrize("warp", [False, True])
def test_learning_is_deterministic(warp):
    g = _wide_learning_graph()
    out = []
    for _ in range(2):
        fg = _fg(g, seed=8, warp_row_words=3 if warp else 0)
        fg.learn(2, 40, 0.01, 0.97, 2, 0.01, 1)
        out.append(np.asarray(fg.weight_value, np.float64).copy())
    assert np.array_equal(out[0], out[1])


@pytest.mark.gpu
def test_latency_mode_learning_is_refused(monkeypatch):
    fg = _fg(_wide_learning_graph(), seed=8)
    monkeypatch.setenv("NUMBSKULL_B200_LEARN_MODE", "1")
    with pytest.raises(NotImplementedError, match="throughput mode"):
        fg.learn(0, 2, 0.01, 0.97, 2, 0.01, 1)
    monkeypatch.setenv("NUMBSKULL_B200_LEARN_MODE", "2")
    fg.learn(0, 2, 0.01, 0.97, 2, 0.01, 1)


# --------------------------------------------------------------------------- host mirrors
@pytest.mark.gpu
def test_wide_values_round_trip_through_the_host_mirrors():
    v = _variables([2, 4097, 300, 65535], [0, 1, 0, 1], evid=[0, 1, 0, 0], init=[1, 4000, 299, 65534])
    fac = [(12, 0, [(1, 4000), (3, 65534)]), (3, 1, [(0, 0), (2, 0)])]
    fg = _fg(_graph(v, fac, 2, weights=[1.0, 0.5]))
    assert np.array_equal(fg.var_value[0], [1, 4000, 299, 65534])          # initial values, built on device
    state = np.array([0, 4096, 256, 65000])
    fg.var_value[0][:] = state
    fg.potentials()                                                        # uploads the edited mirror
    fg._stale.add("var_value")                                             # ... and reads it back
    assert np.array_equal(fg.var_value[0], state)
    fg.inference(0, 5, sample_evidence=False)
    got = fg.var_value[0]
    assert got[1] == 4096 and (got < fg.variable["cardinality"]).all()    # evidence kept, samples in range
    bad = state.copy()
    bad[1] = 4097                                                          # evidence value >= its cardinality
    fg.var_value[0][:] = bad
    with pytest.raises(ValueError):
        fg.potentials()
    ok = state.copy()
    ok[3] = 70000                                                          # non-evidence, out of range: becomes 0
    fg.var_value[0][:] = ok
    fg.potentials()
    fg._stale.add("var_value")
    assert np.array_equal(fg.var_value[0], [0, 4096, 256, 0])


# --------------------------------------------------------------------------- end to end
@pytest.mark.gpu
def test_cli_runs_a_wide_deepdive_graph(tmp_path):
    from numbskull_b200 import synth
    w, v, f, fm, dm, e = synth.wide_categorical(30, card=500, cands=6, feats=2, couplings=2,
                                                rng=np.random.default_rng(2), n_weights=32)
    synth.write_deepdive(str(tmp_path), w, v, f, fm)
    env = dict(os.environ, PYTHONPATH=REPO + os.pathsep + os.environ.get("PYTHONPATH", ""))
    r = subprocess.run([sys.executable, "-c", "from numbskull_b200.numbskull import main; main()", str(tmp_path),
                        "-l", "5", "-i", "20", "-o", str(tmp_path), "-q"], env=env, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = (tmp_path / "inference_result.out.text").read_text().strip().split("\n")
    per_var = np.where(v["cardinality"] == 2, 1, v["cardinality"])     # Boolean variables: one line
    assert len(lines) == int(per_var.sum())
    assert [int(x.split()[0]) for x in lines[:500]] == [0] * 500
    assert float(lines[0].split()[2]) >= 0.0


# --------------------------------------------------------------------------- partitioning
def test_partitioning_a_wide_graph_is_refused():
    from numbskull_b200 import synth
    from numbskull_b200.partition import partition_graph
    w, v, f, fm, dm, e = synth.wide_categorical(8, card=300, rng=np.random.default_rng(1))
    with pytest.raises(ValueError, match="cardinalities above 255 are single-GPU only"):
        partition_graph(w, v, f, fm, 0, 2, 0, 1)
