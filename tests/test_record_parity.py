"""Deterministic energy parity of the RECORD kernels (the ones bench.py runs).

``k_gibbs_tt2`` (PAIR rows), ``k_gibbs_tt`` (FAST rows) and ``k_gibbs_cat`` (CAT
rows) sample from energies they compute out of 8/16-byte truth-table and
categorical records.  ``nb_potentials_records`` evaluates the very device
functions those kernels call (``nb_tt2_delta`` / ``nb_tt_delta`` /
``nb_cat_energies``) for chosen variables; here they are compared with the
oracle's ``potential()`` (reference: numbskull/inference.py:55-71):

  * Boolean rows: ``e1 - e0`` against ``potential(v,1) - potential(v,0)``.
    PAIR records gather float64 weights: agreement to summation-order noise
    (1e-12).  FAST quads inline the weight as fp32: the same 1e-12 against the
    oracle run on the fp32-rounded weights, and the north-star bar (1e-5
    relative to the variable's energies) against the unrounded oracle;
  * categorical rows: every per-value energy, 1e-5 relative (fp32 sums).

Covered: every tabulated factor function with the sampled variable in every
member slot (repeated members included), arity 1-3, neighbour cardinality 2
and 3; every golden run of the numba reference; uniform PAIR slices (hoisted
table/weight word); 10^4 sampled variables of the full-size Ising grid and of
>= 10 M-variable KBC / categorical graphs.
"""
import itertools

import numpy as np
import pytest

from conftest import golden

pytestmark = pytest.mark.gpu

PAIR, FAST, CAT = 0, 1, 2
TT_FUNCS_ANY_ARITY = (-1, 0, 1, 2, 3, 4, 7, 9)
DP_ARITY = {18: 1, 19: 1, 20: 1, 21: 2, 22: 2, 23: 3, 24: 3, 25: 2, 26: 2}


def _fg(g, seed=1, **attrs):
    import numbskull_b200 as nb
    ns = nb.NumbSkull(quiet=True)
    ns.loadFactorGraph(*g)
    fg = ns.factorGraphs[0]
    fg.seed = seed
    for k, v in attrs.items():
        setattr(fg, k, v)
    return fg


def _oracle_of(oracle, fg):
    return oracle.OracleGraph(fg.weight.copy(), fg.variable.copy(), fg.factor.copy(), fg.fmap.copy(),
                              fg.vmap.copy(), fg.factor_index.copy(), nthreads=1, seed=0)


def _oracle_energies(og, ids, evid=False):
    """per requested variable: list of potential(v, k), k < cardinality"""
    card = og.variable["cardinality"]
    return [np.array([og.potential(int(v), k, evid) for k in range(int(card[v]))]) for v in ids]


def _offsets(fg, ids):
    cards = fg.variable["cardinality"][ids].astype(np.int64)
    return np.concatenate(([0], np.cumsum(cards)[:-1])), cards


def _check(fg, og, ids, evid=False, fp32_weights_exact=True, expect=None, only=None):
    """Compare nb_potentials_records with the oracle for the variables `ids`."""
    ids = np.asarray(ids, np.int64)
    got, cls = fg.potentials_records(ids, evid_chain=evid)
    offs, cards = _offsets(fg, ids)
    want = _oracle_energies(og, ids, evid)
    seen = {PAIR: 0, FAST: 0, CAT: 0}
    for i, v in enumerate(ids):
        e = want[i]
        scale = max(1.0, float(np.abs(e).max()))
        if only is not None and cls[i] not in only:
            continue
        if cls[i] in (PAIR, FAST):
            d = got[offs[i] + 1]
            assert got[offs[i]] == 0.0
            tol = 1e-12 * scale if (cls[i] == PAIR or fp32_weights_exact) else 1e-5 * float(np.abs(e).max()) + 1e-9
            assert abs(d - (e[1] - e[0])) <= tol, (int(v), int(cls[i]), d, e)
        elif cls[i] == CAT:
            g = got[offs[i]:offs[i] + cards[i]]
            assert np.all(np.abs(g - e) <= 1e-5 * np.maximum(np.abs(e), scale)), (int(v), g, e)
        else:
            assert np.isnan(got[offs[i]:offs[i] + cards[i]]).all()
            continue
        seen[int(cls[i])] += 1
    if expect:
        for c in expect:
            assert seen[c] > 0, (seen, expect)
    return seen


def _set_state(fg, og, state, evid_state=None, weights=None):
    fg.var_value[0][:] = state
    og.var_value[:] = state
    if evid_state is not None:
        fg.var_value_evid[0][:] = evid_state
        og.var_value_evid[:] = evid_state
    if weights is not None:
        fg.weight_value[0][:] = weights
        og.weight_value[:] = weights


# --------------------------------------------------------------------------- gadgets
def _boolean_gadgets():
    """One 3-variable gadget per (function, arity, slot -> variable map, cards of v1 / v2): a single
    factor with its own weight whose member slots are any of v0 (Boolean), v1, v2 -- repeated
    members included."""
    from numbskull_b200.numbskulltypes import Weight, Variable, Factor, FactorToVar
    specs = []
    for func in TT_FUNCS_ANY_ARITY:
        for arity in (1, 2, 3):
            specs += [(func, m) for m in itertools.product(range(3), repeat=arity)]
    for func, arity in DP_ARITY.items():
        specs += [(func, m) for m in itertools.product(range(3), repeat=arity)]
    gadgets = [(func, m, c1, c2) for func, m in specs for c1 in (2, 3) for c2 in (2, 3)]
    n = len(gadgets)
    rng = np.random.default_rng(11)
    weight = np.zeros(n, Weight)
    weight["initialValue"] = rng.normal(0, 1, n).astype(np.float32)      # fp32-representable
    weight["isFixed"] = rng.random(n) < 0.3
    variable = np.zeros(3 * n, Variable)
    variable["cardinality"] = 2
    factor = np.zeros(n, Factor)
    vids = []
    for i, (func, m, c1, c2) in enumerate(gadgets):
        variable["cardinality"][3 * i + 1] = c1
        variable["cardinality"][3 * i + 2] = c2
        factor[i] = (func, i, 1.0, len(m), len(vids))
        vids += [3 * i + s for s in m]
    variable["isEvidence"] = rng.random(3 * n) < 0.2
    fmap = np.zeros(len(vids), FactorToVar)
    fmap["vid"] = vids
    return (weight, variable, factor, fmap, np.zeros(3 * n, np.bool_), len(vids)), gadgets


def test_boolean_tables_every_function_slot_and_cardinality(oracle):
    g, gadgets = _boolean_gadgets()
    fg = _fg(g)
    og = _oracle_of(oracle, fg)
    card = fg.variable["cardinality"].astype(np.int64)
    ids = np.arange(len(card))
    total = {PAIR: 0, FAST: 0}
    for x0 in (0, 1):
        for x1 in range(3):
            for x2 in range(3):
                state = np.tile(np.array([x0, x1, x2], np.int64), len(gadgets)) % card
                _set_state(fg, og, state, evid_state=(state + 1) % card)
                for evid in (False, True):
                    seen = _check(fg, og, ids, evid=evid)
                    total[PAIR] += seen[PAIR]
                    total[FAST] += seen[FAST]
    assert total[PAIR] > 10000 and total[FAST] > 10000, total
    # the classes are what the sweep runs: every Boolean variable is a record row here
    _, cls = fg.potentials_records(ids)
    assert (cls[card == 2] <= FAST).all()
    fg.clear()


def test_categorical_records_every_slot(oracle):
    """AND_CAT / EQUAL_CAT_CONST gadgets (arity 1-3, cardinality 4): every slot map over three
    variables with random dense_equal_to -- the variable itself repeated with equal or different
    values, a neighbour repeated, a factor that can never fire."""
    from numbskull_b200.numbskulltypes import Weight, Variable, Factor, FactorToVar
    rng = np.random.default_rng(5)
    card = 4
    gadgets = [(func, m, rep) for func in (12, 15) for arity in (1, 2, 3)
               for m in itertools.product(range(3), repeat=arity) for rep in range(4)]
    n = len(gadgets)
    weight = np.zeros(n, Weight)
    weight["initialValue"] = rng.normal(0, 1, n)
    variable = np.zeros(3 * n, Variable)
    variable["dataType"] = 1
    variable["cardinality"] = card
    factor = np.zeros(n, Factor)
    vids, eqs = [], []
    for i, (func, m, rep) in enumerate(gadgets):
        factor[i] = (func, i, 1.0, len(m), len(vids))
        vids += [3 * i + s for s in m]
        eq = rng.integers(0, card, len(m))
        if rep % 2 == 0 and len(m) > 1:          # same dense_equal_to on every slot: a repeated variable can fire
            eq[:] = eq[0]
        eqs += eq.tolist()
    fmap = np.zeros(len(vids), FactorToVar)
    fmap["vid"], fmap["dense_equal_to"] = vids, eqs
    fg = _fg((weight, variable, factor, fmap, np.zeros(3 * n, np.bool_), len(vids)))
    og = _oracle_of(oracle, fg)
    ids = np.arange(3 * n)
    seen_total = 0
    for trial in range(12):
        state = rng.integers(0, card, 3 * n)
        _set_state(fg, og, state, weights=rng.normal(0, 1, n))
        seen_total += _check(fg, og, ids, expect=(CAT,))[CAT]
    assert seen_total > 10000
    fg.clear()


# --------------------------------------------------------------------------- reference golden runs
@pytest.mark.parametrize("name", ["bool_l2", "bool_l1", "cat", "lf", "ising", "pairs", "allfuncs"])
def test_record_energies_on_reference_golden_graphs(oracle, name):
    from numbskull_b200.factorgraph import FactorGraph
    z = golden("run_" + name)
    fg = FactorGraph(z["weight"].copy(), z["variable"].copy(), z["factor"].copy(), z["fmap"].copy(),
                     z["vmap"].copy(), z["factor_index"].copy(), 1, 1, 0, 1, device=0, seed=1)
    og = _oracle_of(oracle, fg)
    card = fg.variable["cardinality"].astype(np.int64)
    ids = np.arange(len(card))
    rng = np.random.default_rng(3)
    n_rec = 0
    for trial in range(4):
        state = rng.integers(0, 1 << 30, len(card)) % card
        w = rng.normal(size=len(fg.weight)).astype(np.float32).astype(np.float64)
        _set_state(fg, og, state, evid_state=state[::-1] % card, weights=w)
        for evid in (False, True):
            seen = _check(fg, og, ids, evid=evid)
            n_rec += sum(seen.values())
    _, cls = fg.potentials_records(ids)
    if name in ("bool_l2", "bool_l1", "ising", "pairs"):
        assert n_rec > 0 and (cls[(card == 2) & (fg.variable["dataType"] == 0)] <= FAST).any()
    fg.clear()


@pytest.mark.parametrize("name", ["wid_compact_top", "wid_wide", "wid_pair_top", "wid_pair_alias", "wid_fast",
                                  "wid_cat"])
def test_energies_at_the_weight_id_limits(oracle, name):
    """Graphs whose weight ids sit at the limits of the record fields (test_sweep_replay's wid_*
    graphs, tables of 2^20 to 2^22 + 512 weights): nb_potentials bit-exact, the record energies as
    on the golden graphs."""
    from test_sweep_replay import _spec
    g, attrs, _ = _spec(name)
    fg = _fg(g, **attrs)
    og = _oracle_of(oracle, fg)
    card = fg.variable["cardinality"].astype(np.int64)
    ids = np.arange(len(card))
    rng = np.random.default_rng(4)
    n_rec = 0
    for trial in range(3):
        state = rng.integers(0, 1 << 30, len(card)) % card
        w = rng.normal(size=len(fg.weight)).astype(np.float32).astype(np.float64)
        _set_state(fg, og, state, evid_state=state[::-1] % card, weights=w)
        for evid in (False, True):
            assert np.array_equal(fg.potentials(evid_chain=evid), og.energies(ids, evid)), "potential() parity"
            n_rec += sum(_check(fg, og, ids, evid=evid).values())
    assert n_rec > 0
    fg.clear()


def test_fp32_inlined_weights_meet_the_energy_bar(oracle):
    """FAST quads carry the weight as fp32: with weights that are NOT fp32-representable the
    difference to the float64 oracle stays within 1e-5 of the variable's energies."""
    from numbskull_b200 import synth
    g = synth.random_graph(4000, 9000, np.random.default_rng(8), funcs=(0, 1, 2, 3, 4, 7, 9), max_arity=3,
                           evidence_frac=0.2)
    fg = _fg(g)
    og = _oracle_of(oracle, fg)
    rng = np.random.default_rng(9)
    _set_state(fg, og, rng.integers(0, 2, 4000), weights=rng.normal(0, 1, len(fg.weight)) * np.pi)
    seen = _check(fg, og, np.arange(4000), fp32_weights_exact=False, expect=(FAST,))
    assert seen[FAST] > 1000
    # ... and the rounding is the ONLY difference: bit-level agreement on the rounded weights
    og.weight_value[:] = og.weight_value.astype(np.float32).astype(np.float64)
    # (FAST rows only: PAIR records gather the float64 weights themselves)
    _check(fg, og, np.arange(4000), fp32_weights_exact=True, expect=(FAST,), only=(FAST,))
    fg.clear()


def test_uniform_pair_slices_small_grid(oracle):
    """Tied (table, weight): the Ising grid stores bare member ids (4 per quad) with the common word
    hoisted per slice; a second grid with per-factor weights takes the 8-byte records."""
    from numbskull_b200 import synth
    rng = np.random.default_rng(2)
    for tied in (True, False):
        g = list(synth.ising_grid(48, 40, coupling=0.37))
        if not tied:
            from numbskull_b200.numbskulltypes import Weight
            nf = len(g[2])
            w = np.zeros(nf, Weight)
            w["initialValue"] = rng.normal(0, 1, nf)
            g[0] = w
            g[2]["weightId"] = np.arange(nf)
        fg = _fg(tuple(g))
        og = _oracle_of(oracle, fg)
        for trial in range(3):
            _set_state(fg, og, rng.integers(0, 2, 48 * 40))
            seen = _check(fg, og, np.arange(48 * 40), expect=(PAIR,))
            assert seen[PAIR] == 48 * 40
        fg.clear()


# --------------------------------------------------------------------------- BASELINE sizes, sampled
def _sampled(fg, og, rng, n=10000, **kw):
    ids = np.unique(rng.integers(0, len(fg.variable), n))
    return _check(fg, og, ids, **kw)


def test_full_size_ising_sampled_energies(oracle):
    """BASELINE config 2 at full size (4096 x 4096): 10^4 sampled variables, random state."""
    from numbskull_b200 import synth
    fg = _fg(synth.ising_grid(4096, 4096))
    og = _oracle_of(oracle, fg)
    rng = np.random.default_rng(1)
    _set_state(fg, og, rng.integers(0, 2, 4096 * 4096))
    seen = _sampled(fg, og, rng, expect=(PAIR,))
    assert seen[PAIR] > 9000
    fg.clear()


def test_kbc_10m_sampled_energies(oracle):
    """BASELINE config 4 shape at 10 M variables / 50 M edges: FAST (and PAIR) rows."""
    from numbskull_b200 import synth
    fg = _fg(synth.kbc(10_000_000, np.random.default_rng(1004)))
    og = _oracle_of(oracle, fg)
    rng = np.random.default_rng(4)
    w = fg.weight_value[0].astype(np.float32).astype(np.float64)
    _set_state(fg, og, rng.integers(0, 2, 10_000_000), weights=w)
    seen = _sampled(fg, og, rng, expect=(FAST,))
    assert seen[FAST] + seen[PAIR] > 9000
    fg.clear()


def test_categorical_10m_sampled_energies(oracle):
    """BASELINE config 5 shape at 10 M variables, cardinality 16: CAT rows."""
    from numbskull_b200 import synth
    fg = _fg(synth.categorical(10_000_000, 16, 3, np.random.default_rng(1005)))
    og = _oracle_of(oracle, fg)
    rng = np.random.default_rng(6)
    _set_state(fg, og, rng.integers(0, 16, 10_000_000))
    seen = _sampled(fg, og, rng, expect=(CAT,))
    assert seen[CAT] > 9000
    fg.clear()


def test_bit_mirror_gives_identical_chains(monkeypatch):
    """Large all-Boolean graphs read member values from a bit-packed mirror of the value array
    (nb_graph::d_valbits; on by default from 10^8 variables).  It only changes WHERE a value is read:
    forced on, the chains, tallies and marginals are bit-identical to the byte path -- on a KBC graph
    with evidence, PAIR and FAST rows and (row-length knob lowered) hub rows, with values written
    from the host between the calls."""
    import numbskull_b200 as nb
    from numbskull_b200 import synth
    g = synth.kbc_fast(200_000, seed=11, hub_frac=0.02)
    runs = []
    for mode in ("-1", "0"):
        monkeypatch.setenv("NUMBSKULL_B200_BIT_MIRROR", mode)
        ns = nb.NumbSkull(quiet=True)
        ns.loadFactorGraph(*g)
        fg = ns.factorGraphs[0]
        fg.seed, fg.warp_row_words = 5, 96
        fg.inference(2, 3, sample_evidence=False)
        a = fg.var_value[0].copy()
        m1 = fg.marginals.copy()
        info = fg.device_info()
        assert info["n_warp_rows"] > 0 and info["n_pair_rows"] > 0 and info["n_fast_rows"] > 0
        fg.var_value[0][::3] = 1 - fg.var_value[0][::3]           # host edit: the mirror is rebuilt per call
        fg.inference(0, 4, sample_evidence=True)
        runs.append((a, m1, fg.var_value[0].copy(), fg.marginals.copy(), fg.count.copy()))
        fg.clear()
    for x, y in zip(runs[0], runs[1]):
        assert np.array_equal(x, y)
