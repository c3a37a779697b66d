"""In-place edits of isEvidence / initialValue / isFixed (FactorGraph.update_variables /
update_weights, nb_update_variables / nb_update_weights_fixed).

An edited graph must be the graph a rebuild from the edited records produces: the same device
arrays (nb_graph_digest) and, from the same chains, bit-identical sweeps and learning.  The graphs
are the row-class fixtures of the Philox replay (test_sweep_replay._spec)."""
import ctypes as C
import os
import sys
import zlib

import numpy as np
import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.dirname(os.path.abspath(__file__))
for p in (REPO, HERE):
    if p not in sys.path:
        sys.path.insert(0, p)

from test_sweep_replay import _graph, _spec   # noqa: E402

SEED = 0x2468_ACE0_1357_9BDF
SPECS = ["pair_uniform", "pair_records", "fast", "cat", "gen_boolean", "gen_cat_empty", "warp", "wide_headers",
         "wide_card", "wide_card_thread", "wid_wide", "wid_pair_top", "wid_pair_alias"]
EDITS = ["query_to_evidence", "evidence_to_query", "initial_value", "fix", "unfix", "all"]


# ============================================================================ helpers
def _records(name):
    """(weight, variable, factor, fmap, vmap, factor_index), FactorGraph attributes."""
    import numbskull_b200 as nb
    g, attrs, _ = _spec(name)
    g = tuple(np.copy(x) if isinstance(x, np.ndarray) else x for x in g)
    ns = nb.NumbSkull(quiet=True)
    ns.loadFactorGraph(*g)
    fg = ns.factorGraphs[0]
    return (fg.weight, fg.variable, fg.factor, fg.fmap, fg.vmap, fg.factor_index), attrs


def _fg(records, attrs):
    """A FactorGraph over copies of the records (same seed and colour seed every time)."""
    import numbskull_b200 as nb
    ns = nb.NumbSkull(quiet=True)
    ns.loadFactorGraphRaw(*[np.copy(r) for r in records])
    fg = ns.factorGraphs[0]
    fg.seed = SEED
    for k, v in attrs.items():
        setattr(fg, k, v)
    return fg


def _recs_of(fg):
    return (fg.weight, fg.variable, fg.factor, fg.fmap, fg.vmap, fg.factor_index)


class Dev(object):
    """Chains, tallies and weights of one device graph through the C ABI."""

    def __init__(self, fg):
        from numbskull_b200 import _lib
        self.fg, self.L, self.lib = fg, _lib.lib(), _lib
        self.g = fg._device_graph()
        self.V, self.W = len(fg.variable), len(fg.weight)
        self.n_count = int(fg.cstart[-1])

    def chk(self, rc):
        self.lib.check(rc)

    def vals(self, chain):
        out = np.empty(self.V, np.int64)
        self.chk(self.L.nb_get_var_values(self.g, chain, self.lib.ptr(out)))
        return out

    def set_vals(self, chain, v):
        v = np.ascontiguousarray(v, np.int64)
        self.chk(self.L.nb_set_var_values(self.g, chain, self.lib.ptr(v)))

    def weights(self):
        out = np.empty(self.W, np.float64)
        self.chk(self.L.nb_get_weights(self.g, self.lib.ptr(out)))
        return out

    def set_weights(self, w):
        w = np.ascontiguousarray(w, np.float64)
        self.chk(self.L.nb_set_weights(self.g, self.lib.ptr(w)))

    def counts(self):
        out = np.zeros(self.n_count, np.int64)
        self.chk(self.L.nb_get_counts(self.g, self.lib.ptr(out), 0))
        return out

    def set_counts(self, c):
        c = np.ascontiguousarray(c, np.int64)
        self.chk(self.L.nb_set_counts(self.g, self.lib.ptr(c)))

    def state(self):
        return self.vals(0), self.vals(1), self.counts(), self.weights()

    def install(self, other):
        """Take over the chains, tallies and weights of `other`."""
        self.set_vals(0, other.vals(0))
        self.set_vals(1, other.vals(1))
        self.set_counts(other.counts())
        self.set_weights(other.weights())

    def epoch(self):
        e = C.c_int64(0)
        self.chk(self.L.nb_begin_epoch(self.g, C.byref(e)))
        return e.value

    def sweeps(self, n, sample_evidence):
        self.chk(self.L.nb_gibbs_sweeps(self.g, n, 0, int(sample_evidence), SEED))

    def learn(self, n, step=0.05, reg=2, lne=True):
        s = C.c_double(step)
        self.chk(self.L.nb_learn_sweeps(self.g, n, C.byref(s), 0.95, reg, 0.5, 3.0, int(lne), SEED, 0))

    def learn_cells(self, n_blocks, epoch, step=0.05, reg=1, lne=True):
        n_colors = self.fg.device_info()["n_colors"]
        for b in range(n_blocks):
            for c in range(n_colors):
                self.chk(self.L.nb_learn_color_phase(self.g, c, b, n_blocks, step, reg, 0.5, 3.0, int(lne), SEED, epoch))

    def blocks(self, step, lne):
        nb = C.c_int(0)
        self.chk(self.L.nb_learn_blocks(self.g, step, int(lne), 0, C.byref(nb)))
        return nb.value


def _same_state(a, b, what):
    for name, x, y in zip(("var_value", "var_value_evid", "count", "weights"), a.state(), b.state()):
        assert np.array_equal(x, y), (what, name, int(np.sum(x != y)))


def _edit(kind, records, rng):
    """update_variables / update_weights arguments of one edit kind."""
    variable, weight = records[1], records[0]
    V = len(variable)
    evid = variable["isEvidence"].astype(np.int64)
    card = variable["cardinality"].astype(np.int64)
    fixed = weight["isFixed"].astype(np.int64)
    var, wts = [], []
    if kind in ("query_to_evidence", "all") and (evid == 0).any():
        ids = np.nonzero(evid == 0)[0]
        ids = rng.choice(ids, max(1, len(ids) // 4), replace=False)
        var.append(dict(var_ids=ids, isEvidence=np.ones(len(ids), np.int8),
                        initialValue=rng.integers(0, 1 << 30, len(ids)) % card[ids]))
        now = evid.copy()
        now[ids] = 1
    else:
        now = evid
    if kind in ("evidence_to_query", "all") and (evid == 1).any():
        ids = np.nonzero(evid == 1)[0]
        ids = rng.choice(ids, max(1, len(ids) // 2), replace=False)
        var.append(dict(var_ids=ids, isEvidence=np.zeros(len(ids), np.int8)))
    if kind in ("initial_value", "all"):
        ids = rng.choice(np.nonzero(evid != 4)[0], max(1, V // 5), replace=False)
        x = rng.integers(0, 1 << 30, len(ids)) % card[ids]
        q = now[ids] != 1             # query variables may hold a value outside the domain: stored as 0
        m = q & (rng.random(len(ids)) < 0.3)
        x[m] = card[ids][m] + 3
        var.append(dict(var_ids=ids, initialValue=x))
    if kind in ("fix", "all") and (fixed == 0).any():
        ids = np.nonzero(fixed == 0)[0]
        # and the largest free id a factor uses: the one at a record field's limit in the wid_* graphs
        used = np.intersect1d(ids, records[2]["weightId"])
        ids = np.union1d(rng.choice(ids, max(1, len(ids) // 3), replace=False), used[-1:])
        wts.append(dict(weight_ids=ids, isFixed=np.ones(len(ids), np.uint8)))
    if kind in ("unfix", "all"):
        ids = np.nonzero(fixed == 1)[0]
        if len(ids) == 0:   # a graph whose weights are all free: fix some first (in the records of both graphs)
            ids = np.arange(min(3, len(fixed)))
            weight["isFixed"][ids] = 1
        wts.append(dict(weight_ids=ids, isFixed=np.zeros(len(ids), np.uint8)))
    return var, wts


def _apply(fg, var, wts):
    for kw in var:
        fg.update_variables(**kw)
    for kw in wts:
        fg.update_weights(**kw)


def _learn_modes(fg):
    return ("2",) if fg.device_info()["value_bytes"] == 2 else ("2", "1")


# ============================================================================ CPU
def test_update_before_the_device_graph_edits_only_the_records():
    records, attrs = _records("gen_card")
    fg = _fg(records, attrs)
    evid = fg.variable["isEvidence"].copy()
    q = np.nonzero(evid == 0)[0][:5]
    fg.update_variables(np.concatenate([q, q[:1]]), isEvidence=[1, 1, 1, 1, 1, 0],
                        initialValue=[0, 0, 0, 0, 0, 0])
    assert fg._g is None
    assert fg.variable["isEvidence"][q[0]] == 0                  # the last entry of a duplicated id wins
    assert (fg.variable["isEvidence"][q[1:]] == 1).all()
    assert (fg.variable["initialValue"][q] == 0).all()
    fg.update_weights([0, 1, 0], [1, 1, 0])
    assert fg._g is None and fg.weight["isFixed"][0] == 0 and fg.weight["isFixed"][1] == 1
    fg.update_variables(q[:2], value=[1, 0])
    assert fg._g is None
    assert fg.var_value[0][q[0]] == 1 and fg.var_value_evid[0][q[1]] == 0


def test_host_validation_without_a_device():
    records, attrs = _records("gen_card")
    fg = _fg(records, attrs)
    before = (fg.variable.copy(), fg.weight.copy())
    V = len(fg.variable)
    card = fg.variable["cardinality"].astype(np.int64)
    q = int(np.nonzero(fg.variable["isEvidence"] == 0)[0][0])
    with pytest.raises(ValueError, match="out of range"):
        fg.update_variables([0, V], isEvidence=[1, 1])
    with pytest.raises(ValueError, match="ghost"):
        fg.update_variables([q], isEvidence=[4])
    with pytest.raises(ValueError, match="initialValue outside"):
        fg.update_variables([q], isEvidence=[1], initialValue=[card[q]])
    with pytest.raises(ValueError, match="outside \\[0, cardinality\\)"):
        fg.update_variables([q], value=[-1])
    with pytest.raises(ValueError, match="out of range"):
        fg.update_weights([len(fg.weight)], [1])
    assert fg._g is None
    assert np.array_equal(fg.variable, before[0]) and np.array_equal(fg.weight, before[1])
    g = _graph(3, nvar=200, nfac=300, ghost_frac=0.1)
    import numbskull_b200 as nb
    ns = nb.NumbSkull(quiet=True)
    ns.loadFactorGraph(*g)
    fg = ns.factorGraphs[0]
    ghost = int(np.nonzero(fg.variable["isEvidence"] == 4)[0][0])
    with pytest.raises(ValueError, match="ghost"):
        fg.update_variables([ghost], initialValue=[0])


# ============================================================================ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("kind", EDITS)
@pytest.mark.parametrize("name", SPECS)
def test_edit_gives_the_rebuilt_graph(name, kind, monkeypatch):
    """A (built from R, then edited to R') against B (built from R'): same device arrays, and from
    the same chains bit-identical inference and learning."""
    records, attrs = _records(name)
    rng = np.random.default_rng(zlib.crc32((name + kind).encode()))
    records = tuple(np.copy(r) for r in records)
    var, wts = _edit(kind, records, rng)
    fa = _fg(records, attrs)
    a = Dev(fa)
    _apply(fa, var, wts)
    fb = _fg(_recs_of(fa), attrs)
    b = Dev(fb)
    assert fa.device_digest() == fb.device_digest()
    a.install(b)
    _same_state(a, b, "installed")
    for se in (False, True):
        a.sweeps(2, se)
        b.sweeps(2, se)
        _same_state(a, b, "inference sample_evidence=%s" % se)
    for mode in _learn_modes(fa):
        monkeypatch.setenv("NUMBSKULL_B200_LEARN_MODE", mode)
        for x in (a, b):
            x.learn(2)
        _same_state(a, b, "learning mode %s, default blocks" % mode)
        assert a.blocks(0.01, False) == b.blocks(0.01, False)
        ea, eb = a.epoch(), b.epoch()
        assert ea == eb
        for x in (a, b):
            x.learn_cells(3, ea, lne=False)
        _same_state(a, b, "learning mode %s, 3 blocks" % mode)


@pytest.mark.gpu
@pytest.mark.parametrize("name", SPECS)
def test_invalidate_after_edits_reproduces_the_graph(name):
    """update_* edit the records too: a rebuild from them is the graph the edits made."""
    records, attrs = _records(name)
    records = tuple(np.copy(r) for r in records)
    var, wts = _edit("all", records, np.random.default_rng(3))
    fa = _fg(records, attrs)
    Dev(fa)
    _apply(fa, var, wts)
    d = fa.device_digest()
    fa.invalidate()
    assert fa.device_digest() == d


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["pair_uniform", "fast", "cat", "warp", "wide_card"])
def test_edit_in_the_middle_of_a_run(name, monkeypatch):
    """Run A, edit it, install its state in B (built from the edited records, epoch counter
    advanced): both continue identically.  pair_uniform flips enough evidence to change the
    learning block count, which only a refreshed visit bound reports."""
    monkeypatch.setenv("NUMBSKULL_B200_LEARN_MODE", "2")
    records, attrs = _records(name)
    records = tuple(np.copy(r) for r in records)
    rng = np.random.default_rng(11)
    fa = _fg(records, attrs)
    a = Dev(fa)
    a.sweeps(3, False)
    a.learn(2)
    step = 0.002
    blocks_before = a.blocks(step, False)
    if name == "pair_uniform":   # every query variable becomes evidence: 5x the evidence visits
        q = np.nonzero(fa.variable["isEvidence"] == 0)[0]
        var = [dict(var_ids=q, isEvidence=np.ones(len(q), np.int8),
                    initialValue=rng.integers(0, 2, len(q)))]
        wts = []
    else:
        var, wts = _edit("all", _recs_of(fa), rng)
    _apply(fa, var, wts)
    fb = _fg(_recs_of(fa), attrs)
    b = Dev(fb)
    b.install(a)
    e = a.epoch()
    for _ in range(e + 1):
        b.epoch()
    assert a.blocks(step, False) == b.blocks(step, False)
    if name == "pair_uniform":
        assert a.blocks(step, False) != blocks_before
    for x in (a, b):
        x.sweeps(2, True)
    _same_state(a, b, "inference after the edit")
    for x in (a, b):
        x.learn(2, step=step, lne=False)
    _same_state(a, b, "learning after the edit")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["gen_cat_empty", "wide_card_thread"])
def test_value_writes_lazy_and_eager_mirrors(name):
    records, attrs = _records(name)
    rng = np.random.default_rng(5)
    V = len(records[1])
    card = records[1]["cardinality"].astype(np.int64)
    ids = rng.choice(np.nonzero(records[1]["isEvidence"] != 4)[0], V // 4, replace=False)
    val = rng.integers(0, 1 << 30, len(ids)) % card[ids]
    out = []
    for eager in (False, True):
        fg = _fg(records, attrs)
        fg.inference(0, 1)
        if eager:
            fg.var_value, fg.var_value_evid   # the caller now holds the arrays: uploaded on every call
        fg.update_variables(ids, value=val)
        for n in ("var_value", "var_value_evid"):   # (a lazy mirror stays lazy: read without exposing it)
            assert np.array_equal(fg._host(n, expose=eager)[0][ids], val), (eager, n)
        assert ("var_value" in fg._exposed) == eager
        fg.inference(0, 3)
        fg.learn(0, 1, 0.01, 0.95, 2, 0.5, 3.0)
        out.append((np.array(fg.var_value[0]), np.array(fg.var_value_evid[0]), np.array(fg.weight_value[0])))
    for x, y in zip(*out):
        assert np.array_equal(x, y)


@pytest.mark.gpu
def test_value_writes_with_the_bit_mirror(monkeypatch):
    """All-Boolean record graph: a value write goes to the bytes, and the bit mirror the sweeps
    gather from is rebuilt from them on entry to nb_gibbs_sweeps."""
    records, attrs = _records("fast")
    rng = np.random.default_rng(6)
    V = len(records[1])
    ids = rng.choice(V, V // 3, replace=False)
    val = rng.integers(0, 2, len(ids))
    out = []
    for mirror in ("0", "-1"):
        monkeypatch.setenv("NUMBSKULL_B200_BIT_MIRROR", mirror)
        fg = _fg(records, attrs)
        d = Dev(fg)
        d.sweeps(2, False)
        fg.update_variables(ids, value=val)
        assert np.array_equal(d.vals(0)[ids], val) and np.array_equal(d.vals(1)[ids], val)
        d.sweeps(3, False)
        out.append(d.state())
    for x, y in zip(*out):
        assert np.array_equal(x, y)


@pytest.mark.gpu
def test_set_var_values_follows_the_edited_evidence():
    records, attrs = _records("gen_card")
    fa = _fg(records, attrs)
    a = Dev(fa)
    card = fa.variable["cardinality"].astype(np.int64)
    q = int(np.nonzero((fa.variable["isEvidence"] == 0) & (card < 8))[0][0])
    e = int(np.nonzero((fa.variable["isEvidence"] == 1) & (card < 8))[0][0])
    fa.update_variables([q, e], isEvidence=[1, 0], initialValue=[0, 0])
    fb = _fg(_recs_of(fa), attrs)
    b = Dev(fb)
    for x in (a, b):
        v = x.vals(0)
        v[e] = card[e] + 1                   # now a query variable: mapped to 0, accepted
        x.set_vals(0, v)
        assert x.vals(0)[e] == 0
        v[q] = card[q] + 1                   # now evidence: refused
        with pytest.raises(ValueError, match="evidence variable"):
            x.set_vals(0, v)


@pytest.mark.gpu
def test_refused_edits_change_nothing():
    from numbskull_b200 import _lib
    g = _graph(21, dt0_cards=(2, 3), cat_frac=0.2, hubs=4, ghost_frac=0.05)
    import numbskull_b200 as nb
    ns = nb.NumbSkull(quiet=True)
    ns.loadFactorGraph(*g)
    fa = ns.factorGraphs[0]
    fa.seed, fa.warp_row_words = SEED, 40
    a = Dev(fa)
    a.sweeps(2, False)
    V = len(fa.variable)
    card = fa.variable["cardinality"].astype(np.int64)
    evid = fa.variable["isEvidence"]
    ghost = int(np.nonzero(evid == 4)[0][0])
    q = int(np.nonzero(evid == 0)[0][0])
    digest, state, recs = fa.device_digest(), a.state(), (fa.variable.copy(), fa.weight.copy())
    bad = [
        (dict(var_ids=[q, V], isEvidence=[1, 1], initialValue=[0, 0]), "out of range"),
        (dict(var_ids=[q, -1], value=[0, 0]), "out of range"),
        (dict(var_ids=[q], isEvidence=[4]), "ghost"),
        (dict(var_ids=[q, ghost], initialValue=[0, 0]), "ghost"),
        (dict(var_ids=[q], isEvidence=[1], initialValue=[card[q]]), "initialValue outside"),
        (dict(var_ids=[q, q], isEvidence=[0, 1], initialValue=[0, -1]), "initialValue outside"),
        (dict(var_ids=[q], value=[card[q]]), "outside \\[0, cardinality\\)"),
    ]
    L = _lib.lib()
    for kw, msg in bad:
        with pytest.raises(ValueError, match=msg):
            fa.update_variables(**kw)
        # the C entry point validates on its own
        ids = np.ascontiguousarray(kw["var_ids"], np.int64)
        cols = [None if kw.get(k) is None else np.ascontiguousarray(kw[k], t)
                for k, t in (("isEvidence", np.int8), ("initialValue", np.int64), ("value", np.int64))]
        with pytest.raises(ValueError, match=msg):
            _lib.check(L.nb_update_variables(a.g, _lib.ptr(ids), len(ids), *[_lib.ptr(c) for c in cols]))
    with pytest.raises(ValueError, match="out of range"):
        fa.update_weights([0, len(fa.weight)], [1, 1])
    w = np.array([len(fa.weight)], np.int64)
    with pytest.raises(ValueError, match="out of range"):
        _lib.check(L.nb_update_weights_fixed(a.g, _lib.ptr(w), 1, _lib.ptr(np.ones(1, np.uint8))))
    assert fa.device_digest() == digest
    for x, y in zip(state, a.state()):
        assert np.array_equal(x, y)
    assert np.array_equal(fa.variable, recs[0]) and np.array_equal(fa.weight, recs[1])
    # duplicates: the last entry wins, on the device as in the records
    fa.update_variables([q, q, q], isEvidence=[1, 1, 0], initialValue=[1, 0, 0])
    assert fa.variable["isEvidence"][q] == 0 and fa.variable["initialValue"][q] == 0
    w0 = int(fa.weight["isFixed"][0])
    fa.update_weights([0, 0], [1 - w0, w0])
    assert fa.weight["isFixed"][0] == w0
    ns2 = nb.NumbSkull(quiet=True)
    ns2.loadFactorGraphRaw(*[np.copy(r) for r in _recs_of(fa)])
    fb = ns2.factorGraphs[0]
    fb.seed, fb.warp_row_words = SEED, 40
    assert fa.device_digest() == fb.device_digest()


@pytest.mark.gpu
def test_unchanged_flags_launch_nothing():
    records, attrs = _records("fast")
    fa = _fg(records, attrs)
    d = Dev(fa)
    digest = fa.device_digest()
    fixed = fa.weight["isFixed"].astype(np.uint8)
    fa.update_weights(np.arange(len(fixed)), fixed)
    assert fa.device_digest() == digest
