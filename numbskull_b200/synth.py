"""Synthetic factor graphs in the reference's record-array form.

Vectorised generators for the benchmark shapes named in BASELINE.json plus
small random graphs for the parity tests, and a writer for the DeepDive
binary ``graph.{meta,weights,variables,factors,domains}`` format (the role
``ising/ising.cpp:88-130`` plays in the reference).  Every generator returns
``(weight, variable, factor, fmap, domain_mask, edges)`` -- exactly the
positional arguments of ``NumbSkull.loadFactorGraph`` (numbskull.py:192).
"""
import os

import numpy as np

from .numbskulltypes import Weight, Variable, Factor, FactorToVar

FUNC = {
    "NOOP": -1, "IMPLY_NATURAL": 0, "OR": 1, "AND": 2, "EQUAL": 3, "ISTRUE": 4,
    "LINEAR": 7, "RATIO": 8, "LOGICAL": 9, "AND_CAT": 12, "IMPLY_MLN": 13,
    "OR_CAT": 14, "EQUAL_CAT_CONST": 15, "IMPLY_NATURAL_CAT": 16, "IMPLY_MLN_CAT": 17,
    "DP_GEN_CLASS_PRIOR": 18, "DP_GEN_LF_PRIOR": 19, "DP_GEN_LF_PROPENSITY": 20,
    "DP_GEN_LF_ACCURACY": 21, "DP_GEN_LF_CLASS_PROPENSITY": 22, "DP_GEN_DEP_FIXING": 23,
    "DP_GEN_DEP_REINFORCING": 24, "DP_GEN_DEP_EXCLUSIVE": 25, "DP_GEN_DEP_SIMILAR": 26,
    "UFO": 30,
}


def _pack(weight, variable, factor, fmap):
    domain_mask = np.zeros(len(variable), np.bool_)
    return weight, variable, factor, fmap, domain_mask, int(len(fmap))


def _variables(n, is_evidence=0, initial=0, data_type=0, cardinality=2):
    v = np.zeros(n, Variable)
    v["isEvidence"] = is_evidence
    v["initialValue"] = initial
    v["dataType"] = data_type
    v["cardinality"] = cardinality
    return v


def _factors(func, wid, arity, feature=1.0):
    f = np.zeros(len(arity), Factor)
    f["factorFunction"] = func
    f["weightId"] = wid
    f["featureValue"] = feature
    f["arity"] = arity
    off = np.zeros(len(arity), np.int64)
    if len(arity) > 1:
        np.cumsum(arity[:-1], out=off[1:])
    f["ftv_offset"] = off
    return f


def ising_grid(n, m, coupling=0.1, fixed=True):
    """n x m Boolean grid, EQUAL(3) factor to the up and the left neighbour,
    members in (self, neighbour) order, one shared weight: the shape of the
    commented block ``ising/ising.cpp:135-200`` (BASELINE config 2)."""
    weight = np.zeros(1, Weight)
    weight["isFixed"] = fixed
    weight["initialValue"] = coupling
    variable = _variables(n * m)

    ii, jj = np.divmod(np.arange(n * m, dtype=np.int64), m)
    has_up, has_left = ii != 0, jj != 0
    nf_cell = has_up.astype(np.int64) + has_left
    first = np.zeros(n * m, np.int64)
    np.cumsum(nf_cell[:-1], out=first[1:])
    nfac = int(nf_cell.sum())

    self_id = np.empty(nfac, np.int64)
    other = np.empty(nfac, np.int64)
    vid = np.arange(n * m, dtype=np.int64)
    up_slot = first[has_up]
    self_id[up_slot] = vid[has_up]
    other[up_slot] = vid[has_up] - m
    left_slot = first[has_left] + has_up[has_left]
    self_id[left_slot] = vid[has_left]
    other[left_slot] = vid[has_left] - 1

    factor = _factors(FUNC["EQUAL"], 0, np.full(nfac, 2, np.int64))
    fmap = np.zeros(2 * nfac, FactorToVar)
    fmap["vid"][0::2] = self_id
    fmap["vid"][1::2] = other
    return _pack(weight, variable, factor, fmap)


def ising_pairs(n_pairs, a=1.0, b=1.0, c=0.5, rng=None):
    """The active block of ``ising/ising.cpp:202-318``: evidence pairs drawn from
    p(x1,x2) ~ exp(+-a +-b +-c), factors ISTRUE(x1), ISTRUE(x2), EQUAL(x1,x2)
    with three learnable weights whose true values are (a, b, c)."""
    rng = rng or np.random.default_rng(0)
    z = np.exp(np.array([-a - b + c, -a + b - c, a - b - c, a + b + c]))
    idx = rng.choice(4, size=n_pairs, p=z / z.sum())
    weight = np.zeros(3, Weight)
    variable = _variables(2 * n_pairs, is_evidence=1)
    variable["initialValue"][0::2] = (idx >= 2)
    variable["initialValue"][1::2] = (idx % 2 == 1)
    func = np.tile(np.array([4, 4, 3], np.int16), n_pairs)
    wid = np.tile(np.array([0, 1, 2], np.int64), n_pairs)
    arity = np.tile(np.array([1, 1, 2], np.int64), n_pairs)
    factor = _factors(func, wid, arity)
    fmap = np.zeros(4 * n_pairs, FactorToVar)
    base = 2 * np.arange(n_pairs, dtype=np.int64)
    fmap["vid"][0::4] = base
    fmap["vid"][1::4] = base + 1
    fmap["vid"][2::4] = base
    fmap["vid"][3::4] = base + 1
    return _pack(weight, variable, factor, fmap)


def lf_model(copies, n_lf, rng=None, accuracy=None, abstain_prob=0.7, init_weight=1.0):
    """Data-programming generative model in the layout of
    ``test_lf_learning.py:22-126`` (BASELINE config 3): per candidate one
    Boolean query y and n_lf evidence labelling functions (dataType 0, card 3);
    DP_GEN_CLASS_PRIOR(18) on y with weight 0, DP_GEN_LF_ACCURACY(21) on
    (y, LF_i) with weight i+1.  LF values follow eval_factor's encoding
    (inference.py:321-332): 0 votes y=0, 1 votes y=1, 2 abstains."""
    rng = rng or np.random.default_rng(0)
    if accuracy is None:
        accuracy = rng.uniform(0.55, 0.95, n_lf)
    accuracy = np.asarray(accuracy, np.float64)
    weight = np.zeros(1 + n_lf, Weight)
    weight["initialValue"] = init_weight
    weight["initialValue"][0] = 0.0

    y = rng.integers(0, 2, copies)
    correct = rng.random((copies, n_lf)) < accuracy[None, :]
    votes = np.where(correct, y[:, None], 1 - y[:, None])
    lf = np.where(rng.random((copies, n_lf)) < abstain_prob, 2, votes)

    per = 1 + n_lf
    variable = _variables(copies * per)
    is_lf = (np.arange(copies * per) % per) != 0
    variable["isEvidence"][is_lf] = 1
    variable["cardinality"][is_lf] = 3
    variable["initialValue"][is_lf] = lf.reshape(-1)

    func = np.tile(np.concatenate(([18], np.full(n_lf, 21))).astype(np.int16), copies)
    wid = np.tile(np.arange(per, dtype=np.int64), copies)
    arity = np.tile(np.concatenate(([1], np.full(n_lf, 2))).astype(np.int64), copies)
    factor = _factors(func, wid, arity)

    epc = 1 + 2 * n_lf
    fmap = np.zeros(copies * epc, FactorToVar)
    yid = (np.arange(copies, dtype=np.int64) * per)
    vids = np.empty((copies, epc), np.int64)
    vids[:, 0] = yid
    vids[:, 1::2] = yid[:, None]
    vids[:, 2::2] = yid[:, None] + 1 + np.arange(n_lf, dtype=np.int64)[None, :]
    fmap["vid"] = vids.reshape(-1)
    return _pack(weight, variable, factor, fmap)


def _windowed_members(rng, nvar, anchors, extra, window, far_frac):
    """anchor + geometric-window offsets (local) or uniform (far) partners."""
    n = len(anchors)
    delta = rng.geometric(1.0 / max(2.0, window / 8.0), size=(n, extra)).astype(np.int64)
    delta = np.minimum(delta, window) * rng.choice(np.array([-1, 1]), size=(n, extra))
    local = np.mod(anchors[:, None] + delta, nvar)
    far = rng.integers(0, nvar, size=(n, extra))
    return np.where(rng.random((n, extra)) < far_frac, far, local)


def kbc(nvar, rng=None, n_weights=1 << 20, evidence_frac=0.1, window=1024, far_frac=0.2,
        hub_frac=0.001, fixed_frac=0.1, mix=(0.5, 0.5, 0.5)):
    """DeepDive KBC-style Boolean graph (BASELINE config 4): one ISTRUE(4) per
    variable plus mix[0]*nvar IMPLY_NATURAL(0) of arity 3, mix[1]*nvar AND(2) of
    arity 2 and mix[2]*nvar OR(1) of arity 3, i.e. 5 edges per variable at the
    default mix.  Members are an anchor and windowed / far partners; a
    ``hub_frac`` fraction of partner slots is redirected onto Zipf hubs.
    Weights are tied by hash(fid) mod n_weights."""
    rng = rng or np.random.default_rng(0)
    n_imp, n_and, n_or = (int(nvar * x) for x in mix)
    weight = np.zeros(n_weights, Weight)
    weight["isFixed"] = rng.random(n_weights) < fixed_frac
    weight["initialValue"] = rng.normal(0.0, 0.5, n_weights)
    variable = _variables(nvar)
    ev = rng.random(nvar) < evidence_frac
    variable["isEvidence"] = ev
    variable["initialValue"][ev] = rng.integers(0, 2, int(ev.sum()))

    nfac = nvar + n_imp + n_and + n_or
    func = np.concatenate((np.full(nvar, 4), np.full(n_imp, 0), np.full(n_and, 2),
                           np.full(n_or, 1))).astype(np.int16)
    arity = np.concatenate((np.full(nvar, 1), np.full(n_imp, 3), np.full(n_and, 2),
                            np.full(n_or, 3))).astype(np.int64)
    fid = np.arange(nfac, dtype=np.uint64)
    wid = ((fid * np.uint64(0x9E3779B97F4A7C15)) >> np.uint64(40)).astype(np.int64) % n_weights
    factor = _factors(func, wid, arity)

    parts = [np.arange(nvar, dtype=np.int64)]
    for cnt, ar in ((n_imp, 3), (n_and, 2), (n_or, 3)):
        anchors = rng.integers(0, nvar, cnt)
        others = _windowed_members(rng, nvar, anchors, ar - 1, window, far_frac)
        if hub_frac > 0:
            nhub = max(1, int(nvar * 1e-5))
            hubs = rng.integers(0, nvar, nhub)
            pick = np.minimum(rng.zipf(1.5, size=others.shape) - 1, nhub - 1)
            others = np.where(rng.random(others.shape) < hub_frac, hubs[pick], others)
        parts.append(np.concatenate((anchors[:, None], others), axis=1).reshape(-1))
    fmap = np.zeros(int(arity.sum()), FactorToVar)
    fmap["vid"] = np.concatenate(parts)
    return _pack(weight, variable, factor, fmap)


def kbc_fast(nvar, seed=1004, n_weights=1 << 20, evidence_frac=0.1, window=1024, far_frac=0.2,
             hub_frac=0.001, fixed_frac=0.1, mix=(0.5, 0.5, 0.5)):
    """Same shape as :func:`kbc`, generated by host threads in the library (``nb_synth_kbc``):
    counter-based randomness, so the graph depends on ``seed`` only.  The numpy generator needs
    minutes and tens of GB of temporaries at the BASELINE size (200 M variables / 1 B edges)."""
    from . import _lib
    n_imp, n_and, n_or = (int(nvar * x) for x in mix)
    weight = np.zeros(n_weights, Weight)
    variable = np.zeros(nvar, Variable)
    factor = np.zeros(nvar + n_imp + n_and + n_or, Factor)
    fmap = np.zeros(nvar + 3 * n_imp + 2 * n_and + 3 * n_or, FactorToVar)
    m3 = np.asarray(mix, np.float64)
    _lib.check(_lib.lib().nb_synth_kbc(nvar, seed, n_weights, evidence_frac, window, far_frac, hub_frac, fixed_frac,
                                       _lib.ptr(m3), _lib.ptr(weight), _lib.ptr(variable), _lib.ptr(factor),
                                       len(factor), _lib.ptr(fmap), len(fmap)))
    return _pack(weight, variable, factor, fmap)


def kbc_block(nvar, lo, hi, seed=1004, n_weights=1 << 20, evidence_frac=0.1, window=1024, far_frac=0.2,
              hub_frac=0.001, fixed_frac=0.1, mix=(0.5, 0.5, 0.5)):
    """Rank-local share of :func:`kbc_fast`'s graph for the owner block ``[lo, hi)``: every factor
    with a member in the block, owned variables first and the remote members as ghosts
    (``isEvidence = 4``) -- the dict :func:`numbskull_b200.partition.extract_local` returns, built
    without ever materialising the global graph (BASELINE config 4 across 8 GPUs)."""
    import ctypes as C
    from . import _lib
    L = _lib.lib()
    m3 = np.asarray(mix, np.float64)
    nf, ne = C.c_int64(0), C.c_int64(0)
    _lib.check(L.nb_synth_kbc_block(nvar, seed, n_weights, window, far_frac, hub_frac, _lib.ptr(m3), lo, hi,
                                    None, C.byref(nf), None, C.byref(ne)))
    factor = np.zeros(nf.value, Factor)
    fmap = np.zeros(ne.value, FactorToVar)
    _lib.check(L.nb_synth_kbc_block(nvar, seed, n_weights, window, far_frac, hub_frac, _lib.ptr(m3), lo, hi,
                                    _lib.ptr(factor), C.byref(nf), _lib.ptr(fmap), C.byref(ne)))
    # ghosts (ascending global id) and local member ids, by host threads (nb_block_ghosts)
    ng = C.c_int64(0)
    _lib.check(L.nb_block_ghosts(_lib.ptr(fmap), len(fmap), nvar, lo, hi, None, C.byref(ng), 0))
    ghosts = np.empty(ng.value, np.int64)
    _lib.check(L.nb_block_ghosts(_lib.ptr(fmap), len(fmap), nvar, lo, hi, _lib.ptr(ghosts), C.byref(ng), 1))
    n_owned = hi - lo
    global_vid = np.concatenate((np.arange(lo, hi, dtype=np.int64), ghosts))
    variable = np.zeros(len(global_vid), Variable)
    _lib.check(L.nb_synth_kbc_variables(seed, evidence_frac, _lib.ptr(global_vid), len(global_vid), _lib.ptr(variable)))
    variable["isEvidence"][n_owned:] = 4
    weight = np.zeros(n_weights, Weight)
    _lib.check(L.nb_synth_kbc_weights(seed, n_weights, fixed_frac, _lib.ptr(weight)))
    return dict(weight=weight, variable=variable, factor=factor, fmap=fmap,
                domain_mask=np.zeros(len(variable), np.bool_), global_vid=global_vid, n_owned=int(n_owned))


def categorical(nvar, card=16, factors_per_var=3, rng=None, n_weights=1 << 20,
                evidence_frac=0.2, window=1024, far_frac=0.2):
    """Categorical graph (BASELINE config 5): dataType 1 variables of
    cardinality ``card``, AND_CAT(12) factors of arity 2 with uniform
    ``dense_equal_to`` and windowed partners, tied learnable weights."""
    rng = rng or np.random.default_rng(0)
    weight = np.zeros(n_weights, Weight)
    weight["initialValue"] = rng.normal(0.0, 0.5, n_weights)
    variable = _variables(nvar, data_type=1, cardinality=card)
    ev = rng.random(nvar) < evidence_frac
    variable["isEvidence"] = ev
    variable["initialValue"] = rng.integers(0, card, nvar)
    nfac = nvar * factors_per_var
    anchors = rng.integers(0, nvar, nfac)
    others = _windowed_members(rng, nvar, anchors, 1, window, far_frac)[:, 0]
    others = np.where(others == anchors, (others + 1) % nvar, others)
    fid = np.arange(nfac, dtype=np.uint64)
    wid = ((fid * np.uint64(0x9E3779B97F4A7C15)) >> np.uint64(40)).astype(np.int64) % n_weights
    factor = _factors(FUNC["AND_CAT"], wid, np.full(nfac, 2, np.int64))
    fmap = np.zeros(2 * nfac, FactorToVar)
    fmap["vid"][0::2] = anchors
    fmap["vid"][1::2] = others
    fmap["dense_equal_to"] = rng.integers(0, card, 2 * nfac)
    return _pack(weight, variable, factor, fmap)


def wide_categorical(n_mentions, card=1000, cands=32, feats=4, couplings=4, rng=None, n_weights=1 << 12,
                     evidence_frac=0.2):
    """Entity-linking shape with cardinalities above 255 (2-byte device values): ``n_mentions``
    dataType 1 variables of cardinality ``card`` (a mention over its candidate entities), each with
    ``cands`` candidate values drawn from ``card``.  Every candidate c of a mention m has one
    EQUAL_CAT_CONST(15) prior (m == c) and ``feats`` AND_CAT(12) features (m == c and f == 1) on
    Boolean evidence variables f; ``couplings`` AND_CAT factors per mention tie it to another
    mention on a shared candidate (both == c).  Weights are tied into ``n_weights`` learnable
    ids; ``evidence_frac`` of the mentions are labelled with one of their candidates.  The values
    a mention takes outside its candidates sit in empty buckets.  Variables: mentions first, then
    ``n_mentions`` feature variables."""
    rng = rng or np.random.default_rng(0)
    M, F = int(n_mentions), int(n_mentions)
    weight = np.zeros(n_weights, Weight)
    weight["initialValue"] = rng.normal(0.0, 0.5, n_weights)
    variable = np.concatenate((_variables(M, data_type=1, cardinality=card), _variables(F, is_evidence=1)))
    variable["initialValue"][M:] = rng.integers(0, 2, F)
    cands = min(cands, card)
    # distinct candidates: evenly spaced values from a random start
    cand = np.sort((rng.integers(0, card, M)[:, None] + np.arange(cands) * (card // cands)) % card, axis=1)
    lab = rng.random(M) < evidence_frac
    variable["isEvidence"][:M] = lab
    variable["initialValue"][:M] = cand[np.arange(M), rng.integers(0, cands, M)]
    m_of = np.repeat(np.arange(M, dtype=np.int64), cands)
    c_of = cand.reshape(-1)
    slot = np.tile(np.arange(cands, dtype=np.int64), M)
    # priors: m == c
    n_pri = M * cands
    w_pri = (slot * 7 + c_of) % n_weights
    # features: m == c and f == 1
    n_feat = n_pri * feats
    fm_m = np.repeat(m_of, feats)
    fm_c = np.repeat(c_of, feats)
    fvar = M + rng.integers(0, F, n_feat)
    w_feat = (np.repeat(c_of, feats) * 131 + np.tile(np.arange(feats), n_pri) * 17 + 1) % n_weights
    # couplings: m == c and m' == c on a candidate c of m
    n_cpl = M * couplings
    a_m = np.repeat(np.arange(M, dtype=np.int64), couplings)
    a_c = cand[a_m, rng.integers(0, cands, n_cpl)]
    b_m = (a_m + rng.integers(1, max(M, 2), n_cpl)) % max(M, 1)
    w_cpl = np.full(n_cpl, n_weights - 1, np.int64)
    func = np.concatenate((np.full(n_pri, FUNC["EQUAL_CAT_CONST"]), np.full(n_feat + n_cpl, FUNC["AND_CAT"])))
    arity = np.concatenate((np.ones(n_pri, np.int64), np.full(n_feat + n_cpl, 2, np.int64)))
    factor = _factors(func, np.concatenate((w_pri, w_feat, w_cpl)), arity)
    fmap = np.zeros(n_pri + 2 * (n_feat + n_cpl), FactorToVar)
    fmap["vid"][:n_pri] = m_of
    fmap["dense_equal_to"][:n_pri] = c_of
    o = n_pri
    fmap["vid"][o:o + 2 * n_feat:2] = fm_m
    fmap["dense_equal_to"][o:o + 2 * n_feat:2] = fm_c
    fmap["vid"][o + 1:o + 2 * n_feat:2] = fvar
    fmap["dense_equal_to"][o + 1:o + 2 * n_feat:2] = 1
    o += 2 * n_feat
    fmap["vid"][o::2] = a_m
    fmap["vid"][o + 1::2] = b_m
    fmap["dense_equal_to"][o::2] = a_c
    fmap["dense_equal_to"][o + 1::2] = a_c
    return _pack(weight, variable, factor, fmap)


BOOLEAN_FUNCS = (0, 1, 2, 3, 4, 7, 8, 9)


def random_graph(nvar, nfac, rng=None, funcs=BOOLEAN_FUNCS, max_arity=4, n_weights=None,
                 evidence_frac=0.3, fixed_frac=0.3, allow_repeats=False, card=2,
                 categorical_frac=0.0, feature_values=False):
    """Small random graph for the parity tests.  Boolean functions draw
    members freely; AND_CAT/OR_CAT/EQUAL_CAT_CONST (12/14/15) get a uniform
    ``dense_equal_to``; DP functions (18-26) get their fixed arity.  With
    ``categorical_frac`` > 0 a share of the variables is dataType 1 with
    cardinality ``card``."""
    rng = rng or np.random.default_rng(0)
    n_weights = n_weights or max(1, nfac // 2)
    weight = np.zeros(n_weights, Weight)
    weight["isFixed"] = rng.random(n_weights) < fixed_frac
    weight["initialValue"] = rng.normal(0, 1.0, n_weights)
    variable = _variables(nvar)
    cat = rng.random(nvar) < categorical_frac
    variable["dataType"][cat] = 1
    variable["cardinality"][cat] = card
    ev = rng.random(nvar) < evidence_frac
    variable["isEvidence"] = ev
    variable["initialValue"] = rng.integers(0, 1 << 30, nvar) % variable["cardinality"]
    variable["initialValue"][~ev] = 0

    dp_arity = {18: 1, 19: 1, 20: 1, 21: 2, 22: 2, 23: 3, 24: 3, 25: 2, 26: 2}
    func = rng.choice(np.array(funcs), nfac).astype(np.int16)
    arity = rng.integers(1, max_arity + 1, nfac).astype(np.int64)
    for f, a in dp_arity.items():
        arity[func == f] = a
    arity[func == 4] = np.where(rng.random(int((func == 4).sum())) < 0.8, 1, arity[func == 4])
    if not allow_repeats:
        arity = np.minimum(arity, nvar)
    factor = _factors(func, rng.integers(0, n_weights, nfac), arity,
                      rng.choice([1.0, 0.5, 2.0], nfac) if feature_values else 1.0)
    fmap = np.zeros(int(arity.sum()), FactorToVar)
    vids = np.empty(len(fmap), np.int64)
    pos = 0
    for a in arity:
        vids[pos:pos + a] = rng.choice(nvar, int(a), replace=allow_repeats)
        pos += a
    fmap["vid"] = vids
    fmap["dense_equal_to"] = rng.integers(0, 1 << 30, len(fmap)) % variable["cardinality"][vids]
    return _pack(weight, variable, factor, fmap)


def write_deepdive(directory, weight, variable, factor, fmap, domains=None):
    """Write the big-endian DeepDive binary files that ``loadFGFromFile``
    parses (record formats: dataloading.py:103-237; writer counterpart
    ising/ising.cpp:88-130).  ``domains`` maps variable id -> sorted int64
    value list (graph.domains)."""
    os.makedirs(directory, exist_ok=True)
    nedges = int(factor["arity"].sum())
    with open(os.path.join(directory, "graph.meta"), "w") as f:
        f.write("%d,%d,%d,%d" % (len(weight), len(variable), len(factor), nedges))

    w = np.zeros(len(weight), np.dtype([("id", ">i8"), ("fixed", "u1"), ("init", ">f8")]))
    w["id"] = np.arange(len(weight))
    w["fixed"] = weight["isFixed"]
    w["init"] = weight["initialValue"]
    w.tofile(os.path.join(directory, "graph.weights"))

    v = np.zeros(len(variable), np.dtype([("id", ">i8"), ("ev", "i1"), ("init", ">i8"),
                                          ("dt", ">i2"), ("card", ">i8")]))
    v["id"] = np.arange(len(variable))
    v["ev"] = variable["isEvidence"]
    v["init"] = variable["initialValue"]
    v["dt"] = variable["dataType"]
    v["card"] = variable["cardinality"]
    v.tofile(os.path.join(directory, "graph.variables"))

    # variable-length factor records: int16 func, int64 arity, arity x (vid, eq), wid, feature
    arity = factor["arity"].astype(np.int64)
    rec_len = 10 + 16 * arity + 16
    start = np.zeros(len(factor), np.int64)
    if len(factor) > 1:
        np.cumsum(rec_len[:-1], out=start[1:])
    buf = np.zeros(int(rec_len.sum()), np.uint8)

    def put(offsets, values, dtype):
        raw = np.ascontiguousarray(values, dtype=dtype).view(np.uint8).reshape(len(offsets), -1)
        for b in range(raw.shape[1]):
            buf[offsets + b] = raw[:, b]

    put(start, factor["factorFunction"], ">i2")
    put(start + 2, arity, ">i8")
    owner = np.repeat(np.arange(len(factor)), arity)
    slot = np.arange(len(fmap)) - np.repeat(factor["ftv_offset"].astype(np.int64), arity)
    moff = start[owner] + 10 + 16 * slot
    vals = fmap["dense_equal_to"].astype(np.int64)
    if domains:
        vals = vals.copy()
        for vid, dom in domains.items():
            sel = fmap["vid"] == vid
            vals[sel] = np.asarray(dom, np.int64)[vals[sel]]
    put(moff, fmap["vid"], ">i8")
    put(moff + 8, vals, ">i8")
    put(start + 10 + 16 * arity, factor["weightId"], ">i8")
    put(start + 18 + 16 * arity, factor["featureValue"], ">f8")
    buf.tofile(os.path.join(directory, "graph.factors"))

    if domains:
        with open(os.path.join(directory, "graph.domains"), "wb") as f:
            for vid in sorted(domains):
                dom = np.asarray(domains[vid], np.int64)
                np.array([vid, len(dom)], ">i8").tofile(f)
                dom.astype(">i8").tofile(f)
