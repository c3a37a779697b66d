"""Every Gibbs draw and learning update, replayed on the host in float64.

The library's draws are deterministic functions of public state: the uniform of a variable depends
only on (global id, epoch, seed, stream tag), and its energies on the chain values and weights
before the colour phase that samples it.  The oracle restates the Philox streams, the decision rule
of every row class and the learning update independently (oracle/nb_oracle.c, no CUDA header
included), so these tests can say "this variable, in this sweep, must take this value":

  * Gibbs, one colour phase at a time (``nb_gibbs_color_phase``): the replay is teacher-forced
    with the GPU's own state before the phase, so one disagreement cannot cascade; the value of
    every sampled variable, the unchanged values of everything else and the exact tally deltas;
  * whole sweeps (``nb_gibbs_sweeps``, stream fan-out on and off, bit mirror forced on): each
    colour replayed from the before / after states of the sweep;
  * learning, one (block, colour) cell at a time (``nb_learn_color_phase``, both execution
    modes): both chains, the truncation draws, the fixed-point gradient sums, the visit counts and
    the closed-form weight update.
  * large learning cells: whole colours sized from the SM count, so that the branches only large
    cells take (SELL slices, several rows per warp or thread, long rows) are replayed too;
    ``learn_branches`` asserts which branch each cell takes.

Tolerance, the same everywhere: the GPU may pick differently from the float64 replay only where
the replay's decision margin (distance of the uniform to the nearest point that changes the pick)
is below NEAR_TIE -- the fp32 exp / CDFs / inlined weights of the kernels.  Such near-ties are
counted, printed, and must stay below 1e-4 of the draws.

The Philox known answers and the comparison with the library's own host-callable Philox
functions (compiled from its header by nvcc into a temporary directory) run without a GPU.
"""
import math
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

import oracle                          # noqa: E402
from oracle import rng as R            # noqa: E402

NEAR_TIE = 1e-5
MAX_TIE_RATE = 1e-4
SEED = 0x1234_5678_9ABC_DEF1
EPOCHS = (1, 2, (1 << 32) + 5, (1 << 40) + 1)
CLASS_NAMES = ("PAIR", "FAST", "CAT", "GEN", "WARP", "WIDE")


# =========================================================================== CPU: the streams
KNOWN_4x32 = [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
]
KNOWN_2x32 = [
    ((0, 0), 0, (0xff1dae59, 0x6cd10df2)),
    ((0x243f6a88, 0x85a308d3), 0x13198a2e, (0xdd7ce038, 0xf62a4c12)),
    ((0xffffffff,) * 2, 0xffffffff, (0x2c3f628b, 0xab4fd7ad)),
]


@pytest.mark.parametrize("ctr,key,want", KNOWN_4x32)
def test_philox4x32_known_answers(ctr, key, want):
    assert tuple(R.philox4x32(ctr, key)) == want


@pytest.mark.parametrize("ctr,key,want", KNOWN_2x32)
def test_philox2x32_known_answers(ctr, key, want):
    assert tuple(R.philox2x32(ctr, key)) == want


def test_stream_word_order_and_uniforms():
    """The multi-draw stream reads the four words of Philox4x32(id, epoch_lo, epoch_hi | tag << 24,
    block; seed) in order, then the next block; next() = u53(first word, second word)."""
    rid, epoch, tag, seed = 0x89ABCDEF, (0x1234 << 32) | 77, 2, 0x0123456789ABCDEF
    ctr = [rid, 77, 0x1234 | (tag << 24)]
    key = [seed & 0xFFFFFFFF, seed >> 32]
    want = R.philox4x32(ctr + [0], key) + R.philox4x32(ctr + [1], key)
    s = R.Stream(rid, epoch, tag, seed)
    assert [s.word() for _ in range(8)] == want
    s = R.Stream(rid, epoch, tag, seed)
    assert s.next() == (((want[0] << 32) | want[1]) >> 11) / 2.0 ** 53
    assert s.next32() == (want[2] + 0.5) / 2.0 ** 32
    assert R.u53(0xFFFFFFFF, 0xFFFFFFFF) == 1.0 - 2.0 ** -53 and R.u53(0, 0x7FF) == 0.0
    # the record rows' single draw: counter (id, epoch_lo), key folded from seed, epoch_hi and tag
    w = R.philox2x32([rid, 77], R.fold_key(seed, epoch, tag))
    assert R.philox2x32_u53(rid, epoch, seed, tag) == R.u53(w[0], w[1])
    assert R.fold_key(seed, epoch, 0) != R.fold_key(seed, epoch & 0xFFFFFFFF, 0)


def test_draw_rules_and_margins():
    # Boolean: P(0) = 1 / (1 + e^(e1 - e0))
    p0 = 1.0 / (1.0 + np.exp(0.7))
    assert R.draw_bool(0.0, 0.7, p0 - 1e-3) == (0, pytest.approx(1e-3))
    assert R.draw_bool(0.0, 0.7, p0 + 1e-3)[0] == 1
    # inverse CDF: first k whose cumulative mass reaches u
    e = np.log([1.0, 2.0, 3.0, 4.0])
    assert R.draw_cdf(e, 0.05) == (0, pytest.approx(0.05))
    assert R.draw_cdf(e, 0.31)[0] == 2 and R.draw_cdf(e, 0.99)[0] == 3
    # reservoir with an empty group: the empty values are picked by a second uniform, ascending
    s = R.Stream(5, 9, 0, 3)
    nonempty = np.array([0, 1, 0, 0, 1, 0], np.uint8)
    e = np.array([0.0, -50.0, 0.0, 0.0, -50.0, 0.0])      # the empty group (4 values) takes the pick
    pick, margin = R.draw_reservoir(e, s, nonempty)
    t = R.Stream(5, 9, 0, 3)
    u = [t.next32() for _ in range(4)]         # values 1 and 4, the empty group, then the pick inside it
    j = min(3, int(u[3] * 4))
    assert pick == [0, 2, 3, 5][j]
    assert margin > 0


def _nvcc():
    for c in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    return None


SHIM = r"""
#include <cstdio>
#include <cstring>
#include "nb_eval.cuh"
int main()
{
    char op[8];
    while (scanf("%7s", op) == 1) {
        if (!strcmp(op, "P4")) {
            unsigned c0, c1, c2, c3; unsigned long long seed; uint32_t o[4];
            if (scanf("%u %u %u %u %llu", &c0, &c1, &c2, &c3, &seed) != 5) return 1;
            nb_philox4x32(c0, c1, c2, c3, seed, o);
            printf("%u %u %u %u\n", o[0], o[1], o[2], o[3]);
        } else if (!strcmp(op, "P2")) {
            unsigned c0, c1, key;
            if (scanf("%u %u %u", &c0, &c1, &key) != 3) return 1;
            double u = nb_philox2x32_u53(c0, c1, key);
            unsigned long long bits; memcpy(&bits, &u, 8);
            printf("%llu\n", bits);
        } else if (!strcmp(op, "FK")) {
            unsigned long long seed, epoch; unsigned tag;
            if (scanf("%llu %llu %u", &seed, &epoch, &tag) != 3) return 1;
            printf("%u\n", nb_fold_key(seed, epoch, tag));
        } else return 1;
    }
    return 0;
}
"""


@pytest.fixture(scope="module")
def philox_shim(tmp_path_factory):
    """The library's own __host__ __device__ Philox functions, compiled for the host by nvcc."""
    nvcc = _nvcc()
    if nvcc is None:
        pytest.skip("nvcc not available")
    d = tmp_path_factory.mktemp("philox_shim")
    src, exe = d / "shim.cu", d / "shim"
    src.write_text(SHIM)
    csrc = os.path.join(REPO, "numbskull_b200", "csrc")
    subprocess.run([nvcc, "-std=c++17", "-O1", "-I", csrc, str(src), "-o", str(exe)], check=True,
                   stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
    return str(exe)


def test_host_restatement_matches_the_library_philox(philox_shim):
    rng = np.random.default_rng(2024)
    n = 400
    u32 = lambda: rng.integers(0, 1 << 32, n, dtype=np.uint64)      # noqa: E731
    c = [u32() for _ in range(4)]
    c[0][:100] |= np.uint64(1 << 31)                                  # ids >= 2^31
    seed = rng.integers(0, 1 << 63, n, dtype=np.uint64) * np.uint64(2) + np.uint64(1)
    epoch = rng.integers(0, 1 << 62, n, dtype=np.uint64)
    epoch[:50] = (np.uint64(1) << np.uint64(32)) + np.arange(50, dtype=np.uint64)   # just above 2^32
    epoch[50:60] = (np.uint64(1) << np.uint64(40)) + np.uint64(1)
    tag = rng.integers(0, 3, n)
    lines = []
    for i in range(n):
        lines.append("P4 %d %d %d %d %d" % (c[0][i], c[1][i], c[2][i], c[3][i], seed[i]))
        lines.append("P2 %d %d %d" % (c[0][i], c[1][i], c[2][i]))
        lines.append("FK %d %d %d" % (seed[i], epoch[i], tag[i]))
    out = subprocess.run([philox_shim], input="\n".join(lines) + "\n", stdout=subprocess.PIPE, text=True,
                         check=True).stdout.split("\n")
    for i in range(n):
        s = int(seed[i])
        want4 = R.philox4x32([int(c[k][i]) for k in range(4)], [s & 0xFFFFFFFF, s >> 32])
        assert [int(x) for x in out[3 * i].split()] == want4, i
        w2 = R.philox2x32([int(c[0][i]), int(c[1][i])], int(c[2][i]))
        got = np.array([int(out[3 * i + 1])], np.uint64).view(np.float64)[0]
        assert got == R.u53(w2[0], w2[1]), i
        assert int(out[3 * i + 2]) == R.fold_key(s, int(epoch[i]), int(tag[i])), i


# =========================================================================== GPU: graphs
def _graph(seed, nvar=3000, nfac=6000, cat_frac=0.0, cat_cards=(6, 12), cat_card_set=None, dt0_cards=(2,),
           funcs0=(0, 1, 2, 3, 4, 7, 9), funcs1=(12, 14, 15), max_arity=4, hubs=0, hub_degree=150, hub_rows=(),
           evidence_frac=0.3, ghost_frac=0.0, fixed_frac=0.2, n_weights=None, w_scale=1.0, feature_values=False,
           wide_arity=0, ratio=False):
    """Random graph for the replay.  dataType-0 variables (cardinalities from dt0_cards) share
    factors of funcs0 (plus RATIO if `ratio`); dataType-1 variables (cardinalities in the range
    cat_cards, or from cat_card_set) factors of funcs1 with dense_equal_to below each member's
    cardinality.  `hubs` variables get `hub_degree` extra pairwise factors each (long rows: warp
    path with several tasks).  Each (dataType, cardinality, incidences) of `hub_rows` makes one more
    hub, a free variable of that type and cardinality with exactly that many incidences; a
    categorical one of these leaves a fifth of its values without incidences (empty buckets)."""
    from numbskull_b200.numbskulltypes import Weight, Variable, Factor, FactorToVar
    rng = np.random.default_rng(seed)
    variable = np.zeros(nvar, Variable)
    cat = rng.random(nvar) < cat_frac
    card = rng.choice(np.array(dt0_cards), nvar)
    if cat_card_set is None:
        card[cat] = rng.integers(cat_cards[0], cat_cards[1] + 1, int(cat.sum()))
    else:
        card[cat] = rng.choice(np.array(cat_card_set), int(cat.sum()))
    hub_dtype = np.array([h[0] for h in hub_rows], bool)
    rows = np.zeros(len(hub_rows), np.int64)                 # the hub_rows variables
    for want in (False, True):
        if (hub_dtype == want).any():
            rows[hub_dtype == want] = rng.choice(np.nonzero(cat == want)[0], int((hub_dtype == want).sum()),
                                                 replace=False)
    card[rows] = [h[1] for h in hub_rows]
    variable["dataType"] = cat
    variable["cardinality"] = card
    ev = rng.random(nvar) < evidence_frac
    variable["isEvidence"] = ev
    variable["isEvidence"][rng.random(nvar) < ghost_frac] = 4
    variable["initialValue"] = rng.integers(0, 1 << 30, nvar) % card
    variable["isEvidence"][rows] = 0
    ids0, ids1 = np.nonzero(~cat)[0], np.nonzero(cat)[0]
    f0 = tuple(funcs0) + ((8,) if ratio else ())
    facs, members = [], []
    for i in range(nfac):
        pool1 = len(ids1) > 0 and (len(ids0) == 0 or rng.random() < cat_frac)
        pool = ids1 if pool1 else ids0
        func = int(rng.choice(funcs1 if pool1 else f0))
        a = int(rng.integers(1, max_arity + 1))
        a = 1 if func == 15 else a
        facs.append(func)
        members.append(rng.choice(pool, min(a, len(pool)), replace=False))
    if wide_arity:                                   # one long factor: 2-word incidence headers
        facs.append(7)
        members.append(rng.choice(ids0, wide_arity, replace=False))
    arity = [np.array([len(m) for m in members])]
    # hub factors, pairwise (hub, other): funcs (3, 7, 9) on dataType 0, AND_CAT on dataType 1
    ninc = np.bincount(np.concatenate(members), minlength=nvar)
    hub_ids = rng.choice(np.setdiff1d(ids0 if len(ids0) else ids1, rows), hubs, replace=False) if hubs else []
    every_hub = np.concatenate((hub_ids, rows)).astype(np.int64)
    for h, m in list(zip(hub_ids, [hub_degree] * hubs)) + [(h, r[2] - ninc[h]) for h, r in zip(rows, hub_rows)]:
        assert m >= 0, "hub row already has more incidences than asked for"
        pool = ids1 if cat[h] else ids0
        other = rng.choice(pool[~np.isin(pool, every_hub)], m)
        facs.extend(np.full(m, 12) if cat[h] else rng.choice((3, 7, 9), m))
        members.append(np.stack([np.full(m, h), other], axis=1).ravel())
        arity.append(np.full(m, 2))
    nf = len(facs)
    n_weights = n_weights or max(1, nf // 3)
    weight = np.zeros(n_weights, Weight)
    weight["isFixed"] = rng.random(n_weights) < fixed_frac
    weight["initialValue"] = rng.normal(0, w_scale, n_weights)
    factor = np.zeros(nf, Factor)
    factor["factorFunction"] = facs
    factor["weightId"] = rng.integers(0, n_weights, nf)
    factor["featureValue"] = rng.choice([1.0, 0.5, 2.0], nf) if feature_values else 1.0
    factor["arity"] = np.concatenate(arity)
    factor["ftv_offset"] = np.concatenate(([0], np.cumsum(factor["arity"])[:-1]))
    vids = np.concatenate(members).astype(np.int64)
    fmap = np.zeros(len(vids), FactorToVar)
    fmap["vid"] = vids
    fmap["dense_equal_to"] = rng.integers(0, 1 << 30, len(vids)) % card[vids]
    for h in rows[cat[rows]]:                        # empty buckets: a fifth of the values get no incidence
        at = np.nonzero(vids == h)[0]
        fmap["dense_equal_to"][at] = rng.choice(rng.permutation(card[h])[:card[h] - card[h] // 5], len(at))
    return weight, variable, factor, fmap, np.zeros(nvar, np.bool_), len(vids)


def _spec(name):
    """(graph, FactorGraph attributes, row classes that must be present)."""
    from numbskull_b200 import synth
    if name == "pair_uniform":
        g = list(synth.ising_grid(48, 48, coupling=0.37, fixed=False))
        rng = np.random.default_rng(1)
        g[1]["isEvidence"] = rng.random(len(g[1])) < 0.2
        g[1]["initialValue"] = rng.integers(0, 2, len(g[1]))
        return tuple(g), {}, ("PAIR",)
    if name == "pair_records":
        return _graph(2, nvar=3000, nfac=4000, max_arity=2, funcs0=(2, 3, 4, 9)), {}, ("PAIR",)
    if name == "fast":
        return synth.kbc(4000, np.random.default_rng(3), n_weights=1024, window=64, hub_frac=0.0), {}, ("FAST",)
    if name == "gen_boolean":
        return _graph(4, ratio=True, feature_values=True, max_arity=5), {}, ("GEN",)
    if name == "gen_card":
        return _graph(5, dt0_cards=(1, 2, 3, 4, 5, 8), funcs0=(3, 7, 9, 8)), {}, ("GEN",)
    if name == "gen_cat_empty":
        return _graph(6, cat_frac=1.0, cat_cards=(2, 12), nfac=2500, funcs1=(12, 14, 15), max_arity=4,
                      w_scale=0.3), {}, ("GEN", "CAT")
    if name == "cat":
        return synth.categorical(4000, 16, 3, np.random.default_rng(7), n_weights=512, window=64), {}, ("CAT",)
    if name == "warp":
        return (_graph(8, dt0_cards=(2, 2, 3, 6), cat_frac=0.3, hubs=24, hub_degree=150),
                {"warp_row_words": 40}, ("WARP", "GEN"))
    if name == "saturating":
        return (_graph(9, dt0_cards=(2, 2, 3, 6), cat_frac=0.3, cat_cards=(3, 8), hubs=8, w_scale=40.0),
                {"warp_row_words": 40}, ("GEN", "WARP"))
    if name == "wide_headers":
        return _graph(10, dt0_cards=(2, 3), wide_arity=40, max_arity=3, hubs=4), {"warp_row_words": 40}, ("GEN",)
    if name == "global_vid":
        g = _graph(11, dt0_cards=(2, 3), cat_frac=0.2, hubs=6, ghost_frac=0.05)
        gid = (np.int64(7) << 32) + np.random.default_rng(1).permutation(1 << 20)[:len(g[1])].astype(np.int64) * 3
        return g, {"global_vid": gid, "warp_row_words": 40}, ("GEN", "WARP", "PAIR")
    if name in ("wide_card", "wide_card_thread"):
        g = synth.wide_categorical(400, card=700, cands=16, feats=2, couplings=2, rng=np.random.default_rng(12),
                                   n_weights=256)
        if name == "wide_card":          # mentions and features on the warp path
            return g, {"warp_row_words": 32}, ("WIDE", "WARP")
        return g, {}, ("GEN",)           # every row one thread: generic rows above cardinality 255
    if name == "big_table":
        return _graph(13, dt0_cards=(2, 3), cat_frac=0.2, n_weights=5000, nfac=9000, hubs=4,
                      funcs0=(0, 1, 2, 3, 4, 7, 9)), {"warp_row_words": 40}, ("GEN",)
    if name == "hub_tasks":          # HUB_TASKS: rows of 32, 33 and more than 64 warp tasks
        return _graph(17, dt0_cards=(2, 2, 3), cat_frac=0.3, hub_rows=[(d, c, n) for (d, c), n in HUB_TASKS]), {}, \
            ("WARP", "GEN", "CAT")
    if name == "hub_tasks_wide":     # a categorical hub above 255 values (2-byte graph): nb_warp_sample_wide
        return _graph(18, dt0_cards=(2, 3), cat_frac=0.3, hub_rows=[(1, 700, 2100)]), {}, ("WIDE", "GEN")
    if name == "hub_mirror":         # all-Boolean; hubs of ~ 0.3 x 2 x 4000 = 2400 IMPLY and as many OR incidences
        return synth.kbc(8000, np.random.default_rng(19), n_weights=1024, window=64, hub_frac=0.3), {}, \
            ("FAST", "WARP")
    if name == "card_band":          # 1-byte graph, cardinalities 33 - 255, each as GEN and as WARP rows
        return (_graph(20, nvar=4000, nfac=9000, dt0_cards=CARD_BAND[0], cat_frac=0.5, cat_card_set=CARD_BAND[1],
                       max_arity=3), {"warp_row_words": 14}, ("GEN", "WARP"))
    if name == "cat32":              # CAT rows at NB_CAT_MAX_CARD, and cardinality-33 rows next to them
        g = synth.categorical(4000, 32, 3, np.random.default_rng(21), n_weights=512, window=64)
        g[1]["cardinality"][np.random.default_rng(22).choice(len(g[1]), 40, replace=False)] = 33
        return g, {}, ("CAT",)
    if name == "thread_row_long":    # one Boolean hub of > NB_META_MAX_ROWLEN words, as long as thread rows may be
        return (_graph(23, dt0_cards=(2,), feature_values=True, hub_rows=[(0, 2, 46000)]), {"warp_row_words": 1 << 20},
                ("GEN",))
    if name == "tally_chunks":       # > 3 x 2^18 tallies (test_tally_widths): Boolean record rows, cardinality-40 GEN rows
        return _graph(30, nvar=60001, nfac=60000, dt0_cards=(2, 2, 40), max_arity=3), {}, ("PAIR", "FAST", "GEN")
    # weight ids at the limits of the record fields (WID_COMPACT, WID_PAIR): fixtures above with their
    # weights moved into large tables
    if name in ("wid_compact_top", "wid_wide"):   # every row class; weight 0 tied to a tenth of the factors
        g = _every_class()
        n = len(g[0])
        if name == "wid_compact_top":             # W = 2^20: the last compact id, headers stay compact
            ids = _wid_targets(n, WID_COMPACT, WID_COMPACT, [WID_COMPACT - 1], 24)
            return _move_weights(g, WID_COMPACT, ids, 24), {"warp_row_words": 40}, CLASS_NAMES[:5]
        # W = 2^20 + 1: the table alone makes the headers wide, and only weight 0 sits at 2^20
        ids = _wid_targets(n, WID_COMPACT + 1, WID_COMPACT, [WID_COMPACT, 0, WID_COMPACT - 1], 25)
        return _move_weights(g, WID_COMPACT + 1, ids, 25), {"warp_row_words": 40}, CLASS_NAMES[:5]
    if name == "wid_pair_top":       # pair_uniform's one weight at 2^22 - 1 (W = 2^22)
        g, _, cls = _spec("pair_uniform")
        return _move_weights(g, WID_PAIR, np.array([WID_PAIR - 1]), 26), {}, cls
    if name == "wid_pair_alias":     # ids 0 and 2^22 (W = 2^22 + 1): the same 22-bit field, different weights
        g = list(_grid(48))
        g[2]["weightId"] = np.where(np.random.default_rng(27).random(len(g[2])) < 0.2, 1, 0)
        g[0] = np.concatenate([g[0], g[0]])
        g[0]["initialValue"][1] = -0.81
        return _move_weights(tuple(g), WID_PAIR + 1, np.array([0, WID_PAIR]), 27), {}, ("PAIR", "FAST")
    if name in ("wid_fast", "wid_cat"):   # FAST / CAT records with ids on both sides of 2^22 (W = 2^22 + 512)
        g, attrs, cls = _spec(name[4:])
        ids = _wid_targets(len(g[0]), WID_PAIR + 512, WID_PAIR, [WID_PAIR - 1, WID_PAIR, WID_PAIR + 511], 28)
        return _move_weights(g, WID_PAIR + 512, ids, 28), attrs, cls
    # Large cells, sized from the SM count S to about twice the threshold of the branch they are for
    # (learn_branches; the grids' two colours hold n^2 / 2 rows each)
    S = _sms()
    if name in ("pair_slices", "pair_slices_windows"):      # > 128 S rows: slices in both modes, one tied weight
        return _grid(math.isqrt(512 * S - 1) + 1), ({"sigma_shift": 12} if name.endswith("windows") else {}), ("PAIR",)
    if name == "pair_slices_untied":                         # W > 2048 (global tables): > 512 S rows
        return _grid(math.isqrt(2048 * S - 1) + 1, n_weights=5000, fixed_frac=0.1), {}, ("PAIR",)
    if name == "pair_blocks":                                # 3 blocks of cells of > 128 S rows
        return _grid(math.isqrt(1536 * S - 1) + 1), {}, ("PAIR",)
    if name == "fast_slices":                                # largest colour ~ 1/3 of the rows: > 32 S FAST rows
        return (synth.kbc(200 * S, np.random.default_rng(3), n_weights=1000, window=64, hub_frac=0.0, fixed_frac=0.2),
                {}, ("FAST",))
    if name == "lf_many":                                    # one colour of ~ 4100 S LF rows (GEN), one of 41 S labels
        return synth.lf_model(41 * S, 100, np.random.default_rng(14)), {}, ("PAIR", "GEN")
    if name == "lf_long":                                    # label rows of 301 incidences, kept off the warp path
        return synth.lf_model(64, 300, np.random.default_rng(15)), {"warp_row_words": 4096}, ("PAIR", "GEN")
    if name == "cat_many":                                   # largest colour ~ 55 % of the rows: > 512 S CAT rows
        return (synth.categorical(1900 * S, 16, 1, np.random.default_rng(16), n_weights=512, window=64), {},
                ("CAT",))
    # rows of 3 or 4 incidences (9 or 12 words) on the warp path: a colour of ~ n^2 / 2 warp rows
    if name == "warp_crowd":                                 # > 2 x 64 S rows (8 warps x cap = 8 S CTAs)
        return _grid(math.isqrt(320 * S - 1) + 1), {"warp_row_words": 8}, ("WARP", "PAIR")
    if name == "warp_crowd_untied":                          # W > 2048 (cap = 32 S CTAs): > 2 x 256 S rows
        return (_grid(math.isqrt(1280 * S - 1) + 1, n_weights=5000, fixed_frac=0.1), {"warp_row_words": 8},
                ("WARP", "PAIR"))
    raise KeyError(name)


# hub rows of "hub_tasks": ((dataType, cardinality), incidences).  A warp task takes NB_WARP_TASK = 64
# incidences and k_gibbs_warp_finish's lanes stride over a row's tasks: 32 tasks fill the lanes once, 33
# wrap once, more than 64 wrap twice.  Cardinality 2 takes the e[4] path, 6 the shared-array atomics, the
# categorical ones the bucket index (ent.y), with empty buckets.
HUB_TASKS = [((0, 2), 2048), ((0, 2), 4500), ((0, 6), 2049), ((0, 6), 4161),
             ((1, 40), 2048), ((1, 40), 4300), ((1, 200), 2049), ((1, 200), 5000)]
# "card_band": dataType-0 and categorical cardinalities of a 1-byte graph, all above the lanes of a warp
# but 5 (and above NB_CAT_MAX_CARD); 128 - 255 are values of uint8_t with the top bit set
CARD_BAND = ((5, 40, 255), (33, 64, 127, 128, 200, 255))

# Weight ids are packed into fixed-width fields: 20 bits in compact generic headers (a larger table
# makes the whole graph take 2-word headers), 22 bits in the 8-byte pair records and the hoisted
# tt2_common word (a row with a larger id is FAST instead of PAIR)
WID_COMPACT, WID_PAIR = 1 << 20, 1 << 22


def _union(*gs):
    """Disjoint union of graphs (weight, variable, factor, fmap, domain_mask, edges)."""
    w, v, f, m = [], [], [], []
    nw = nv = nm = 0
    for g in gs:
        fac, fmap = g[2].copy(), g[3].copy()
        fac["weightId"] += nw
        fac["ftv_offset"] += nm
        fmap["vid"] += nv
        w.append(g[0])
        v.append(g[1])
        f.append(fac)
        m.append(fmap)
        nw, nv, nm = nw + len(g[0]), nv + len(g[1]), nm + len(fmap)
    return np.concatenate(w), np.concatenate(v), np.concatenate(f), np.concatenate(m), np.zeros(nv, np.bool_), nm


def _every_class():
    """PAIR, FAST, CAT, GEN (categorical ones with MARK words) and WARP rows in one graph, with
    weight 0 tied to a tenth of the factors, so that one weight id reaches every row class."""
    g = _union(_spec("fast")[0], _spec("cat")[0], _spec("warp")[0], _spec("pair_records")[0])
    g[2]["weightId"][np.random.default_rng(29).random(len(g[2])) < 0.1] = 0
    return g


def _wid_targets(n, W, limit, pinned, seed):
    """n distinct weight ids below W: old id i < len(pinned) goes to pinned[i]; of the others, half go
    to [limit - 4n, limit) and half to [limit, W) (all of them below `limit` when W <= limit)."""
    rng = np.random.default_rng(seed)
    pinned = np.asarray(pinned, np.int64)
    k = n - len(pinned)
    above = np.setdiff1d(np.arange(limit, W), pinned)
    n_above = min(len(above), k // 2)
    below = np.setdiff1d(np.arange(max(0, limit - 4 * n), min(limit, W)), pinned)
    rest = np.concatenate([rng.choice(above, n_above, replace=False), rng.choice(below, k - n_above, replace=False)])
    return np.concatenate([pinned, rng.permutation(rest)])


def _move_weights(g, W, ids, seed):
    """g with its weights moved into a table of W: old weight i becomes weight ids[i] (ids distinct, so
    the tying, isFixed and initialValue of every used weight are kept).  The unused weights get random
    values and flags: an incidence that reads a wrong id reads a different weight."""
    from numbskull_b200.numbskulltypes import Weight
    rng = np.random.default_rng(seed)
    ids = np.asarray(ids, np.int64)
    assert len(ids) == len(g[0]) and len(np.unique(ids)) == len(ids) and ids.max() < W
    weight = np.zeros(W, Weight)
    weight["isFixed"] = rng.random(W) < 0.2
    weight["initialValue"] = rng.normal(0.0, 1.0, W)
    weight[ids] = g[0]
    factor = g[2].copy()
    factor["weightId"] = ids[factor["weightId"]]
    return (weight, g[1], factor) + tuple(g[3:])


def _check_spec(r):
    """The property each of the larger replay graphs exists for, from the records."""
    name, O = r.name, oracle.oracle
    fm = r.fg.fmap
    ninc = np.bincount(fm["vid"], minlength=r.V)
    live = r.evid != 4
    warp_path = np.isin(r.cls, (O.WARP, O.WIDE)) & live
    if name in ("hub_tasks", "hub_mirror"):
        hub = warp_path & (ninc >= 2048)
        tasks = {(int(r.card[v]), -(-int(ninc[v]) // 64)) for v in np.nonzero(hub)[0]}
        if name == "hub_tasks":
            assert tasks == {(c, -(-n // 64)) for (_, c), n in HUB_TASKS}, tasks
            assert {32, 33} <= {t for _, t in tasks} and max(t for _, t in tasks) > 64, tasks
        else:                            # more than 32 tasks: the task sum wraps before the mirror update
            assert (r.card == 2).all() and tasks and max(t for _, t in tasks) > 32, tasks
    if name == "hub_tasks_wide":
        assert r.info["value_bytes"] == 2
        (hub,) = np.nonzero((r.card > 255) & warp_path)[0]
        assert r.cls[hub] == O.WIDE and ninc[hub] > 2048
        size = np.bincount(fm["dense_equal_to"][fm["vid"] == hub], minlength=r.card[hub])
        assert (size == 0).any(), "no empty bucket"
        end = np.cumsum(size[size > 0])          # buckets in value order, as the row holds them
        assert ((end - size[size > 0]) // 32 != (end - 1) // 32).any(), "no bucket straddles 32 incidences"
    if name == "card_band":
        assert r.info["value_bytes"] == 1
        dtype = r.fg.variable["dataType"]
        for d, cards in enumerate(CARD_BAND):
            for c in cards:
                for cl in (O.GEN, O.WARP):
                    assert ((dtype == d) & (r.card == c) & (r.cls == cl) & live).any(), (d, c, CLASS_NAMES[cl])
    if name == "cat32":
        assert ((r.cls == O.CAT) & (r.card == 32) & live).any()
        c33 = (r.card == 33) & live
        assert c33.any() and (r.cls[c33] != O.CAT).all()
    if name == "thread_row_long":        # at least (1 + arity) words per incidence
        fac = r.fg.factor
        fidx = np.repeat(np.arange(len(fac)), fac["arity"])
        hub = int(np.argmax(ninc))
        assert (1 + fac["arity"][fidx[fm["vid"] == hub]]).sum() > 131071 and r.evid[hub] == 0
    if name.startswith("wid_"):
        W = len(r.fg.weight)
        fac = r.fg.factor
        wid = fac["weightId"][np.repeat(np.arange(len(fac)), fac["arity"])].astype(np.int64)
        top = np.zeros(r.V, np.int64)            # largest weight id among a row's incidences
        np.maximum.at(top, fm["vid"], wid)

        def rows_with(ids):
            has = np.zeros(r.V, bool)
            has[fm["vid"][np.isin(wid, ids)]] = True
            return has & live

        assert r.info["max_arity"] <= 31
        if name in ("wid_compact_top", "wid_wide"):
            at = WID_COMPACT - 1 if name == "wid_compact_top" else WID_COMPACT
            assert W == at + 1 and r.info["wide_headers"] == int(name == "wid_wide")
            for c in range(5):                   # the id at the limit in every row class
                assert (rows_with([at]) & (r.cls == c)).any(), CLASS_NAMES[c]
            gen = np.isin(r.cls, (O.GEN, O.WARP)) & (r.fg.variable["dataType"] == 1)
            assert (rows_with([at]) & gen).any(), "no categorical generic row (MARK words) at the limit"
        if name == "wid_pair_top":
            assert W == WID_PAIR and (wid == WID_PAIR - 1).all() and (r.cls[live] == O.PAIR).all()
            import numbskull_b200 as nb
            ns = nb.NumbSkull(quiet=True)
            ns.loadFactorGraph(*_spec("pair_uniform")[0])
            fg = ns.factorGraphs[0]
            quads = fg.device_info()["tt2_quads"]
            fg.clear()
            assert r.info["tt2_quads"] == quads, "the grid's slices are no longer uniform"
        if name == "wid_pair_alias":             # a row reading id 2^22 cannot take a pair record
            assert W == WID_PAIR + 1 and set(np.unique(wid)) == {0, WID_PAIR}
            w = r.fg.weight
            assert w["initialValue"][0] != w["initialValue"][WID_PAIR] and w["isFixed"][0] == w["isFixed"][WID_PAIR]
            alias = rows_with([WID_PAIR])
            assert alias.any() and (live & ~alias).any()
            assert (r.cls[alias] == O.FAST).all() and (r.cls[live & ~alias] == O.PAIR).all()
        if name in ("wid_fast", "wid_cat"):      # records on both sides of 2^22, and at W - 1
            c = O.FAST if name == "wid_fast" else O.CAT
            assert W == WID_PAIR + 512 and (rows_with([W - 1, WID_PAIR]) & (r.cls == c)).any()
            assert ((top >= WID_PAIR) & (r.cls == c) & live).any() and ((top < WID_PAIR) & (r.cls == c) & live).any()
            assert not ((top >= WID_PAIR) & (r.cls == O.PAIR) & live).any()


def _sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _grid(n, n_weights=1, fixed_frac=0.0):
    """n x n Ising grid (EQUAL to the up and left neighbours), 20 % evidence, random initial values;
    n_weights > 1 spreads the factors over a table of that many weights, fixed_frac of them fixed."""
    from numbskull_b200 import synth
    from numbskull_b200.numbskulltypes import Weight
    g = list(synth.ising_grid(n, n, coupling=0.37, fixed=False))
    rng = np.random.default_rng(n)
    g[1]["isEvidence"] = rng.random(len(g[1])) < 0.2
    g[1]["initialValue"] = rng.integers(0, 2, len(g[1]))
    if n_weights > 1:
        g[0] = np.zeros(n_weights, Weight)
        g[0]["isFixed"] = rng.random(n_weights) < fixed_frac
        g[0]["initialValue"] = rng.normal(0.0, 0.5, n_weights)
        g[2]["weightId"] = rng.integers(0, n_weights, len(g[2]))
    return tuple(g)


class Replay(object):
    """One device graph, driven through the C ABI, and its oracle twin."""

    def __init__(self, name):
        import numbskull_b200 as nb
        from numbskull_b200 import _lib
        g, attrs, self.expect = _spec(name)
        self.name = name
        ns = nb.NumbSkull(quiet=True)
        ns.loadFactorGraph(*g)
        fg = self.fg = ns.factorGraphs[0]
        fg.seed = SEED
        for k, v in attrs.items():
            setattr(fg, k, v)
        self.L, self._lib = _lib.lib(), _lib
        self.g = fg._device_graph()
        self.og = oracle.OracleGraph(fg.weight.copy(), fg.variable.copy(), fg.factor.copy(), fg.fmap.copy(),
                                     fg.vmap.copy(), fg.factor_index.copy(), nthreads=1, seed=0)
        self.V = len(fg.variable)
        self.card = fg.variable["cardinality"].astype(np.int64)
        self.evid = fg.variable["isEvidence"].astype(np.int64)
        self.init = fg.variable["initialValue"].astype(np.int64)
        self.cstart = fg.cstart
        self.colors = fg.colors()
        self.info = fg.device_info()
        _, cls = fg.potentials_records(np.arange(self.V, dtype=np.int64))
        cls = cls.astype(np.int32)
        cls[(cls == oracle.oracle.WARP) & (self.card > 255)] = oracle.oracle.WIDE
        self.cls = cls
        gid = attrs.get("global_vid")
        self.rid = ((np.arange(self.V, dtype=np.int64) if gid is None else np.asarray(gid, np.int64))
                    & 0xFFFFFFFF).astype(np.uint32)
        self.draws = 0
        self.ties = []
        live = self.evid != 4
        present = {CLASS_NAMES[c] for c in np.unique(cls[live])}
        for c in self.expect:
            assert c in present, (name, c, present, self.info)
        _check_spec(self)

    # ---- state through the C ABI ----
    def _chk(self, rc):
        self._lib.check(rc)

    def get_vals(self, chain):
        out = np.empty(self.V, np.int64)
        self._chk(self.L.nb_get_var_values(self.g, chain, self._lib.ptr(out)))
        return out

    def set_vals(self, chain, v):
        v = np.ascontiguousarray(v, np.int64)
        self._chk(self.L.nb_set_var_values(self.g, chain, self._lib.ptr(v)))

    def get_w(self):
        out = np.empty(len(self.fg.weight), np.float64)
        self._chk(self.L.nb_get_weights(self.g, self._lib.ptr(out)))
        return out

    def set_w(self, w):
        w = np.ascontiguousarray(w, np.float64)
        self._chk(self.L.nb_set_weights(self.g, self._lib.ptr(w)))

    def counts(self):
        out = np.zeros(int(self.cstart[-1]), np.int64)
        self._chk(self.L.nb_get_counts(self.g, self._lib.ptr(out), 0))
        return out

    def random_state(self, rng, weights=True):
        for chain in (0, 1):
            self.set_vals(chain, rng.integers(0, 1 << 30, self.V) % self.card)
        if weights:
            w = self.og.weight["initialValue"] * rng.uniform(0.5, 1.5, len(self.fg.weight))
            self.set_w(w)

    def cell_ids(self, color, block, n_blocks):
        import ctypes as C
        out = np.empty(self.V, np.int64)
        n = C.c_int64(0)
        self._chk(self.L.nb_learn_cell_ids(self.g, color, block, n_blocks, self._lib.ptr(out), C.byref(n)))
        return out[:n.value]

    # ---- comparison ----
    def compare(self, what, ids, got, want, margin, epoch, tag, evid_chain=False):
        ids = np.asarray(ids, np.int64)
        assert (got >= 0).all() and (got < self.card[ids]).all(), (what, "pick out of range")
        diff = got != want
        bad = diff & (margin >= NEAR_TIE)
        if bad.any():
            rows = []
            for i in np.nonzero(bad)[0][:5]:
                v = int(ids[i])
                fam = 0 if self.cls[v] <= oracle.oracle.CAT else 1
                u = R.first_uniforms(self.rid[v:v + 1], [fam], SEED, epoch, tag)[0]
                e = self.og.energies([v], evid_chain)
                rows.append("var %d class %s card %d epoch %d tag %d: gpu %d replay %d margin %.3g first uniform %.17g "
                            "energies %s" % (v, CLASS_NAMES[self.cls[v]], self.card[v], epoch, tag, got[i], want[i],
                                             margin[i], u, np.array2string(e[:12], precision=6)))
            raise AssertionError("%s on %s: %d of %d draws differ beyond the margin\n  %s"
                                 % (what, self.name, int(bad.sum()), len(ids), "\n  ".join(rows)))
        self.draws += len(ids)
        for i in np.nonzero(diff)[0]:
            self.ties.append((what, int(ids[i]), float(margin[i])))

    def finish(self):
        print("%s: %d draws replayed, %d near-ties %s" % (self.name, self.draws, len(self.ties), self.ties[:5]))
        assert self.draws > 0
        assert len(self.ties) <= MAX_TIE_RATE * self.draws, self.ties
        self.fg.clear()

    # ---- Gibbs ----
    def sampled(self, sample_evidence):
        return (self.evid != 4) & ((self.evid == 0) | bool(sample_evidence))

    def tally(self, ids, vals):
        want = np.zeros(int(self.cstart[-1]), np.int64)
        b = self.card[ids] == 2
        np.add.at(want, self.cstart[ids[b]], vals[ids[b]])
        np.add.at(want, self.cstart[ids[~b]] + vals[ids[~b]], 1)
        return want

    def gibbs_phase(self, color, burnin, sample_evidence, epoch):
        before, c0 = self.get_vals(0), self.counts()
        self.og.var_value[:] = before
        self.og.weight_value[:] = self.get_w()
        self._chk(self.L.nb_gibbs_color_phase(self.g, color, int(burnin), int(sample_evidence), SEED, epoch))
        after, c1 = self.get_vals(0), self.counts()
        moving = self.sampled(sample_evidence) & (self.colors == color)
        assert np.array_equal(after[~moving], before[~moving]), "a variable outside the phase changed"
        ids = np.nonzero(moving)[0]
        pick, margin = self.og.replay_draws(ids, self.cls[ids], self.rid[ids], SEED, epoch, R.TAG_FREE)
        self.compare("gibbs c%d" % color, ids, after[ids], pick, margin, epoch, R.TAG_FREE)
        want = np.zeros_like(c0) if burnin else self.tally(ids, after)
        assert np.array_equal(c1 - c0, want), "tally deltas differ"
        return len(ids)

    def whole_sweeps(self, n, sample_evidence):
        """n sweeps of a fresh graph through nb_gibbs_sweeps (the first one as burn-in): sweep k runs
        at epoch k, colour c samples from the values of colours < c after the sweep."""
        for k in range(n):
            burnin = k == 0
            before, c0 = self.get_vals(0), self.counts()
            self.og.weight_value[:] = self.get_w()
            self._chk(self.L.nb_gibbs_sweeps(self.g, 1, int(burnin), int(sample_evidence), SEED))
            after, c1 = self.get_vals(0), self.counts()
            moving = self.sampled(sample_evidence) & (self.colors >= 0)
            assert np.array_equal(after[~moving], before[~moving])
            for c in range(self.info["n_colors"]):
                self.og.var_value[:] = np.where((self.colors < c) & (self.colors >= 0), after, before)
                ids = np.nonzero(moving & (self.colors == c))[0]
                pick, margin = self.og.replay_draws(ids, self.cls[ids], self.rid[ids], SEED, k, R.TAG_FREE)
                self.compare("sweep %d c%d" % (k, c), ids, after[ids], pick, margin, k, R.TAG_FREE)
            ids = np.nonzero(moving)[0]
            want = np.zeros_like(c0) if burnin else self.tally(ids, after)
            assert np.array_equal(c1 - c0, want), "tally deltas differ"

    # ---- learning ----
    def learn_cell(self, color, block, n_blocks, step, reg, reg_param, trunc, lne, epoch):
        F0, E0, w0 = self.get_vals(0), self.get_vals(1), self.get_w()
        self.og.var_value[:], self.og.var_value_evid[:], self.og.weight_value[:] = F0, E0, w0
        cell = self.cell_ids(color, block, n_blocks)
        assert (self.colors[cell] == color).all()
        if n_blocks == 1:
            assert np.array_equal(np.sort(cell), np.nonzero(self.colors == color)[0])
        self._chk(self.L.nb_learn_color_phase(self.g, color, block, n_blocks, step, reg, reg_param, trunc, int(lne),
                                              SEED, epoch))
        F1, E1, w1 = self.get_vals(0), self.get_vals(1), self.get_w()
        act = np.sort(cell[self.evid[cell] != 4])
        inside = np.zeros(self.V, bool)
        inside[act] = True
        assert np.array_equal(F1[~inside], F0[~inside]) and np.array_equal(E1[~inside], E0[~inside]), \
            "a variable outside the cell changed"
        lab = act[self.evid[act] == 1]
        assert np.array_equal(E1[lab], self.init[lab]), "evidence chain of labelled variables != initialValue"
        free = act[self.evid[act] != 1]
        pick, margin = self.og.replay_draws(free, self.cls[free], self.rid[free], SEED, epoch, R.TAG_EVID, True)
        self.compare("learn evid c%d b%d" % (color, block), free, E1[free], pick, margin, epoch, R.TAG_EVID, True)
        pick, margin = self.og.replay_draws(act, self.cls[act], self.rid[act], SEED, epoch, R.TAG_FREE)
        self.compare("learn free c%d b%d" % (color, block), act, F1[act], pick, margin, epoch, R.TAG_FREE)
        # gradients from the draws the GPU made (a near-tie must not turn into a weight mismatch)
        grad = act if lne else lab
        if reg == 1:
            # record rows with one draw (PAIR / FAST) take the Philox2x32 truncation draw; CAT, GEN and
            # WARP rows the multi-draw stream's (nb_cnt_inc)
            fam = (self.cls[grad] > oracle.oracle.FAST).astype(np.int32)
            u = R.first_uniforms(self.rid[grad], fam, SEED, epoch, R.TAG_TRUNC)
            inc = (u < 1.0 / trunc).astype(np.uint32)
        else:
            inc = np.full(len(grad), 1 if reg == 2 else 0, np.uint32)
        G, cnt = self.og.cell_gradients(grad, E1[grad], F1[grad], inc)
        fixed = self.fg.weight["isFixed"].astype(bool)
        touched = ((G != 0) | (cnt != 0)) & ~fixed
        want = w0.copy()
        for i in np.nonzero(touched)[0]:
            want[i] = apply_update(w0[i], G[i] / R.GRAD_UNIT, int(cnt[i]), reg, step, reg_param, trunc)
        assert np.array_equal(w1[~touched], w0[~touched]), "a weight without visits (or a fixed one) moved"
        tol = 1e-12 * (np.abs(want) + np.abs(w0) + step * np.abs(G) / R.GRAD_UNIT)
        err = np.abs(w1 - want)
        if (err > tol).any():
            i = int(np.argmax(err - tol))
            raise AssertionError("weight %d: gpu %.17g replay %.17g (before %.17g, G %d / 2^20, visits %d)"
                                 % (i, w1[i], want[i], w0[i], G[i], cnt[i]))
        return int(touched.sum())


def apply_update(w, G, cnt, reg, step, reg_param, trunc):
    """Closed form of `cnt` per-visit updates with the summed gradient G (DESIGN.md, learning)."""
    if reg == 2:
        if cnt == 0:
            return w - step * G
        s = 1.0 / (1.0 + reg_param * step)
        sn = s ** cnt
        geo = (1.0 - sn) / (cnt * (1.0 - s)) if s < 1.0 else 1.0
        return w * sn - step * G * geo
    w = w - step * G
    if reg == 1 and cnt > 0:
        l1 = reg_param * step * trunc * cnt
        w = max(0.0, w - l1) if w > 0.0 else min(0.0, w + l1)
    return w


# =========================================================================== GPU: Gibbs phases
GIBBS_GRAPHS = ["pair_uniform", "pair_records", "fast", "gen_boolean", "gen_card", "gen_cat_empty", "cat", "warp",
                "saturating", "wide_headers", "global_vid", "wide_card", "wide_card_thread", "hub_tasks", "hub_tasks_wide",
                "card_band", "cat32", "thread_row_long", "wid_compact_top", "wid_wide", "wid_pair_top", "wid_pair_alias",
                "wid_fast", "wid_cat"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", GIBBS_GRAPHS)
def test_gibbs_phases_replay_exactly(name):
    r = Replay(name)
    if name == "wide_headers":
        assert r.info["wide_headers"] == 1
    if name.startswith("wide_card"):
        assert r.info["value_bytes"] == 2
    if name == "wide_card_thread":
        assert ((r.cls == oracle.oracle.GEN) & (r.card > 255)).any()
    rng = np.random.default_rng(sum(map(ord, name)))
    n = 0
    for i, epoch in enumerate(EPOCHS):
        r.random_state(rng)
        for burnin, sample_evidence in ((0, 0), (1, 1), (0, 1)):
            for c in range(r.info["n_colors"]):
                n += r.gibbs_phase(c, burnin, sample_evidence, epoch + 7 * c * (i % 2))
    assert n > 0
    if name == "card_band":
        assert (r.get_vals(0)[r.sampled(True)] >= 128).any()
    if name == "thread_row_long":
        # too long for the 17-bit length of thread rows.  Only this class check catches a partly walked
        # row here: the hub's energy saturates, so its draws match either way.  The LEARN cases of
        # thread_row_long are the ones that see the wrong gradient sums of such a walk.
        assert r.cls[np.argmax(np.bincount(r.fg.fmap["vid"], minlength=r.V))] == oracle.oracle.WARP
    r.finish()


# =========================================================================== GPU: whole sweeps
def _whole_sweeps(name, sample_evidence):
    r = Replay(name)
    r.whole_sweeps(4, sample_evidence)
    r.finish()


@pytest.mark.gpu
@pytest.mark.parametrize("name,mirror", [("fast", "-1"), ("fast", "0"), ("warp", "-1"), ("gen_cat_empty", "-1"),
                                         ("wide_card", "-1"), ("hub_mirror", "0"), ("hub_tasks", "-1"),
                                         ("wid_compact_top", "-1"), ("wid_wide", "-1"), ("wid_pair_top", "-1"),
                                         ("wid_pair_top", "0"), ("wid_pair_alias", "-1"), ("wid_pair_alias", "0"),
                                         ("wid_fast", "0"), ("wid_cat", "-1")])
def test_whole_sweeps_replay_with_fan_out(name, mirror, monkeypatch):
    """nb_gibbs_sweeps with the row classes of a colour on concurrent streams (the default); "0"
    forces the bit-packed value mirror on (all-Boolean graphs)."""
    monkeypatch.setenv("NUMBSKULL_B200_BIT_MIRROR", mirror)
    _whole_sweeps(name, sample_evidence=True)


@pytest.mark.gpu
def test_whole_sweeps_replay_without_fan_out():
    """The same with NUMBSKULL_B200_FAN_OUT=0 (read once per process: a child interpreter)."""
    env = dict(os.environ, NUMBSKULL_B200_FAN_OUT="0", NUMBSKULL_B200_BIT_MIRROR="0")
    code = ("import sys; sys.path[:0] = [%r, %r]; import test_sweep_replay as t; "
            "[t._whole_sweeps(n, s) for n, s in (('fast', True), ('warp', False), ('gen_cat_empty', True))]"
            % (REPO, os.path.dirname(os.path.abspath(__file__))))
    p = subprocess.run([sys.executable, "-c", code], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                       text=True)
    print(p.stdout[-3000:])
    assert p.returncode == 0


# =========================================================================== GPU: learning cells
LEARN = [  # graph, regularization, learn_non_evidence
    ("fast", 2, True), ("fast", 1, False), ("pair_records", 0, True),
    ("gen_boolean", 2, True), ("gen_card", 1, True), ("gen_cat_empty", 2, False), ("gen_cat_empty", 1, True),
    ("cat", 1, True), ("cat", 2, False), ("warp", 2, True), ("warp", 1, True), ("warp", 0, False),
    ("big_table", 2, True), ("big_table", 1, False),
    ("wide_headers", 2, True), ("wide_headers", 1, False), ("global_vid", 1, True), ("global_vid", 2, False),
    ("saturating", 2, True), ("saturating", 0, True), ("pair_uniform", 1, True), ("pair_uniform", 2, False),
    ("hub_tasks", 2, True), ("hub_tasks", 1, False), ("card_band", 1, True), ("card_band", 2, False),
    ("cat32", 2, True), ("cat32", 1, False),
    ("thread_row_long", 2, True), ("thread_row_long", 1, True),     # the hub's own gradient: learn_non_evidence
    ("wid_compact_top", 2, True), ("wid_wide", 1, True), ("wid_wide", 2, False), ("wid_pair_top", 1, True),
    ("wid_pair_alias", 2, True), ("wid_fast", 1, True), ("wid_cat", 2, True),
]


def _learn(r, reg, lne, n_blocks_list, rng, reg_param=0.5):
    step, trunc = 0.05, 3.0
    touched = 0
    for i, epoch in enumerate((3, (1 << 32) + 5, (1 << 40) + 1)):
        r.random_state(rng)
        n_blocks = n_blocks_list[i % len(n_blocks_list)]
        for b in range(n_blocks):
            for c in range(r.info["n_colors"]):
                touched += r.learn_cell(c, b, n_blocks, step, reg, reg_param, trunc, lne, epoch)
    return touched


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["1", "2"])
@pytest.mark.parametrize("name,reg,lne", LEARN)
def test_learning_cells_replay_exactly(name, reg, lne, mode, monkeypatch):
    """One (block, colour) cell at a time in latency (1) and throughput (2) mode."""
    monkeypatch.setenv("NUMBSKULL_B200_LEARN_MODE", mode)
    r = Replay(name)
    if name == "big_table":
        assert len(r.fg.weight) > 2048
    rng = np.random.default_rng(len(name) * 31 + reg)
    touched = _learn(r, reg, lne, (1, 3), rng)
    assert touched > 0
    if name == "card_band":
        assert all((r.get_vals(chain)[r.evid == 0] >= 128).any() for chain in (0, 1))
    r.finish()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["wide_card", "wide_card_thread", "hub_tasks_wide"])
def test_learning_cells_replay_on_a_two_byte_graph(name, monkeypatch):
    monkeypatch.setenv("NUMBSKULL_B200_LEARN_MODE", "2")
    r = Replay(name)
    assert _learn(r, 2, True, (1, 2), np.random.default_rng(5)) > 0
    r.finish()


@pytest.mark.gpu
def test_learning_cells_at_the_default_block_count(monkeypatch):
    """Tied weights at a small step: the library's own block count cuts the id windows further
    (k_sub > 1); every cell of one epoch is replayed."""
    import ctypes as C
    monkeypatch.setenv("NUMBSKULL_B200_LEARN_MODE", "1")
    r = Replay("pair_uniform")
    nb = C.c_int(0)
    step = 0.002
    r._chk(r.L.nb_learn_blocks(r.g, step, 1, 0, C.byref(nb)))
    assert nb.value > 1
    r.random_state(np.random.default_rng(3))
    seen = set()
    for b in range(nb.value):
        for c in range(r.info["n_colors"]):
            seen.update(r.cell_ids(c, b, nb.value).tolist())
            r.learn_cell(c, b, nb.value, step, 2, 0.5, 3.0, True, 9)
    assert seen == set(np.nonzero(r.evid != 4)[0].tolist())
    r.finish()


# =========================================================================== GPU: large learning cells
def learn_branches(r, color, cell, mode, sms):
    """The code paths of nb_learn.cu that cell `cell` (ids of colour `color`) takes in latency mode
    (1: k_learn_cells, a grid of 2 CTAs of 256 threads per SM) or throughput mode (2: the lean
    launches of launch_cell_lean_t, at most `cap` CTAs each), by the library's own rules:
      * truth-table rows (PAIR + FAST) go one warp per row (learn_tt_rows) when the colour is
        flagged long-row (learn_prepare: incidences >= 16 x rows) or the cell has at most 2 rows
        per warp of the grid, else SELL slices (learn_tt_slices);
      * a warp takes several rows when there are more rows than warps; a row of more than
        NB_ROW_STASH x 32 = 256 incidences re-reads its tail;
      * GEN (learn_thread_rows) and CAT (learn_cat_rows) threads take several rows when the cell
        has more of them than the grid has threads;
      * a warp of learn_warp_rows takes several WARP rows when the cell has more of them than the
        grid has warps.
    Slices whose learnable incidences all share one weight id reduce it warp-wide (the tied branch);
    with several ids the lanes can add one by one."""
    fm, fac, w = r.fg.fmap, r.fg.factor, r.fg.weight
    ninc = np.bincount(fm["vid"], minlength=r.V)
    live = np.nonzero((r.colors == color) & (r.evid != 4))[0]
    tt_cls = (oracle.oracle.PAIR, oracle.oracle.FAST)
    long_rows = np.isin(r.cls[live], tt_cls).any() and ninc[live].sum() >= 16 * len(live)
    cls = r.cls[cell]
    tt_ids = cell[np.isin(cls, tt_cls)]
    tt, cat, gen = len(tt_ids), int((cls == oracle.oracle.CAT).sum()), int((cls == oracle.oracle.GEN).sum())
    warp = int(np.isin(cls, (oracle.oracle.WARP, oracle.oracle.WIDE)).sum())
    if mode == 1:
        rows_warps, threads = 16 * sms, 512 * sms
        slices = not long_rows and tt > 2 * rows_warps
        warps = 16 * sms
    else:
        cap = sms * (8 if len(w) <= 2048 else 32)
        slices = not long_rows and tt > 2 * cap * 8
        rows_warps = min((tt + 7) // 8, cap) * 8
        threads = cap * 256          # a thread takes several rows once the grid is capped
        warps = cap * 8              # k_cell_warp: at most cap CTAs of 8 warps
    out = set()
    if tt and slices:
        out.add("tt_slices")
        fidx = np.repeat(np.arange(len(fac)), fac["arity"])
        inc = np.isin(fm["vid"], tt_ids)
        wids = np.unique(fac["weightId"][fidx[inc]])
        wids = wids[~w["isFixed"][wids].astype(bool)]
        out.add("tt_slices_tied" if len(wids) == 1 else "tt_slices_per_lane")
    elif tt:
        out.add("tt_rows")
        if tt > rows_warps:
            out.add("tt_rows_several_per_warp")
        if ninc[tt_ids].max() > 256:
            out.add("tt_rows_tail")
    if gen > threads:
        out.add("gen_several_per_thread")
    if cat > threads:
        out.add("cat_several_per_thread")
    if warp > warps:
        out.add("warp_several_per_warp")
    return out


LARGE = [  # graph, mode, regularization, learn_non_evidence, branches that must be taken
    ("pair_slices", 1, 2, True, {"tt_slices_tied"}), ("pair_slices", 2, 1, False, {"tt_slices_tied"}),
    ("pair_slices_untied", 1, 0, True, {"tt_slices_per_lane"}),
    ("pair_slices_untied", 2, 2, False, {"tt_slices_per_lane"}),
    ("fast_slices", 1, 1, True, {"tt_slices_per_lane"}), ("fast_slices", 1, 2, False, {"tt_slices_per_lane"}),
    ("lf_many", 1, 1, False, {"gen_several_per_thread", "tt_rows_several_per_warp"}),
    ("lf_many", 2, 2, True, {"gen_several_per_thread"}),
    ("lf_long", 1, 2, True, {"tt_rows_tail"}), ("lf_long", 2, 1, True, {"tt_rows_tail"}),
    ("cat_many", 1, 1, True, {"cat_several_per_thread"}), ("cat_many", 1, 0, False, {"cat_several_per_thread"}),
    ("warp_crowd", 1, 2, True, {"warp_several_per_warp"}), ("warp_crowd", 2, 1, False, {"warp_several_per_warp"}),
    ("warp_crowd_untied", 2, 2, True, {"warp_several_per_warp"}),
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,mode,reg,lne,want", LARGE, ids=["%s-m%d-r%d-%s" % c[:4] for c in LARGE])
def test_large_learning_cells_replay_exactly(name, mode, reg, lne, want, monkeypatch):
    """Whole colours as cells (one block), large enough for the branches that only large cells
    take; every cell is replayed, and the branches it takes are checked, so that a smaller fixture or
    a moved threshold cannot quietly turn this back into a small-cell test."""
    monkeypatch.setenv("NUMBSKULL_B200_LEARN_MODE", str(mode))
    r = Replay(name)
    sms = _sms()
    taken = set()
    for c in range(r.info["n_colors"]):
        taken |= learn_branches(r, c, r.cell_ids(c, 0, 1), mode, sms)
    assert want <= taken, (name, mode, taken)
    # a whole colour visits a weight 10^3 - 10^5 times: at the small cells' reg_param every L1 update
    # would clamp the weights to 0 and every L2 shrink s^n underflow, whatever the visit counts
    assert _learn(r, reg, lne, (1,), np.random.default_rng(len(name) * 31 + reg), reg_param=1e-5) > 0
    r.finish()


@pytest.mark.gpu
def test_large_learning_cells_in_cut_id_windows(monkeypatch):
    """Id windows of 4096 variables (the size graphs of 2^22 variables or more get) and more blocks
    than windows, so that the plan cuts every window further (CellPlan::k_sub > 1): the cells of each
    epoch partition the live variables, and every one of them is replayed."""
    monkeypatch.setenv("NUMBSKULL_B200_LEARN_MODE", "1")
    r = Replay("pair_slices_windows")
    n_win = (r.V >> 12) + 1
    n_blocks = 2 * n_win + 1
    rng = np.random.default_rng(12)
    live = set(np.nonzero(r.evid != 4)[0].tolist())
    for epoch in (3, (1 << 32) + 5, (1 << 40) + 1):
        r.random_state(rng)
        seen = []
        for b in range(n_blocks):
            for c in range(r.info["n_colors"]):
                seen.extend(r.cell_ids(c, b, n_blocks).tolist())
                r.learn_cell(c, b, n_blocks, 0.05, 2, 0.5, 3.0, True, epoch)
        assert len(seen) == len(live) and set(seen) == live
    r.finish()


def _visit_bound(fg, colors, lne):
    """Sum over colours of the most visits one weight gets in a colour (color_visit_bounds)."""
    fm, fac, w, var = fg.fmap, fg.factor, fg.weight, fg.variable
    fidx = np.repeat(np.arange(len(fac)), fac["arity"])
    vid, wid = fm["vid"], fac["weightId"][fidx]
    ev = var["isEvidence"][vid]
    keep = (ev != 4) & (colors[vid] >= 0) & ~w["isFixed"][wid].astype(bool) & (bool(lne) | (ev == 1))
    hist = np.zeros((int(colors.max()) + 1, len(w)), np.int64)
    np.add.at(hist, (colors[vid[keep]], wid[keep]), 1)
    return int(hist.max(axis=1).sum())


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["pair_blocks", "lf_many", "warp_crowd"])
def test_large_learning_modes_agree_bit_for_bit(name, monkeypatch):
    """Whole epochs (FactorGraph.learn, decaying step) of 3 blocks of large cells: the persistent
    launch (mode 1: rotating tables, next-cell range lookup, per-CTA weight copies) and the lean
    launches (mode 2) give identical weights and chains.  Both modes take the same truth-table
    branch in every cell -- slices on the tied grid, rows on the long-row label colour and on the
    corner rows of the warp grid -- since the two branches sum the float64 energies in different
    orders.  The warp grid's Boolean warp rows reduce with shuffles, in the same order in both modes."""
    import ctypes as C
    import numbskull_b200 as nb
    lne, step = True, 0.01
    r = Replay(name)
    bv = -(-_visit_bound(r.fg, r.colors, lne) // 3)
    n_blocks = C.c_int(0)
    r._chk(r.L.nb_learn_blocks(r.g, step, int(lne), bv, C.byref(n_blocks)))
    assert n_blocks.value == 3
    sms = _sms()
    for mode in (1, 2):
        for b in range(3):
            for c in range(r.info["n_colors"]):
                br = learn_branches(r, c, r.cell_ids(c, b, 3), mode, sms)
                if name == "pair_blocks":
                    assert "tt_slices_tied" in br, (mode, b, c, br)
                else:
                    assert "tt_slices" not in br, (mode, b, c, br)
    r.fg.clear()
    g, attrs, _ = _spec(name)
    runs = []
    for mode in ("1", "2"):
        monkeypatch.setenv("NUMBSKULL_B200_LEARN_MODE", mode)
        ns = nb.NumbSkull(quiet=True)
        ns.loadFactorGraph(*g)
        fg = ns.factorGraphs[0]
        fg.seed, fg.batch_visits = SEED, bv
        for k, v in attrs.items():
            setattr(fg, k, v)
        fg.learn(0, 4, step, 0.9, 2, 0.01, 1, learn_non_evidence=lne)
        runs.append((fg.weight_value.copy(), fg.var_value.copy(), fg.var_value_evid.copy()))
        fg.clear()
    for a, b in zip(runs[0], runs[1]):
        assert np.array_equal(a, b)
