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

Tolerance, the same everywhere: the GPU may pick differently from the float64 replay only where
the replay's decision margin (distance of the uniform to the nearest point that changes the pick)
is below NEAR_TIE -- the fp32 exp / CDFs / inlined weights of the kernels.  Such near-ties are
counted, printed, and must stay below 1e-4 of the draws.

The Philox known answers and the comparison with the library's own host-callable Philox
functions (compiled from its header by nvcc into a temporary directory) run without a GPU.
"""
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
def _graph(seed, nvar=3000, nfac=6000, cat_frac=0.0, cat_cards=(6, 12), dt0_cards=(2,), funcs0=(0, 1, 2, 3, 4, 7, 9),
           funcs1=(12, 14, 15), max_arity=4, hubs=0, hub_degree=150, evidence_frac=0.3, ghost_frac=0.0,
           fixed_frac=0.2, n_weights=None, w_scale=1.0, feature_values=False, wide_arity=0, ratio=False):
    """Random graph for the replay.  dataType-0 variables (cardinalities from dt0_cards) share
    factors of funcs0 (plus RATIO if `ratio`); dataType-1 variables (cardinalities in cat_cards)
    factors of funcs1 with dense_equal_to below each member's cardinality.  `hubs` variables get
    `hub_degree` extra pairwise factors each (long rows: warp path with several tasks)."""
    from numbskull_b200.numbskulltypes import Weight, Variable, Factor, FactorToVar
    rng = np.random.default_rng(seed)
    variable = np.zeros(nvar, Variable)
    cat = rng.random(nvar) < cat_frac
    card = rng.choice(np.array(dt0_cards), nvar)
    card[cat] = rng.integers(cat_cards[0], cat_cards[1] + 1, int(cat.sum()))
    variable["dataType"] = cat
    variable["cardinality"] = card
    ev = rng.random(nvar) < evidence_frac
    variable["isEvidence"] = ev
    variable["isEvidence"][rng.random(nvar) < ghost_frac] = 4
    variable["initialValue"] = rng.integers(0, 1 << 30, nvar) % card
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
    hub_ids = rng.choice(ids0 if len(ids0) else ids1, hubs, replace=False) if hubs else []
    for h in hub_ids:
        pool = ids0 if variable["dataType"][h] == 0 else ids1
        for _ in range(hub_degree):
            o = int(rng.choice(pool))
            facs.append(int(rng.choice((3, 7, 9)) if variable["dataType"][h] == 0 else 12))
            members.append(np.array([h, o] if o != h else [h]))
    if wide_arity:                                   # one long factor: 2-word incidence headers
        facs.append(7)
        members.append(rng.choice(ids0, wide_arity, replace=False))
    nf = len(facs)
    n_weights = n_weights or max(1, nf // 3)
    weight = np.zeros(n_weights, Weight)
    weight["isFixed"] = rng.random(n_weights) < fixed_frac
    weight["initialValue"] = rng.normal(0, w_scale, n_weights)
    factor = np.zeros(nf, Factor)
    factor["factorFunction"] = facs
    factor["weightId"] = rng.integers(0, n_weights, nf)
    factor["featureValue"] = rng.choice([1.0, 0.5, 2.0], nf) if feature_values else 1.0
    factor["arity"] = [len(m) for m in members]
    factor["ftv_offset"] = np.concatenate(([0], np.cumsum(factor["arity"])[:-1]))
    vids = np.concatenate(members).astype(np.int64)
    fmap = np.zeros(len(vids), FactorToVar)
    fmap["vid"] = vids
    fmap["dense_equal_to"] = rng.integers(0, 1 << 30, len(vids)) % card[vids]
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
    raise KeyError(name)


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
                "saturating", "wide_headers", "global_vid", "wide_card", "wide_card_thread"]


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
    r.finish()


# =========================================================================== GPU: whole sweeps
def _whole_sweeps(name, sample_evidence):
    r = Replay(name)
    r.whole_sweeps(4, sample_evidence)
    r.finish()


@pytest.mark.gpu
@pytest.mark.parametrize("name,mirror", [("fast", "-1"), ("fast", "0"), ("warp", "-1"), ("gen_cat_empty", "-1"),
                                         ("wide_card", "-1")])
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
]


def _learn(r, reg, lne, n_blocks_list, rng):
    step, reg_param, trunc = 0.05, 0.5, 3.0
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
    r.finish()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["wide_card", "wide_card_thread"])
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
