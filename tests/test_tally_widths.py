"""The tallies at every width they cross PCIe with.

k_counts_to_old narrows the int32 device tallies to 1, 2 or 4 bytes for the copy to the host, by a
bound the library keeps on the host (no tally may exceed it), and the host widens them back in
chunks of 2^18 entries, with non-temporal stores behind a scalar prologue.  Every reader
(nb_get_counts with and without accumulate, nb_get_counts_marginals, nb_get_marginals,
nb_get_counts_compact) is compared exactly with numpy: installed counts plus the tallies the replay
derives from the values the GPU drew (test_sweep_replay.Replay.tally), on both sides of the 255 /
256 and 65535 / 65536 edges and up to the int32 top.

The graph ("tally_chunks") has PAIR / FAST rows (which tally into count_b), cardinality-40 GEN rows
and 840586 tallies: three full chunks, a short last one, and a count that is not a multiple of 4.
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
if HERE not in sys.path:
    sys.path.insert(0, HERE)

from test_sweep_replay import REPO, SEED, Replay   # noqa: E402

BOUNDS = (254, 255, 65534, 65535, (1 << 31) - 3)
DIVISOR = 3.0
INT32_MAX = (1 << 31) - 1


def _dtype(bound):
    return np.uint8 if bound <= 255 else (np.uint16 if bound <= 65535 else np.int32)


def _misaligned(n, dtype):
    """n zeros starting 8 bytes past a 32-byte boundary: the widening loops run their scalar prologue."""
    buf = np.zeros(n + 4, dtype)
    a = buf[(8 - buf.ctypes.data % 32) % 32 // 8:][:n]
    assert a.ctypes.data % 32 == 8
    return a


def _same(what, got, want):
    bad = np.nonzero(got.view(np.int64) != want.view(np.int64))[0] if got.dtype == np.float64 else \
        np.nonzero(got != want)[0]
    assert len(bad) == 0, "%s: %d of %d entries differ, first at %d: %r against %r" % (
        what, len(bad), len(want), bad[0], got[bad[0]], want[bad[0]])


def _check_readers(r, want, bound):
    """Every reader of the tallies against `want` (int64, cstart layout); no tally exceeds `bound`."""
    L, lib, n = r.L, r._lib, len(want)
    assert want.max() <= bound
    got = _misaligned(n, np.int64)
    r._chk(L.nb_get_counts(r.g, lib.ptr(got), 0))
    _same("nb_get_counts", got, want)
    base = (1 << 31) + 12345 + np.arange(n, dtype=np.int64) * 977          # accumulate onto values above 2^31
    got[:] = base
    r._chk(L.nb_get_counts(r.g, lib.ptr(got), 1))
    _same("nb_get_counts, accumulate", got, base + want)
    got[:] = base
    m = _misaligned(n, np.float64)
    r._chk(L.nb_get_counts_marginals(r.g, lib.ptr(got), 1, lib.ptr(m), DIVISOR))
    _same("nb_get_counts_marginals counts", got, base + want)
    _same("nb_get_counts_marginals marginals", m, (base + want).astype(np.float64) / DIVISOR)
    m[:] = -1.0
    r._chk(L.nb_get_marginals(r.g, lib.ptr(m), DIVISOR))
    _same("nb_get_marginals", m, want.astype(np.float64) / DIVISOR)
    c = r.fg.counts_compact()
    assert c.dtype == _dtype(bound), (c.dtype, bound)
    _same("counts_compact", c.astype(np.int64), want)


def _graph():
    r = Replay("tally_chunks")
    n = int(r.cstart[-1])
    assert n > 3 * (1 << 18) and n % 4 != 0
    return r, n


def _live(r):
    return r.sampled(True) & (r.colors >= 0)


def _install(r, c):
    c = np.ascontiguousarray(c, np.int64)
    r._chk(r.L.nb_set_counts(r.g, r._lib.ptr(c)))
    return c


def _sweep(r, burnin=0):
    r._chk(r.L.nb_gibbs_sweeps(r.g, 1, burnin, 1, SEED))


def _phase(r, color, epoch, burnin=0):
    r._chk(r.L.nb_gibbs_color_phase(r.g, color, burnin, 1, SEED, epoch))


def run_widths():
    """For each bound: counts up to it installed, then one tallying sweep, then one tallying colour
    phase; every reader after each step."""
    r, n = _graph()
    rng = np.random.default_rng(7)
    bslots = r.cstart[:-1][r.card == 2]
    for bound in BOUNDS:
        r.random_state(rng, weights=False)
        c = rng.integers(0, bound + 1, n)
        c[bslots[rng.random(len(bslots)) < 0.5]] = bound
        c[-1] = bound
        want = _install(r, c)
        _check_readers(r, want, bound)
        _sweep(r)
        want = want + r.tally(np.nonzero(_live(r))[0], r.get_vals(0))
        _check_readers(r, want, bound + 1)
        _phase(r, 0, 1 << 40)
        want = want + r.tally(np.nonzero(_live(r) & (r.colors == 0))[0], r.get_vals(0))
        _check_readers(r, want, bound + 2)
        print("bound %d: %d tallies at %d, %d and %d bytes" % (
            bound, n, *[np.dtype(_dtype(b)).itemsize for b in (bound, bound + 1, bound + 2)]))
    r.fg.clear()


@pytest.mark.gpu
@pytest.mark.parametrize("threads", ["1", "5"])
def test_tallies_at_every_width(threads):
    """NUMBSKULL_B200_HOST_THREADS is read once per process: a child interpreter per value."""
    env = dict(os.environ, NUMBSKULL_B200_HOST_THREADS=threads)
    code = "import sys; sys.path[:0] = [%r, %r]; import test_tally_widths as t; t.run_widths()" % (REPO, HERE)
    p = subprocess.run([sys.executable, "-c", code], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                       text=True)
    print(p.stdout[-4000:])
    assert p.returncode == 0


@pytest.mark.gpu
def test_colour_phases_at_one_epoch_raise_the_bound():
    """nb_gibbs_color_phase may run a colour twice at one epoch, and a first call may come at
    epoch -1: each tallying launch can add 1 to a tally, whatever its epoch."""
    r, n = _graph()
    ids = np.nonzero(_live(r) & (r.colors == 0))[0]
    want = _install(r, np.full(n, 255))            # a fresh graph: its first tallying call at epoch -1
    _phase(r, 0, -1)
    want = want + r.tally(ids, r.get_vals(0))
    assert want.max() == 256
    _check_readers(r, want, 256)
    want = _install(r, np.full(n, 254))
    for k in (1, 2):                                 # colour 0 twice at epoch 9
        r.random_state(np.random.default_rng(k), weights=False)
        _phase(r, 0, 9)
        want = want + r.tally(ids, r.get_vals(0))
        _check_readers(r, want, 254 + k)
    assert want.max() == 256
    r.fg.clear()


@pytest.mark.gpu
def test_tallies_stop_at_the_int32_top():
    """Counts installed at 2^31 - 2 take one tallying sweep (exact, through the int32 path); the next
    tallying sweep or phase is refused before anything runs, burn-in sweeps stay allowed, and a
    reset lets the sweeps go on."""
    r, n = _graph()
    L, g = r.L, r.g
    want = _install(r, np.full(n, INT32_MAX - 1))
    _sweep(r)
    want = want + r.tally(np.nonzero(_live(r))[0], r.get_vals(0))
    assert want.max() == INT32_MAX
    _check_readers(r, want, INT32_MAX)
    vals = (r.get_vals(0), r.get_vals(1))
    e = C.c_int64(0)
    r._chk(L.nb_begin_epoch(g, C.byref(e)))
    e0 = e.value
    refused = []
    for what, call in (("sweep", lambda: _sweep(r)), ("phase", lambda: _phase(r, 0, 3))):
        try:
            call()
        except NotImplementedError:
            refused.append(what)
        got = r.counts()
        assert got.min() >= 0, "%s: tallies wrapped past 2^31 - 1 (smallest %d)" % (what, got.min())
        _same("tallies after the refused " + what, got, want)
        for chain in (0, 1):
            assert np.array_equal(r.get_vals(chain), vals[chain]), (what, "values changed")
    assert refused == ["sweep", "phase"]
    r._chk(L.nb_begin_epoch(g, C.byref(e)))
    assert e.value == e0 + 1, "the refused sweep advanced the epoch counter"
    _sweep(r, burnin=1)                              # burn-in: no tallies
    _phase(r, 1, 5, burnin=1)
    _same("tallies after burn-in", r.counts(), want)
    assert not np.array_equal(r.get_vals(0), vals[0])
    r._chk(L.nb_reset_counts(g))
    _sweep(r)
    _same("tallies after a reset", r.counts(), r.tally(np.nonzero(_live(r))[0], r.get_vals(0)))
    r.fg.clear()
