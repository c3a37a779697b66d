"""ctypes front-end of ``nb_oracle.c`` (TEST INFRASTRUCTURE ONLY).

``OracleGraph`` mirrors the state ``FactorGraph.__init__`` builds in the
reference (numbskull/factorgraph.py:30-73) and drives the C restatement of
``gibbsthread`` / ``learnthread`` over it.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libnb_oracle.so")
_lib = None


def build(force=False):
    """Compile the oracle with gcc (no GPU, no reference sources involved)."""
    src = os.path.join(_HERE, "nb_oracle.c")
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(src):
        subprocess.check_call(["make", "-s", "-C", _HERE, "libnb_oracle.so"])
    return _SO


class _Graph(C.Structure):
    _fields_ = [
        ("weight", C.c_void_p), ("n_weight", C.c_int64),
        ("variable", C.c_void_p), ("n_var", C.c_int64),
        ("factor", C.c_void_p), ("n_factor", C.c_int64),
        ("fmap", C.c_void_p), ("n_fmap", C.c_int64),
        ("vmap", C.c_void_p), ("n_vmap", C.c_int64),
        ("factor_index", C.c_void_p), ("n_findex", C.c_int64),
        ("cstart", C.c_void_p),
        ("count", C.c_void_p),
        ("var_value", C.c_void_p),
        ("var_value_evid", C.c_void_p),
        ("weight_value", C.c_void_p),
    ]


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_SO)
        L.nbo_eval_factor.restype = C.c_double
        L.nbo_eval_factor.argtypes = [C.POINTER(_Graph), C.c_int64, C.c_int64, C.c_int64,
                                      C.c_void_p, C.POINTER(C.c_int)]
        L.nbo_potential.restype = C.c_double
        L.nbo_potential.argtypes = [C.POINTER(_Graph), C.c_int64, C.c_int64, C.c_void_p,
                                    C.POINTER(C.c_int)]
        L.nbo_pool_create.restype = C.c_void_p
        L.nbo_pool_create.argtypes = [C.POINTER(_Graph), C.c_int, C.c_uint32]
        L.nbo_pool_destroy.argtypes = [C.c_void_p]
        L.nbo_gibbs_epochs.restype = C.c_int
        L.nbo_gibbs_epochs.argtypes = [C.POINTER(_Graph), C.c_void_p, C.c_int64, C.c_int, C.c_int]
        L.nbo_learn_epochs.restype = C.c_int
        L.nbo_learn_epochs.argtypes = [C.POINTER(_Graph), C.c_void_p, C.c_int64,
                                       C.POINTER(C.c_double), C.c_double, C.c_int, C.c_double,
                                       C.c_double, C.c_int]
        L.nbo_compute_var_map.restype = None
        L.nbo_compute_var_map.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64,
                                          C.c_void_p, C.c_int64, C.c_void_p, C.c_int64,
                                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]
        L.nbo_exact_marginals.restype = C.c_int
        L.nbo_exact_marginals.argtypes = [C.POINTER(_Graph), C.c_int, C.c_void_p,
                                          C.POINTER(C.c_double)]
        L.nbo_mt_seed.argtypes = [C.c_void_p, C.c_uint32]
        L.nbo_mt_double.restype = C.c_double
        L.nbo_mt_double.argtypes = [C.c_void_p]
        u32p = C.POINTER(C.c_uint32)
        L.nbo_philox4x32.argtypes = [u32p, u32p, u32p]
        L.nbo_philox2x32.argtypes = [u32p, C.c_uint32, u32p]
        L.nbo_u53.restype = C.c_double
        L.nbo_u53.argtypes = [C.c_uint32, C.c_uint32]
        L.nbo_fold_key.restype = C.c_uint32
        L.nbo_fold_key.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32]
        L.nbo_philox2x32_u53.restype = C.c_double
        L.nbo_philox2x32_u53.argtypes = [C.c_uint32, C.c_uint64, C.c_uint64, C.c_uint32]
        L.nbo_stream_init.argtypes = [C.c_void_p, C.c_uint32, C.c_uint64, C.c_uint32, C.c_uint64]
        L.nbo_stream_word.restype = C.c_uint32
        L.nbo_stream_word.argtypes = [C.c_void_p]
        L.nbo_stream_next.restype = C.c_double
        L.nbo_stream_next.argtypes = [C.c_void_p]
        L.nbo_stream_next32.restype = C.c_double
        L.nbo_stream_next32.argtypes = [C.c_void_p]
        L.nbo_draw_bool.restype = C.c_int64
        L.nbo_draw_bool.argtypes = [C.c_double, C.c_double, C.c_double, C.POINTER(C.c_double)]
        L.nbo_draw_cdf.restype = C.c_int64
        L.nbo_draw_cdf.argtypes = [C.c_void_p, C.c_int64, C.c_double, C.POINTER(C.c_double)]
        L.nbo_draw_reservoir.restype = C.c_int64
        L.nbo_draw_reservoir.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.POINTER(C.c_double)]
        L.nbo_energies.restype = C.c_int
        L.nbo_energies.argtypes = [C.POINTER(_Graph), C.c_int, C.c_void_p, C.c_int64, C.c_void_p]
        L.nbo_replay_draws.restype = C.c_int
        L.nbo_replay_draws.argtypes = [C.POINTER(_Graph), C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                                       C.c_uint64, C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p]
        L.nbo_first_uniforms.restype = None
        L.nbo_first_uniforms.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32,
                                         C.c_void_p]
        L.nbo_cell_gradients.restype = C.c_int
        L.nbo_cell_gradients.argtypes = [C.POINTER(_Graph), C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_void_p, C.c_void_p]
        L.nbo_sizeof_stream.restype = C.c_int
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _raise(err):
    if err & 1:
        raise NotImplementedError("Factor function is not implemented.")


def compute_var_map(variable, factor, fmap, vmap, factor_index, domain_mask,
                    factors_to_skip=None):
    """dataloading.py:16-81, in place on the caller's record arrays."""
    if factors_to_skip is None:
        factors_to_skip = np.empty(0, np.int64)
    dm = np.ascontiguousarray(domain_mask, dtype=np.uint8)
    lib().nbo_compute_var_map(_p(variable), len(variable), _p(factor), len(factor),
                              _p(fmap), len(fmap), _p(vmap), len(vmap), _p(factor_index),
                              _p(dm), _p(factors_to_skip), len(factors_to_skip))


# ---------------------------------------------------------------------------
# Counter-based streams of the CUDA library (restated in nb_oracle.c)
# ---------------------------------------------------------------------------
TAG_FREE, TAG_EVID, TAG_TRUNC = 0, 1, 2
PAIR, FAST, CAT, GEN, WARP, WIDE = range(6)   # row classes (WIDE: warp rows above cardinality 255)
GRAD_UNIT = float(1 << 20)                     # the library reduces gradients in 2^-20 units


def philox4x32(ctr, key):
    """Philox4x32-10 of a 4-word counter and 2-word key -> 4 words."""
    c, k, o = (C.c_uint32 * 4)(*ctr), (C.c_uint32 * 2)(*key), (C.c_uint32 * 4)()
    lib().nbo_philox4x32(c, k, o)
    return list(o)


def philox2x32(ctr, key):
    """Philox2x32-10 of a 2-word counter and 1-word key -> 2 words."""
    c, o = (C.c_uint32 * 2)(*ctr), (C.c_uint32 * 2)()
    lib().nbo_philox2x32(c, key, o)
    return list(o)


def u53(hi, lo):
    return lib().nbo_u53(hi, lo)


def fold_key(seed, epoch, tag):
    return lib().nbo_fold_key(seed, epoch, tag)


def philox2x32_u53(rid, epoch, seed, tag):
    """The single uniform of a record row in sweep `epoch`."""
    return lib().nbo_philox2x32_u53(rid, epoch, seed, tag)


class Stream(object):
    """The multi-draw uniform stream of one (variable, epoch, tag)."""

    def __init__(self, rid, epoch, tag, seed):
        self._s = C.create_string_buffer(lib().nbo_sizeof_stream())
        lib().nbo_stream_init(self._s, rid, epoch, tag, seed)

    def word(self):
        return lib().nbo_stream_word(self._s)

    def next(self):
        return lib().nbo_stream_next(self._s)

    def next32(self):
        return lib().nbo_stream_next32(self._s)


def draw_bool(e0, e1, u):
    """-> (pick, margin) of the Boolean rule."""
    m = C.c_double(0)
    return lib().nbo_draw_bool(e0, e1, u, C.byref(m)), m.value


def draw_cdf(e, u):
    e = np.ascontiguousarray(e, np.float64)
    m = C.c_double(0)
    return lib().nbo_draw_cdf(_p(e), len(e), u, C.byref(m)), m.value


def draw_reservoir(e, stream, nonempty=None):
    e = np.ascontiguousarray(e, np.float64)
    ne = None if nonempty is None else np.ascontiguousarray(nonempty, np.uint8)
    m = C.c_double(0)
    return lib().nbo_draw_reservoir(_p(e), len(e), None if ne is None else _p(ne), stream._s, C.byref(m)), m.value


def first_uniforms(rng_id, family, seed, epoch, tag):
    """First uniform of each stream: family 0 = Philox2x32 (record rows), 1 = multi-draw stream."""
    rid = np.ascontiguousarray(rng_id, np.uint32)
    fam = np.ascontiguousarray(family, np.int32)
    out = np.empty(len(rid), np.float64)
    lib().nbo_first_uniforms(_p(rid), len(rid), _p(fam), seed, epoch, tag, _p(out))
    return out


class OracleGraph(object):
    """State of one factor graph, as the reference's FactorGraph keeps it."""

    def __init__(self, weight, variable, factor, fmap, vmap, factor_index, nthreads=1, seed=0):
        for a, sz in ((weight, 9), (variable, 27), (factor, 34), (fmap, 16), (vmap, 24)):
            assert a.dtype.itemsize == sz and a.flags.c_contiguous
        assert factor_index.dtype == np.int64
        self.weight, self.variable, self.factor = weight, variable, factor
        self.fmap, self.vmap, self.factor_index = fmap, vmap, factor_index
        nvar = len(variable)
        # factorgraph.py:40-46
        cs = np.empty(nvar + 1, np.int64)
        cs[0] = 0
        cs[1:] = variable["cardinality"]
        cs[cs == 2] = 1
        self.cstart = np.cumsum(cs)
        self.count = np.zeros(int(self.cstart[nvar]), np.int64)
        self.var_value = np.ascontiguousarray(variable["initialValue"], dtype=np.int64).copy()
        self.var_value_evid = self.var_value.copy()
        self.weight_value = np.ascontiguousarray(weight["initialValue"], dtype=np.float64).copy()
        self.marginals = np.zeros(len(self.count))
        self.nthreads = nthreads
        self._g = _Graph(_p(weight), len(weight), _p(variable), nvar, _p(factor), len(factor),
                         _p(fmap), len(fmap), _p(vmap), len(vmap), _p(factor_index),
                         len(factor_index), _p(self.cstart), _p(self.count), _p(self.var_value),
                         _p(self.var_value_evid), _p(self.weight_value))
        self._pool = lib().nbo_pool_create(C.byref(self._g), nthreads, seed)

    def __del__(self):
        if getattr(self, "_pool", None):
            lib().nbo_pool_destroy(self._pool)
            self._pool = None

    def eval_factor(self, factor_id, var_samp, value, evid_chain=False):
        err = C.c_int(0)
        vals = self.var_value_evid if evid_chain else self.var_value
        r = lib().nbo_eval_factor(C.byref(self._g), factor_id, var_samp, value, _p(vals),
                                  C.byref(err))
        _raise(err.value)
        return r

    def potential(self, var_samp, value, evid_chain=False):
        err = C.c_int(0)
        vals = self.var_value_evid if evid_chain else self.var_value
        r = lib().nbo_potential(C.byref(self._g), var_samp, value, _p(vals), C.byref(err))
        _raise(err.value)
        return r

    def potentials(self, evid_chain=False):
        """Energies for every (variable, value), laid out per variable in
        ``cardinality`` consecutive entries (NOT the count layout)."""
        out = []
        for v in range(len(self.variable)):
            for k in range(int(self.variable[v]["cardinality"])):
                out.append(self.potential(v, k, evid_chain))
        return np.array(out)

    def energies(self, ids, evid_chain=False):
        """potential(v, k) for every value of the listed variables, concatenated (batched)."""
        ids = np.ascontiguousarray(ids, np.int64)
        out = np.empty(int(self.variable["cardinality"][ids].astype(np.int64).sum()), np.float64)
        _raise(lib().nbo_energies(C.byref(self._g), int(bool(evid_chain)), _p(ids), len(ids), _p(out)))
        return out

    def replay_draws(self, ids, cls, rng_id, seed, epoch, tag, evid_chain=False):
        """float64 replay of the library's draw of each listed variable under the current state:
        returns (pick, margin); see nbo_replay_draws."""
        ids = np.ascontiguousarray(ids, np.int64)
        cls = np.ascontiguousarray(cls, np.int32)
        rid = np.ascontiguousarray(rng_id, np.uint32)
        pick = np.empty(len(ids), np.int64)
        margin = np.empty(len(ids), np.float64)
        _raise(lib().nbo_replay_draws(C.byref(self._g), int(bool(evid_chain)), _p(ids), len(ids), _p(cls), _p(rid),
                                      seed, epoch, tag, _p(pick), _p(margin)))
        return pick, margin

    def cell_gradients(self, ids, ev, prop, cnt_inc):
        """Per-weight fixed-point gradient sums (2^-20 units) and visit counts of one learning cell
        whose variables `ids` drew `ev` (evidence chain) and `prop` (free chain)."""
        ids = np.ascontiguousarray(ids, np.int64)
        ev = np.ascontiguousarray(ev, np.int64)
        prop = np.ascontiguousarray(prop, np.int64)
        ci = np.ascontiguousarray(cnt_inc, np.uint32)
        G = np.zeros(len(self.weight), np.int64)
        cnt = np.zeros(len(self.weight), np.int64)
        _raise(lib().nbo_cell_gradients(C.byref(self._g), _p(ids), len(ids), _p(ev), _p(prop), _p(ci), _p(G),
                                        _p(cnt)))
        return G, cnt

    def burnIn(self, epochs, sample_evidence):
        _raise(lib().nbo_gibbs_epochs(C.byref(self._g), self._pool, epochs,
                                      int(bool(sample_evidence)), 1))

    def inference(self, burnin_epochs, epochs, sample_evidence=False):
        """factorgraph.py:145-175."""
        if burnin_epochs > 0:
            self.burnIn(burnin_epochs, sample_evidence)
        _raise(lib().nbo_gibbs_epochs(C.byref(self._g), self._pool, epochs,
                                      int(bool(sample_evidence)), 0))
        if epochs != 0:
            self.marginals = self.count / float(epochs)

    def learn(self, burnin_epochs, epochs, stepsize, decay, regularization, reg_param,
              truncation, learn_non_evidence=False):
        """factorgraph.py:177-208; returns the final stepsize."""
        if burnin_epochs > 0:
            self.burnIn(burnin_epochs, True)
        step = C.c_double(stepsize)
        _raise(lib().nbo_learn_epochs(C.byref(self._g), self._pool, epochs, C.byref(step),
                                      decay, regularization, reg_param, float(truncation),
                                      int(bool(learn_non_evidence))))
        return step.value


def exact_marginals(og, clamp_evidence=False):
    """Brute-force marginals in the ``count`` layout (tiny graphs only)."""
    out = np.zeros(len(og.count))
    logz = C.c_double(0)
    _raise(lib().nbo_exact_marginals(C.byref(og._g), int(clamp_evidence), _p(out),
                                     C.byref(logz)))
    return out
