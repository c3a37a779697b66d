"""FactorGraph: the drop-in seam (reference: numbskull/factorgraph.py:27-229).

Same constructor signature, public arrays and methods as the reference class.
The epoch loops that used to hand the arrays to the numba ``gibbsthread`` /
``learnthread`` through ``run_pool`` (factorgraph.py:13-24, :135-141, :156-163,
:196-202) call the CUDA library instead.  ``workers`` (nthreads) is accepted and
ignored on the GPU.

Host / device coherence.  The reference mutates its numpy arrays in place, so
state simply persists between calls.  Here the working copy lives in HBM and
the public arrays (``var_value``, ``var_value_evid``, ``weight_value``,
``count``, ``marginals``) are properties over host mirrors:

* an array the caller never touched is NOT copied at call boundaries: the
  device copy is authoritative and the host mirror is refreshed lazily, the
  first time somebody reads the attribute (``marginals`` is computed from the
  device tallies at that moment, without materialising the int64 ``count``);
* an array the caller has obtained a reference to (read or assigned the
  attribute) may be edited behind our back (salt/src/numbskull_master.py:213-224
  pokes ``var_value`` / ``weight_value`` between calls), so from then on it is
  uploaded on entry to ``burnIn`` / ``inference`` / ``learn`` and refreshed on
  exit -- the round-trip behaviour of the reference, at its cost;
* ``weight_value`` is small: it is compared with the last uploaded copy on
  entry and downloaded after every ``learn``;
* the record arrays (``variable`` / ``weight`` / ``factor`` / ``fmap``) are read
  once, when the device graph is built.  ``variable.isEvidence``,
  ``variable.initialValue`` and ``weight.isFixed`` -- the fields the reference
  reads on every sweep -- are edited in place with :meth:`update_variables` /
  :meth:`update_weights`, which write the records and patch the device graph
  without a rebuild.  Any other record edit (cardinality, dataType,
  featureValue, weightId, factors, fmap), or an edit of those fields made
  directly in the arrays, needs :meth:`invalidate`.
"""
from __future__ import print_function

import ctypes as C
import os
import sys

import numpy as np

from . import _lib
from .timer import Timer


def _default_seed():
    env = os.environ.get("NUMBSKULL_B200_SEED")
    if env is not None:
        return int(env) & 0xFFFFFFFFFFFFFFFF
    return int.from_bytes(os.urandom(8), "little")


class FactorGraph(object):
    """Device-backed factor graph with the reference's interface."""

    def __init__(self, weight, variable, factor, fmap, vmap, factor_index,
                 var_copies, weight_copies, fid, workers, device=None, seed=None):
        self.weight = weight
        self.variable = variable
        self.factor = factor
        self.fmap = fmap
        self.vmap = vmap
        self.factor_index = factor_index

        nvar = self.variable.shape[0]
        # exclusive cumsum of (1 if cardinality == 2 else cardinality), factorgraph.py:40-45
        per_var = self.variable["cardinality"].astype(np.int64)
        per_var[per_var == 2] = 1
        self.cstart = np.zeros(nvar + 1, np.int64)
        np.cumsum(per_var, out=self.cstart[1:])

        init = self.variable["initialValue"].astype(np.int64)
        self._var_value_evid = np.tile(init, (var_copies, 1))
        self._var_value = np.tile(init, (var_copies, 1))
        self._weight_value = np.tile(self.weight["initialValue"].astype(np.float64),
                                     (weight_copies, 1))
        self._count = np.zeros(self.cstart[nvar], np.int64)
        self._marginals = np.zeros(self.cstart[nvar])
        # coherence state (see the module docstring)
        self._dev_row = {"var_value": None, "var_value_evid": None, "weight_value": None}  # host row held in HBM
        self._stale = set()       # host mirrors older than the device copy
        self._exposed = set()     # arrays the caller holds a reference to
        self._w_shadow = None     # weights as last uploaded / downloaded
        self._count_dev_valid = True   # device tallies == count (both zero at creation)
        self._marg_epochs = 0
        self._pristine = True

        # scratch the reference exposes; kept for shape compatibility only
        maxcard = int(self.variable["cardinality"].max()) if nvar else 0
        self.Z = np.zeros((workers, maxcard))
        maxlen = int(self.vmap["factor_index_length"].max()) if self.vmap.size else 0
        self.fids = np.zeros((workers, 2 * maxlen), factor_index.dtype)

        self.fid = fid
        assert(workers > 0)
        self.threads = workers
        self.inference_epoch_time = 0.0
        self.inference_total_time = 0.0
        self.learning_epoch_time = 0.0
        self.learning_total_time = 0.0

        # ---- device side ----
        self.device = device if device is not None else int(os.environ.get("LOCAL_RANK", 0))
        self.seed = _default_seed() if seed is None else int(seed)
        self.color_seed = int(os.environ.get("NUMBSKULL_B200_COLOR_SEED", 0x5EED))
        self.batch_visits = 0          # learning mini-batch policy, 0 = library default
        self.global_vid = None         # set by the partitioner for multi-GPU graphs
        self.preset_color = None
        self.warp_row_words = int(os.environ.get("NUMBSKULL_B200_WARP_ROW_WORDS", 0))  # 0 = default
        self.sigma_shift = int(os.environ.get("NUMBSKULL_B200_SIGMA_SHIFT", 0))        # 0 = default
        self.deferred_coloring = False  # partitioned graphs: colouring is driven by partition.py
        self._g = None

    # ------------------------------------------------------------------
    # device graph management
    # ------------------------------------------------------------------
    def _device_graph(self):
        """Build (once) the HBM-resident form of the graph."""
        if self._g is None:
            L = _lib.lib()
            self._keep = dict(
                weight=np.ascontiguousarray(self.weight), variable=np.ascontiguousarray(self.variable),
                factor=np.ascontiguousarray(self.factor), fmap=np.ascontiguousarray(self.fmap),
                vmap=np.ascontiguousarray(self.vmap),
                factor_index=_lib.contiguous(self.factor_index, np.int64),
                global_vid=None if self.global_vid is None else _lib.contiguous(self.global_vid, np.int64),
                preset_color=None if self.preset_color is None else _lib.contiguous(self.preset_color, np.int32))
            k = self._keep
            desc = _lib.GraphDesc(
                _lib.ptr(k["weight"]), len(k["weight"]), _lib.ptr(k["variable"]), len(k["variable"]),
                _lib.ptr(k["factor"]), len(k["factor"]), _lib.ptr(k["fmap"]), len(k["fmap"]),
                _lib.ptr(k["vmap"]), len(k["vmap"]), _lib.ptr(k["factor_index"]), len(k["factor_index"]),
                self.device, self.color_seed, _lib.ptr(k["global_vid"]),
                int(self.warp_row_words), int(self.sigma_shift), _lib.ptr(k["preset_color"]),
                int(bool(self.deferred_coloring)))
            g = C.c_void_p()
            _lib.check(L.nb_graph_create(C.byref(desc), C.byref(g)))
            self._g = g
            self._keep = None
            if self._pristine:
                # nb_graph_create starts both chains at initialValue == row 0 of the untouched mirrors
                for name in ("var_value", "var_value_evid"):
                    if name not in self._exposed:
                        self._dev_row[name] = 0
            self._pristine = False
        return self._g

    def device_info(self):
        info = _lib.GraphInfo()
        _lib.check(_lib.lib().nb_graph_get_info(self._device_graph(), C.byref(info)))
        return info.as_dict()

    def colors(self):
        """Colour of every variable (original order); -1 for non-owned variables."""
        out = np.empty(self.variable.shape[0], np.int32)
        _lib.check(_lib.lib().nb_graph_get_colors(self._device_graph(), _lib.ptr(out)))
        return out

    def color_edges(self):
        n = self.device_info()["n_colors"]
        out = np.zeros(max(n, 1), np.int64)
        _lib.check(_lib.lib().nb_graph_color_edges(self._device_graph(), _lib.ptr(out)))
        return out[:n]

    def potentials(self, var_ids=None, evid_chain=False, var_copy=0, weight_copy=0):
        """Conditional energies potential(v, k) (inference.py:55-71) for every
        value of the given variables, concatenated per variable."""
        g = self._device_graph()
        self._sync_device(var_copy, weight_copy)
        if var_ids is None:
            var_ids = np.arange(self.variable.shape[0], dtype=np.int64)
        var_ids = _lib.contiguous(var_ids, np.int64)
        cards = self.variable["cardinality"][var_ids].astype(np.int64)
        offs = np.zeros(len(var_ids), np.int64)
        if len(var_ids) > 1:
            np.cumsum(cards[:-1], out=offs[1:])
        out = np.zeros(int(cards.sum()), np.float64)
        _lib.check(_lib.lib().nb_potentials(g, int(bool(evid_chain)), _lib.ptr(var_ids), len(var_ids),
                                            _lib.ptr(offs), _lib.ptr(out), len(out)))
        return out

    def potentials_records(self, var_ids=None, evid_chain=False, var_copy=0, weight_copy=0):
        """The energies the RECORD kernels sample from (nb_potentials_records): returns
        ``(out, row_class)`` with ``out`` laid out like :meth:`potentials`.  PAIR / FAST rows (class
        0 / 1) hold ``{0, potential(v,1) - potential(v,0)}``, CAT rows (class 2) their fp32 per-value
        energies; entries of generic rows (class 3 / 4) stay NaN."""
        g = self._device_graph()
        self._sync_device(var_copy, weight_copy)
        if var_ids is None:
            var_ids = np.arange(self.variable.shape[0], dtype=np.int64)
        var_ids = _lib.contiguous(var_ids, np.int64)
        cards = self.variable["cardinality"][var_ids].astype(np.int64)
        offs = np.zeros(len(var_ids), np.int64)
        if len(var_ids) > 1:
            np.cumsum(cards[:-1], out=offs[1:])
        out = np.zeros(int(cards.sum()), np.float64)
        cls = np.zeros(len(var_ids), np.int32)
        _lib.check(_lib.lib().nb_potentials_records(g, int(bool(evid_chain)), _lib.ptr(var_ids), len(var_ids),
                                                    _lib.ptr(offs), _lib.ptr(out), len(out), _lib.ptr(cls)))
        generic = np.repeat(cls >= 3, cards)
        out[generic] = np.nan
        return out, cls

    # ------------------------------------------------------------------
    # host mirrors
    # ------------------------------------------------------------------
    def _host(self, name, expose=True):
        """The host mirror `name`, refreshed from the device if it is stale.  `expose` records that
        the caller now holds a reference (and may edit the array behind our back)."""
        if name in self._stale:
            self._fetch(name)
        if expose:
            self._exposed.add(name)
        return getattr(self, "_" + name)

    def _assign(self, name, value):
        setattr(self, "_" + name, value)
        self._exposed.add(name)
        self._stale.discard(name)
        if name in self._dev_row:
            self._dev_row[name] = None
        if name == "count":
            self._count_dev_valid = False

    var_value = property(lambda self: self._host("var_value"), lambda self, v: self._assign("var_value", v))
    var_value_evid = property(lambda self: self._host("var_value_evid"),
                              lambda self, v: self._assign("var_value_evid", v))
    weight_value = property(lambda self: self._host("weight_value"), lambda self, v: self._assign("weight_value", v))
    count = property(lambda self: self._host("count"), lambda self, v: self._assign("count", v))
    marginals = property(lambda self: self._host("marginals"), lambda self, v: self._assign("marginals", v))

    def _row(self, arr, copy, dtype):
        """Row `arr[copy]` as a C-contiguous array the library can read AND write in place (true
        for arrays built by __init__; anything else goes through a copy)."""
        row = arr[copy]
        if row.dtype == dtype and row.flags.c_contiguous and row.flags.writeable:
            return row, None
        tmp = np.ascontiguousarray(row, dtype=dtype)
        return tmp, row

    def _fetch(self, name):
        """Refresh the host mirror `name` from the device."""
        L, g = _lib.lib(), self._g
        self._stale.discard(name)
        if g is None:
            return
        if name in ("var_value", "var_value_evid"):
            buf, dst = self._row(getattr(self, "_" + name), self._dev_row[name], np.int64)
            _lib.check(L.nb_get_var_values(g, 0 if name == "var_value" else 1, _lib.ptr(buf)))
            if dst is not None:
                dst[:] = buf
        elif name == "weight_value":
            buf, dst = self._row(self._weight_value, self._dev_row[name], np.float64)
            _lib.check(L.nb_get_weights(g, _lib.ptr(buf)))
            if dst is not None:
                dst[:] = buf
            self._w_shadow = np.array(buf, copy=True)
        elif name == "count":
            c = self._count
            if not (isinstance(c, np.ndarray) and c.dtype == np.int64 and c.flags.c_contiguous and c.flags.writeable):
                self._count = c = np.zeros(self.cstart[-1], np.int64)
            _lib.check(L.nb_get_counts(g, _lib.ptr(c), 0))        # the device tallies are cumulative
        elif name == "marginals":
            m = self._marginals
            if not (isinstance(m, np.ndarray) and m.dtype == np.float64 and m.shape == (int(self.cstart[-1]),)
                    and m.flags.c_contiguous and m.flags.writeable):
                m = np.empty(int(self.cstart[-1]), np.float64)
            # (the reference binds a fresh array on every inference, factorgraph.py:173; this one is
            # refilled in place -- first-touch page faults of a new 134 MB array cost more than the sweep)
            _lib.check(L.nb_get_marginals(g, _lib.ptr(m), float(self._marg_epochs)))
            self._marginals = m

    def _sync_device(self, var_copy, weight_copy, evid=True, counts=False, force=False):
        """Make the device copy current before a sweep: upload what the caller may have edited."""
        L, g = _lib.lib(), self._device_graph()
        names = [("var_value", 0)] + ([("var_value_evid", 1)] if evid else [])
        for name, chain in names:
            if not force and self._dev_row[name] == var_copy and name not in self._exposed:
                continue
            if name in self._stale:          # HBM holds a newer version of another row: write it back first
                self._fetch(name)
            row = self._row(getattr(self, "_" + name), var_copy, np.int64)[0]
            _lib.check(L.nb_set_var_values(g, chain, _lib.ptr(row)))
            self._dev_row[name] = var_copy
        if "weight_value" in self._stale and self._dev_row["weight_value"] != weight_copy:
            self._fetch("weight_value")
        if "weight_value" not in self._stale:
            w = self._row(self._weight_value, weight_copy, np.float64)[0]
            if (force or self._dev_row["weight_value"] != weight_copy or self._w_shadow is None
                    or not np.array_equal(w, self._w_shadow)):
                _lib.check(L.nb_set_weights(g, _lib.ptr(w)))
                self._w_shadow = np.array(w, copy=True)
                self._dev_row["weight_value"] = weight_copy
        if counts and (not self._count_dev_valid or "count" in self._exposed):
            c = _lib.contiguous(self._count, np.int64)
            if len(c) != int(self.cstart[-1]):
                raise ValueError("count must have cstart[-1] entries")
            _lib.check(L.nb_set_counts(g, _lib.ptr(c)))
            self._count_dev_valid = True

    def _mark_device_newer(self, *names):
        """After a sweep: the listed arrays changed in HBM.  Mirrors the caller holds a reference to
        are refreshed right away (they must look like the reference's in-place arrays)."""
        for name in names:
            self._stale.add(name)
            if name in self._exposed and name != "marginals":
                self._fetch(name)

    def _upload(self, var_copy, weight_copy, evid=True):
        """Force the rows into HBM (tools and the partitioned runner)."""
        self._sync_device(var_copy, weight_copy, evid=evid, force=True)

    def _download(self, var_copy, weight_copy, evid=False, weights=False, counts=False, epochs=0):
        """Refresh the listed host mirrors now."""
        self._stale.add("var_value")
        self._fetch("var_value")
        if evid:
            self._stale.add("var_value_evid")
            self._fetch("var_value_evid")
        if weights:
            self._stale.add("weight_value")
            self._fetch("weight_value")
        if counts:
            self._fetch("count")
            if epochs:
                self._marg_epochs = epochs
                self._fetch("marginals")

    def counts_compact(self):
        """The cumulative tallies (``count``) at their natural width -- uint8 while no tally can
        exceed 255 sweeps, then uint16 / int32 -- DMA-ed into page-locked host memory the library
        owns: no host-side conversion, so the read scales with the number of GPUs.  The returned
        array is a view that the next call overwrites; ``count`` / ``marginals`` stay available."""
        L, g = _lib.lib(), self._device_graph()
        n = int(self.cstart[-1])
        if getattr(self, "_pinned", None) is None:
            p = C.c_void_p()
            _lib.check(L.nb_host_alloc(C.byref(p), 4 * max(n, 1)))
            self._pinned = p
        elem = C.c_int32(0)
        _lib.check(L.nb_get_counts_compact(g, self._pinned, 4 * max(n, 1), C.byref(elem)))
        dtype = {1: np.uint8, 2: np.uint16, 4: np.int32}[elem.value]
        buf = (C.c_char * (n * elem.value)).from_address(self._pinned.value)
        return np.frombuffer(buf, dtype=dtype, count=n)

    def invalidate(self):
        """Drop the device graph after the record arrays (variable / weight / factor / fmap /
        vmap / factor_index) were edited; it is rebuilt from them on the next call.  The chains,
        weights and counts carry over."""
        for name in ("var_value", "var_value_evid", "weight_value", "count", "marginals"):
            self._host(name, expose=False)
        if self._g is not None:
            _lib.lib().nb_graph_destroy(self._g)
            self._g = None
        self._dev_row = {k: None for k in self._dev_row}
        self._count_dev_valid = False
        self._pristine = False

    def clear(self):
        """factorgraph.py:75-78 (the thread pool's role is played by the device graph)."""
        for name in ("var_value", "var_value_evid", "weight_value", "marginals"):
            self._host(name, expose=False)
        self._stale.discard("count")
        self._count[:] = 0
        if self._g is not None:
            _lib.lib().nb_graph_destroy(self._g)
            self._g = None
        self._dev_row = {k: None for k in self._dev_row}
        self._count_dev_valid = True       # a rebuilt graph starts with zero tallies, like count
        self._pristine = False

    # ------------------------------------------------------------------
    # in-place record edits
    # ------------------------------------------------------------------
    @staticmethod
    def _last_wins(ids, n_records, what, *columns):
        """Ids in range, one entry per id (the last occurrence, as numpy's a[ids] = x) in increasing
        id order, and the matching entries of each column (None stays None)."""
        ids = np.asarray(ids, np.int64).reshape(-1)
        cols = [None if c is None else np.broadcast_to(np.asarray(c), ids.shape) for c in columns]
        bad = (ids < 0) | (ids >= n_records)
        if bad.any():
            raise ValueError("%s id %d out of range [0, %d)" % (what, int(ids[np.argmax(bad)]), n_records))
        uniq, first_of_reversed = np.unique(ids[::-1], return_index=True)
        pick = len(ids) - 1 - first_of_reversed
        return uniq, [None if c is None else c[pick] for c in cols]

    def update_variables(self, var_ids, isEvidence=None, initialValue=None, value=None, var_copy=0):
        """Edit ``isEvidence`` / ``initialValue`` of the listed variables in place, without a
        rebuild; ``value`` also sets both chains (``var_value[var_copy]`` and
        ``var_value_evid[var_copy]``) of those variables.  A duplicated id takes its last entry.
        ``self.variable`` is edited too, so a later :meth:`invalidate` rebuilds the same graph.
        Everything is validated before anything is written (ValueError)."""
        V = self.variable.shape[0]
        ids, (ev, ini, val) = self._last_wins(var_ids, V, "variable", isEvidence, initialValue, value)
        if len(ids) == 0 or (ev is None and ini is None and val is None):
            return
        ev = None if ev is None else ev.astype(np.int8)
        ini = None if ini is None else ini.astype(np.int64)
        val = None if val is None else val.astype(np.int64)
        # the checks of the build (and of nb_update_variables), against the records
        rec = self.variable[ids]
        card = rec["cardinality"].astype(np.int64)
        if ev is not None and (ev == 4).any():
            raise ValueError("isEvidence 4 marks a ghost, which only the partitioner creates (variable %d)"
                             % int(ids[np.argmax(ev == 4)]))
        ghost = rec["isEvidence"] == 4
        if ghost.any():
            raise ValueError("variable %d is a ghost (isEvidence 4): the partitioner owns it" % int(ids[np.argmax(ghost)]))
        e = rec["isEvidence"].astype(np.int64) if ev is None else ev.astype(np.int64)
        x = rec["initialValue"].astype(np.int64) if ini is None else ini
        bad = (e == 1) & ((x < 0) | (x >= card))
        if bad.any():
            raise ValueError("invalid factor graph: evidence variable with initialValue outside [0, cardinality) "
                             "(index %d)" % int(ids[np.argmax(bad)]))
        if val is not None:
            bad = (val < 0) | (val >= card)
            if bad.any():
                raise ValueError("value of variable %d lies outside [0, cardinality)" % int(ids[np.argmax(bad)]))

        names = ("var_value", "var_value_evid")
        if self._g is not None:
            L = _lib.lib()
            # the device chains take the value only if they hold row var_copy (else the host row is edited
            # and uploaded by the next call)
            dev_val = val is not None and all(self._dev_row[n] == var_copy for n in names)
            _lib.check(L.nb_update_variables(self._g, _lib.ptr(ids), len(ids), _lib.ptr(ev), _lib.ptr(ini),
                                             _lib.ptr(val) if dev_val else None))
            if val is not None:
                for n in names:
                    if dev_val:
                        # exposed mirrors are uploaded on entry to the next call: they must agree; a stale
                        # mirror is refreshed from the device when it is read
                        if n not in self._stale:
                            getattr(self, "_" + n)[var_copy][ids] = val
                    else:
                        if n in self._stale and self._dev_row[n] == var_copy:
                            self._fetch(n)
                        getattr(self, "_" + n)[var_copy][ids] = val
                        if self._dev_row[n] == var_copy:
                            self._dev_row[n] = None
        elif val is not None or ini is not None:
            # no device graph yet: the chains it will start from are the host rows, not initialValue
            for n in names:
                if val is not None:
                    getattr(self, "_" + n)[var_copy][ids] = val
            self._pristine = False
        if ev is not None:
            self.variable["isEvidence"][ids] = ev
        if ini is not None:
            self.variable["initialValue"][ids] = ini

    def update_weights(self, weight_ids, isFixed):
        """Edit ``weight.isFixed`` of the listed weights in place, without a rebuild (a duplicated id
        takes its last entry); ``self.weight`` is edited too."""
        ids, (fx,) = self._last_wins(weight_ids, self.weight.shape[0], "weight", isFixed)
        if len(ids) == 0:
            return
        fx = (np.asarray(fx) != 0).astype(np.uint8)
        if self._g is not None:
            _lib.check(_lib.lib().nb_update_weights_fixed(self._g, _lib.ptr(ids), len(ids), _lib.ptr(fx)))
        self.weight["isFixed"][ids] = fx

    def device_digest(self):
        """{array name: 64-bit digest} of the device arrays a build derives from the records
        (nb_graph_digest): equal digests = the same device graph."""
        out = np.zeros(len(_lib.DIGEST_ARRAYS), np.uint64)
        _lib.check(_lib.lib().nb_graph_digest(self._device_graph(), _lib.ptr(out), len(out)))
        return {n: int(d) for n, d in zip(_lib.DIGEST_ARRAYS, out)}

    def __del__(self):
        try:
            if getattr(self, "_pinned", None) is not None:
                _lib.lib().nb_host_free(self._pinned)
                self._pinned = None
            if getattr(self, "_g", None) is not None:
                _lib.lib().nb_graph_destroy(self._g)
                self._g = None
        except Exception:
            pass

    #################
    #    GETTERS    #
    #################

    def getWeights(self, weight_copy=0):
        return self.weight_value[weight_copy][:]

    def getMarginals(self, varIds=None):
        if not varIds:
            return self.marginals
        else:
            return self.marginals[varIds]

    #####################
    #    DIAGNOSTICS    #
    #####################

    def diagnostics(self, epochs):
        """Marginal histogram, same text as factorgraph.py:99-113."""
        print('Inference took %.03f sec.' % self.inference_total_time)
        epochs = epochs or 1
        bins = 10
        count = self._host("count", expose=False)
        assert (count >= 0).all() and (count <= epochs).all()
        hist = np.bincount(np.minimum(count * bins // epochs, bins - 1), minlength=bins)
        for i in range(bins):
            start = i / 10.0
            end = (i + 1) / 10.0
            print("Prob. " + str(start) + ".." + str(end) + ": \
                  " + str(hist[i]) + " variables")

    def diagnosticsLearning(self, weight_copy=0):
        print('Learning epoch took %.03f sec.' % self.learning_epoch_time)
        print("Weights:")
        for (i, w) in enumerate(self.weight):
            print("    weightId:", i)
            print("        isFixed:", w["isFixed"])
            print("        weight: ", self._host("weight_value", expose=False)[weight_copy][i])
            print()

    ################################
    #    INFERENCE AND LEARNING    #
    ################################

    def _sweeps(self, epochs, burnin, sample_evidence):
        _lib.check(_lib.lib().nb_gibbs_sweeps(self._g, int(epochs), int(bool(burnin)),
                                              int(bool(sample_evidence)), self.seed))

    def burnIn(self, epochs, sample_evidence, diagnostics=False,
               var_copy=0, weight_copy=0, _resident=False):
        """factorgraph.py:129-143."""
        if diagnostics:
            print("FACTOR " + str(self.fid) + ": STARTED BURN-IN...")
        if not _resident:
            self._sync_device(var_copy, weight_copy, evid=False)
        self._sweeps(epochs, True, sample_evidence)
        if not _resident and epochs > 0:
            self._mark_device_newer("var_value")
        if diagnostics:
            print("FACTOR " + str(self.fid) + ": DONE WITH BURN-IN")

    def inference(self, burnin_epochs, epochs, sample_evidence=False,
                  diagnostics=False, var_copy=0, weight_copy=0):
        """factorgraph.py:145-175."""
        self._sync_device(var_copy, weight_copy, evid=False, counts=True)   # the Gibbs sweep only touches chain 0
        if burnin_epochs > 0:
            self.burnIn(burnin_epochs, sample_evidence, diagnostics=diagnostics,
                        var_copy=var_copy, weight_copy=weight_copy, _resident=True)
        if diagnostics:
            print("FACTOR " + str(self.fid) + ": STARTED INFERENCE")
        if diagnostics:
            for ep in range(epochs):
                with Timer() as timer:
                    self._sweeps(1, False, sample_evidence)
                self.inference_epoch_time = timer.interval
                self.inference_total_time += timer.interval
                print('Inference epoch #%d took %.03f sec.' % (ep, self.inference_epoch_time))
        elif epochs > 0:
            with Timer() as timer:
                self._sweeps(epochs, False, sample_evidence)
            self.inference_epoch_time = timer.interval / epochs
            self.inference_total_time += timer.interval
        # count += tallies (the device tallies are cumulative) and, if epochs != 0,
        # marginals = count / epochs (factorgraph.py:172-173) -- materialised when somebody reads them
        changed = ["var_value"] if burnin_epochs > 0 or epochs > 0 else []
        if epochs > 0:
            changed.append("count")
            self._marg_epochs = epochs
            changed.append("marginals")
        self._mark_device_newer(*changed)
        if diagnostics:
            print("FACTOR " + str(self.fid) + ": DONE WITH INFERENCE")
        if diagnostics:
            self.diagnostics(epochs)

    def learn(self, burnin_epochs, epochs, stepsize, decay, regularization,
              reg_param, truncation, diagnostics=False, verbose=False,
              learn_non_evidence=False, var_copy=0, weight_copy=0):
        """factorgraph.py:177-208."""
        L = _lib.lib()
        self._sync_device(var_copy, weight_copy)
        if burnin_epochs > 0:
            self.burnIn(burnin_epochs, True, diagnostics=diagnostics,
                        var_copy=var_copy, weight_copy=weight_copy, _resident=True)
        if diagnostics:
            print("FACTOR " + str(self.fid) + ": STARTED LEARNING")

        def run(n, step):
            s = C.c_double(step)
            _lib.check(L.nb_learn_sweeps(self._g, int(n), C.byref(s), float(decay), int(regularization),
                                         float(reg_param), float(truncation),
                                         int(bool(learn_non_evidence)), self.seed, int(self.batch_visits)))
            return s.value

        if diagnostics:
            for ep in range(epochs):
                print("FACTOR " + str(self.fid) + ": EPOCH #" + str(ep))
                print("Current stepsize = " + str(stepsize))
                if verbose:
                    self._stale.add("weight_value")
                    self._fetch("weight_value")
                    self.diagnosticsLearning(weight_copy)
                sys.stdout.flush()
                with Timer() as timer:
                    stepsize = run(1, stepsize)
                self.learning_epoch_time = timer.interval
                self.learning_total_time += timer.interval
        elif epochs > 0:
            with Timer() as timer:
                stepsize = run(epochs, stepsize)
            self.learning_epoch_time = timer.interval / epochs
            self.learning_total_time += timer.interval
        if burnin_epochs > 0 or epochs > 0:
            self._mark_device_newer("var_value", "var_value_evid")
        if epochs > 0:
            self._stale.add("weight_value")
            self._fetch("weight_value")          # small; keeps the comparison copy current
        if diagnostics:
            print("FACTOR " + str(self.fid) + ": DONE WITH LEARNING")

    def dump_weights(self, fout, weight_copy=0):
        """Dump <wid, weight> text file in DW format (factorgraph.py:210-214)."""
        w = self._host("weight_value", expose=False)[weight_copy]
        with open(fout, 'w') as out:
            out.write(''.join('%d %f\n' % (i, x) for i, x in enumerate(w.tolist())))

    def dump_probabilities(self, fout, epochs):
        """Dump <vid, value, prob> text file in DW format (factorgraph.py:216-229)."""
        epochs = epochs or 1
        card = self.variable["cardinality"].astype(np.int64)
        nvar = len(card)
        binary = card == 2
        per_var = np.where(binary, 1, card)
        vid = np.repeat(np.arange(nvar, dtype=np.int64), per_var)
        k = np.arange(len(vid), dtype=np.int64) - np.repeat(self.cstart[:-1], per_var)
        value = np.ones(len(vid), np.int64)
        nb = ~np.repeat(binary, per_var)
        if nb.any():
            vtf = np.repeat(self.variable["vtf_offset"].astype(np.int64), per_var)
            value[nb] = self.vmap["value"][vtf[nb] + k[nb]]
        prob = self._host("count", expose=False).astype(np.float64) / epochs
        with open(fout, 'w') as out:
            step = 1 << 20
            for s in range(0, len(vid), step):
                out.write(''.join('%d %d %.3f\n' % t for t in zip(vid[s:s + step].tolist(),
                                                                  value[s:s + step].tolist(),
                                                                  prob[s:s + step].tolist())))
