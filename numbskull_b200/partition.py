"""Variable-partitioned multi-GPU execution (one process per GPU).

Follows the reference's master/minion scheme (salt/src/numbskull_master.py:343,
numbskull_minion.py:185, messages.py:1308-1319): every rank OWNS a block of
variables, holds every factor that touches one of them, and keeps the remote
members of those factors as ghost variables with ``isEvidence == 4`` -- the
flag both reference kernels skip (inference.py:21-23, learning.py:24-26).
Where the reference ships values once per epoch, here the owner's fresh
values go to the ghost copies after EVERY colour, so the partitioned sampler
is the same chromatic Gibbs chain as the single-GPU one: colours come from a
distributed Jones-Plassmann run whose priorities depend only on the global
variable id, and the Philox streams are keyed by the global id too, so an
N-GPU run reproduces the 1-GPU samples bit for bit.

Learning adds the reference's per-epoch weight-delta sum
(numbskull_master.py:223-224): w <- w_prev + sum_r (w_r - w_prev), one
all-reduce per epoch.

``torch.distributed`` is plumbing only (rendezvous, point-to-point transport:
NCCL over NVLink on GPUs, gloo in the CPU tests of the host logic).
"""
from __future__ import print_function

import ctypes as C

import numpy as np

from .numbskulltypes import Factor, FactorToVar, Variable


# --------------------------------------------------------------------------- partitioning
def block_bounds(n, world):
    """Contiguous owner blocks: rank r owns global ids [b[r], b[r+1])."""
    return np.array([(r * n) // world for r in range(world + 1)], np.int64)


def extract_local(weight, variable, factor, fmap, lo, hi):
    """Owner-computes sub-graph of the block [lo, hi) of a global graph.

    Keeps (in global order) every factor with at least one owned member;
    local variables are the owned block followed by the ghosts in increasing
    global id; ghosts get ``isEvidence = 4``.  Returns a dict with the local
    record arrays, ``global_vid`` and ``n_owned``."""
    arity = factor["arity"].astype(np.int64)
    fid_of_entry = np.repeat(np.arange(len(factor), dtype=np.int64), arity)
    # entries of a factor are contiguous at ftv_offset; build the entry index explicitly
    entry = np.repeat(factor["ftv_offset"].astype(np.int64), arity) + \
        (np.arange(len(fid_of_entry), dtype=np.int64) - np.repeat(np.cumsum(arity) - arity, arity))
    vids = fmap["vid"][entry].astype(np.int64)
    owned_entry = (vids >= lo) & (vids < hi)
    keep_factor = np.zeros(len(factor), bool)
    keep_factor[fid_of_entry[owned_entry]] = True
    keep_entry = keep_factor[fid_of_entry]

    loc_factor = factor[keep_factor].copy()
    loc_arity = loc_factor["arity"].astype(np.int64)
    off = np.zeros(len(loc_factor), np.int64)
    if len(loc_factor) > 1:
        np.cumsum(loc_arity[:-1], out=off[1:])
    loc_factor["ftv_offset"] = off
    loc_entries = entry[keep_entry]
    loc_vids = vids[keep_entry]

    ghosts = np.unique(loc_vids[(loc_vids < lo) | (loc_vids >= hi)])
    n_owned = hi - lo
    global_vid = np.concatenate((np.arange(lo, hi, dtype=np.int64), ghosts))
    loc_variable = variable[global_vid].copy()
    loc_variable["isEvidence"][n_owned:] = 4
    loc_variable["vtf_offset"] = 0

    loc_fmap = np.zeros(len(loc_entries), FactorToVar)
    is_owned = (loc_vids >= lo) & (loc_vids < hi)
    lid = np.where(is_owned, loc_vids - lo, n_owned + np.searchsorted(ghosts, loc_vids))
    loc_fmap["vid"] = lid
    loc_fmap["dense_equal_to"] = fmap["dense_equal_to"][loc_entries]
    return dict(weight=weight.copy(), variable=loc_variable, factor=loc_factor, fmap=loc_fmap,
                domain_mask=np.zeros(len(loc_variable), np.bool_), global_vid=global_vid,
                n_owned=int(n_owned))


def extract_local_by_owner(weight, variable, factor, fmap, owner, rank):
    """:func:`extract_local` for an arbitrary placement: ``owner[v]`` is the rank that owns global
    variable ``v`` (an imported partition, e.g. :func:`owners_from_salt_keys`, or a locality-aware
    one, :func:`locality_owners`).  Owned variables keep their relative order; ghosts follow in
    increasing global id with ``isEvidence = 4``.  Host threads in the library (nb_extract_local);
    :func:`_extract_local_by_owner_numpy` is the same rule in numpy (the tests compare them)."""
    import ctypes as C
    from . import _lib
    from .numbskulltypes import Factor
    L = _lib.lib()
    owner32 = np.ascontiguousarray(owner, np.int32)
    assert len(owner32) == len(variable)
    factor_c, fmap_c = np.ascontiguousarray(factor), np.ascontiguousarray(fmap)
    nf, ne, no, ng = C.c_int64(0), C.c_int64(0), C.c_int64(0), C.c_int64(0)
    args = (_lib.ptr(factor_c), len(factor_c), _lib.ptr(fmap_c), len(fmap_c), _lib.ptr(owner32), len(owner32), int(rank),
            C.byref(nf), C.byref(ne), C.byref(no), C.byref(ng))
    _lib.check(L.nb_extract_local(*args, None, None, None))
    loc_factor = np.zeros(nf.value, Factor)
    loc_fmap = np.zeros(ne.value, FactorToVar)
    global_vid = np.empty(no.value + ng.value, np.int64)
    _lib.check(L.nb_extract_local(*args, _lib.ptr(loc_factor), _lib.ptr(loc_fmap), _lib.ptr(global_vid)))
    n_owned = no.value
    loc_variable = variable[global_vid].copy()
    loc_variable["isEvidence"][n_owned:] = 4
    loc_variable["vtf_offset"] = 0
    return dict(weight=weight.copy(), variable=loc_variable, factor=loc_factor, fmap=loc_fmap,
                domain_mask=np.zeros(len(loc_variable), np.bool_), global_vid=global_vid,
                n_owned=int(n_owned), owner=np.asarray(owner))


def _extract_local_by_owner_numpy(weight, variable, factor, fmap, owner, rank):
    """The rule of :func:`extract_local_by_owner`, vectorised numpy (reference for the tests)."""
    owner = np.asarray(owner)
    assert len(owner) == len(variable)
    arity = factor["arity"].astype(np.int64)
    fid_of_entry = np.repeat(np.arange(len(factor), dtype=np.int64), arity)
    entry = np.repeat(factor["ftv_offset"].astype(np.int64), arity) + \
        (np.arange(len(fid_of_entry), dtype=np.int64) - np.repeat(np.cumsum(arity) - arity, arity))
    vids = fmap["vid"][entry].astype(np.int64)
    owned_entry = owner[vids] == rank
    keep_factor = np.zeros(len(factor), bool)
    keep_factor[fid_of_entry[owned_entry]] = True
    keep_entry = keep_factor[fid_of_entry]

    loc_factor = factor[keep_factor].copy()
    loc_arity = loc_factor["arity"].astype(np.int64)
    off = np.zeros(len(loc_factor), np.int64)
    if len(loc_factor) > 1:
        np.cumsum(loc_arity[:-1], out=off[1:])
    loc_factor["ftv_offset"] = off
    loc_entries = entry[keep_entry]
    loc_vids = vids[keep_entry]

    owned = np.nonzero(owner == rank)[0].astype(np.int64)
    ghosts = np.unique(loc_vids[owner[loc_vids] != rank])
    n_owned = len(owned)
    global_vid = np.concatenate((owned, ghosts))
    loc_variable = variable[global_vid].copy()
    loc_variable["isEvidence"][n_owned:] = 4
    loc_variable["vtf_offset"] = 0

    loc_fmap = np.zeros(len(loc_entries), FactorToVar)
    mine = owner[loc_vids] == rank
    loc_fmap["vid"] = np.where(mine, np.searchsorted(owned, loc_vids), n_owned + np.searchsorted(ghosts, loc_vids))
    loc_fmap["dense_equal_to"] = fmap["dense_equal_to"][loc_entries]
    return dict(weight=weight.copy(), variable=loc_variable, factor=loc_factor, fmap=loc_fmap,
                domain_mask=np.zeros(len(loc_variable), np.bool_), global_vid=global_vid,
                n_owned=int(n_owned), owner=owner)


def owners_from_salt_keys(keys, world):
    """Placement from the reference's semantic-partition keys (salt/src/messages.py:175-179,229-236:
    the first character of ``partition_key`` is the partition type, the master's SQL filter
    ``numbskull_master.py:329-332`` keeps 'A', 'B', 'D', 'F' rows; minion ``i`` gets the rows whose
    key carries its id).  'A' / 'B' variables belong to the master = rank 0; 'C<i>' / 'D<i>' (and any
    other keyed type) to minion ``i`` = rank ``1 + i mod (world - 1)``; the variable still appears as
    a ghost wherever one of its factors lives, which is what the visible-to-both types 'B' / 'D'
    ask for.  ``keys``: sequence of str / bytes, e.g. ``["A", "B", "C0", "D1"]``."""
    out = np.zeros(len(keys), np.int32)
    for i, k in enumerate(keys):
        k = k.decode() if isinstance(k, bytes) else str(k)
        t, rest = k[:1].upper(), k[1:].lstrip("uU")
        if t in ("A", "B") or world == 1:
            out[i] = 0
        else:
            idx = int(rest) if rest.isdigit() else 0
            out[i] = 1 + idx % (world - 1)
    return out


def locality_owners(variable, factor, fmap, world):
    """Locality-aware placement for graphs whose variable ids carry no locality: a reverse
    Cuthill-McKee ordering of the variable graph (variables adjacent iff they share a factor; every
    factor contributes a path over its members) cut into ``world`` contiguous pieces of equal
    size.  The role METIS plays in the reference (salt/src/messages.py:591-640 find_metis_parts);
    host-side scipy, meant for graphs up to a few 10^7 edges."""
    import scipy.sparse as sp
    from scipy.sparse.csgraph import reverse_cuthill_mckee
    n = len(variable)
    arity = factor["arity"].astype(np.int64)
    off = factor["ftv_offset"].astype(np.int64)
    fid = np.repeat(np.arange(len(factor), dtype=np.int64), arity)
    entry = np.repeat(off, arity) + (np.arange(len(fid), dtype=np.int64) - np.repeat(np.cumsum(arity) - arity, arity))
    vids = fmap["vid"][entry].astype(np.int64)
    same = fid[1:] == fid[:-1]
    a, b = vids[:-1][same], vids[1:][same]
    g = sp.coo_matrix((np.ones(len(a), np.int8), (a, b)), shape=(n, n)).tocsr()
    g = g + g.T
    order = np.asarray(reverse_cuthill_mckee(g.tocsr(), symmetric_mode=True), np.int64)
    owner = np.empty(n, np.int32)
    owner[order] = (np.arange(n, dtype=np.int64) * world // max(n, 1)).astype(np.int32)
    return owner


def ghost_fraction(local):
    """Ghost copies per owned variable of one rank's share (what the halo exchange moves)."""
    return (len(local["variable"]) - local["n_owned"]) / max(1, local["n_owned"])


def ising_strip(rows, cols, rank, world, coupling=0.1):
    """Rank ``rank``'s share of a (rows*world) x cols Ising grid (BASELINE config 2
    shape, weak scaling): it owns ``rows`` grid rows and sees the row above and
    below as ghosts.  Built locally -- the global graph is never materialised."""
    from . import synth
    top = 1 if rank > 0 else 0
    bot = 1 if rank < world - 1 else 0
    w, v, f, fm, dm, e = synth.ising_grid(rows + top + bot, cols, coupling)
    first_global_row = rank * rows - top
    gv = first_global_row * cols + np.arange(len(v), dtype=np.int64)
    lo, hi = top * cols, (top + rows) * cols          # owned block in sub-grid ids
    local = extract_local(w, v, f, fm, lo, hi)
    # extract_local numbers owned first, then ghosts; translate its ids to the true global ids
    local["global_vid"] = gv[local["global_vid"]]
    return local, (rows * world) * cols


# --------------------------------------------------------------------------- plumbing
def exchange_arrays(send, rank, world, device, group=None):
    """All-to-all of variable-length int64 arrays: ``send[p]`` goes to rank p; returns the list of
    arrays received from every rank.  Counts travel in one all_gather, payloads point-to-point
    (tensors, not pickled Python lists: at the 1 B-edge scale a rank has 10^7 ghosts)."""
    import torch
    import torch.distributed as dist
    if world == 1:
        return [np.asarray(send[0], np.int64)]
    stage = dist.get_backend(group) == "gloo"
    dev = torch.device("cpu") if stage else device
    counts = torch.tensor([len(x) for x in send], dtype=torch.int64, device=dev)
    allc = [torch.zeros(world, dtype=torch.int64, device=dev) for _ in range(world)]
    dist.all_gather(allc, counts, group=group)
    recv_counts = [int(allc[p][rank].item()) for p in range(world)]
    sbufs = [torch.from_numpy(np.ascontiguousarray(x, dtype=np.int64)).to(dev) for x in send]
    rbufs = [torch.empty(n, dtype=torch.int64, device=dev) for n in recv_counts]
    ops = []
    for p in range(world):
        if p == rank:
            continue
        if len(send[p]):
            ops.append(dist.P2POp(dist.isend, sbufs[p], p, group=group))
        if recv_counts[p]:
            ops.append(dist.P2POp(dist.irecv, rbufs[p], p, group=group))
    if ops:
        for req in dist.batch_isend_irecv(ops):
            req.wait()
    if not stage:
        torch.cuda.synchronize()
    out = [b.cpu().numpy() for b in rbufs]
    out[rank] = np.asarray(send[rank], np.int64)
    return out


# --------------------------------------------------------------------------- halo plan
class HaloPlan(object):
    """Who needs whose values.  ``send_ids[p]`` are local ids of owned variables
    that rank p holds as ghosts, ``recv_ids[p]`` the local ids of this rank's
    ghosts owned by p, in matching order."""

    def __init__(self, global_vid, n_owned, owner_of, rank, world, group=None, device="cpu"):
        self.rank, self.world = rank, world
        ghosts = np.asarray(global_vid[n_owned:], np.int64)
        owned = np.asarray(global_vid[:n_owned], np.int64)          # ascending global ids
        owner = np.asarray(owner_of(ghosts), np.int64)
        requests = [ghosts[owner == p] for p in range(world)]
        self.recv_ids = [np.nonzero(owner == p)[0].astype(np.int64) + n_owned for p in range(world)]
        asked_by = exchange_arrays(requests, rank, world, device, group)    # what every rank wants from me
        self.send_ids = []
        for p in range(world):
            asked = np.asarray(asked_by[p], np.int64)
            loc = np.searchsorted(owned, asked)
            assert len(asked) == 0 or (loc < n_owned).all() and np.array_equal(owned[loc], asked)
            self.send_ids.append(loc.astype(np.int64))
        assert len(self.send_ids[rank]) == 0 and len(self.recv_ids[rank]) == 0

    def restrict(self, keep_local):
        """Per-peer (send, recv) id lists of the variables flagged in ``keep_local``."""
        send = [ids[keep_local[ids]] for ids in self.send_ids]
        recv = [ids[keep_local[ids]] for ids in self.recv_ids]
        return send, recv


class Exchange(object):
    """One fixed communication pattern: gather -> point-to-point -> scatter."""

    def __init__(self, send, recv, rank, world, dtype, device, group=None):
        import torch
        self.torch = torch
        self.rank, self.world, self.group = rank, world, group
        self.send_counts = [len(x) for x in send]
        self.recv_counts = [len(x) for x in recv]
        self.n_send, self.n_recv = sum(self.send_counts), sum(self.recv_counts)
        cat = lambda xs: np.concatenate(xs) if xs else np.zeros(0, np.int64)  # noqa: E731
        self.send_ids = torch.from_numpy(cat(send).astype(np.int32)).to(device)
        self.recv_ids = torch.from_numpy(cat(recv).astype(np.int32)).to(device)
        self.send_buf = torch.zeros(max(self.n_send, 1), dtype=dtype, device=device)
        self.recv_buf = torch.zeros(max(self.n_recv, 1), dtype=dtype, device=device)
        # gloo moves host memory only: device buffers are staged through the CPU (1-GPU tests);
        # NCCL sends the device buffers directly over NVLink
        import torch.distributed as dist
        self.stage = (world > 1 and self.send_buf.is_cuda and dist.get_backend(group) == "gloo")

    def run(self, gather, scatter):
        """gather(ids, out) fills out[i] = x[ids[i]]; scatter(ids, buf) sets x[ids[i]] = buf[i]."""
        import torch.distributed as dist
        if self.n_send:
            gather(self.send_ids, self.send_buf[:self.n_send])
        sbuf = self.send_buf.cpu() if self.stage else self.send_buf
        rbuf = self.recv_buf.cpu() if self.stage else self.recv_buf
        ops, so, ro = [], 0, 0
        for p in range(self.world):
            ns, nr = self.send_counts[p], self.recv_counts[p]
            if ns:
                ops.append(dist.P2POp(dist.isend, sbuf[so:so + ns], p, group=self.group))
            if nr:
                ops.append(dist.P2POp(dist.irecv, rbuf[ro:ro + nr], p, group=self.group))
            so += ns
            ro += nr
        if ops:
            for req in dist.batch_isend_irecv(ops):
                req.wait()
        if self.stage:
            self.recv_buf.copy_(rbuf)
        if self.n_recv:
            scatter(self.recv_ids, self.recv_buf[:self.n_recv])


# --------------------------------------------------------------------------- runner
def _check_single_byte(variable):
    """The halo moves one byte per value: graphs with a cardinality above 255 (2-byte device
    values) run on one GPU only."""
    if len(variable) and int(variable["cardinality"].max()) > 255:
        raise ValueError("cardinalities above 255 are single-GPU only")


class PartitionedGibbs(object):
    """One rank of a partitioned factor graph on its GPU."""

    def __init__(self, local, n_global, rank, world, device, seed, color_seed=0x5EED, group=None):
        _check_single_byte(local["variable"])
        import torch
        import torch.distributed as dist
        from . import _lib
        from .dataloading import assign_vtf_offsets, compute_var_map
        from .factorgraph import FactorGraph
        from .numbskulltypes import VarToFactor
        self.torch, self.dist, self.lib = torch, dist, _lib
        self.rank, self.world, self.group = rank, world, group
        self.n_owned = local["n_owned"]
        self.global_vid = local["global_vid"]
        self.dev = torch.device("cuda", device)
        torch.cuda.set_device(self.dev)

        variable = local["variable"]
        n_vtf = assign_vtf_offsets(variable)
        vmap = np.zeros(n_vtf, VarToFactor)
        findex = np.zeros(len(local["fmap"]), np.int64)
        compute_var_map(variable, local["factor"], local["fmap"], vmap, findex, local["domain_mask"])
        fg = FactorGraph(local["weight"], variable, local["factor"], local["fmap"], vmap, findex, 1, 1,
                         rank, 1, device=device, seed=seed)
        fg.global_vid = self.global_vid
        fg.color_seed = color_seed
        fg.deferred_coloring = True
        self.fg = fg
        L = _lib.lib()
        g = fg._device_graph()
        # everything (library kernels and NCCL transport) is ordered on torch's current stream
        _lib.check(L.nb_set_stream(g, C.c_void_p(torch.cuda.current_stream().cuda_stream)))

        if local.get("owner") is not None:                     # imported / locality-aware placement
            owner_arr = np.asarray(local["owner"])
            owner_of = lambda gids: owner_arr[gids]               # noqa: E731
        else:                                                   # contiguous owner blocks
            bounds = block_bounds(n_global, world)
            assert bounds[rank + 1] - bounds[rank] == self.n_owned and (self.n_owned == 0 or self.global_vid[0] == bounds[rank])
            owner_of = lambda gids: np.searchsorted(bounds, gids, side="right") - 1   # noqa: E731
        self.plan = HaloPlan(self.global_vid, self.n_owned, owner_of, rank, world, group, self.dev)

        # ---- distributed Jones-Plassmann ----
        full = Exchange(self.plan.send_ids, self.plan.recv_ids, rank, world, torch.int32, self.dev, group)
        def run_jp(mode, cap):
            """One distributed colouring attempt; returns (finished, rounds, global colour count)."""
            _lib.check(L.nb_color_restart(g, mode))
            rounds, finished = 0, False
            while cap <= 0 or rounds < cap:
                rem = C.c_int64(0)
                _lib.check(L.nb_color_round(g, C.byref(rem)))
                full.run(lambda ids, out: _lib.check(L.nb_gather_colors_dev(g, ids.data_ptr(), ids.numel(), out.data_ptr())),
                         lambda ids, buf: _lib.check(L.nb_scatter_colors_dev(g, ids.data_ptr(), ids.numel(), buf.data_ptr())))
                t = torch.tensor([rem.value], device=self.dev, dtype=torch.int64)
                if world > 1:
                    dist.all_reduce(t, group=group)
                rounds += 1
                if int(t.item()) == 0:
                    finished = True
                    break
            torch.cuda.synchronize()
            if not finished:
                return False, rounds, 0
            colors = fg.colors()
            t = torch.tensor([int(colors.max()) + 1 if len(colors) else 0], device=self.dev, dtype=torch.int64)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
            return True, rounds, int(t.item())

        # same policy as the single-GPU build (nb_build.cu color_graph): hashed priorities; if that
        # needs more than two colours, the natural order under the round cap; keep the smaller one.
        # Rounds are counted identically on one GPU and across ranks, so the choice is the same.
        _, rounds, self.n_colors = run_jp(0, 0)
        self.jp_mode = 0
        cap = int(L.nb_color_natural_round_cap())
        t = torch.tensor([int(fg.device_info()["max_arity"])], device=self.dev, dtype=torch.int64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
        if self.n_colors > 2 and cap > 0 and int(t.item()) <= 2:
            done, r1, nc = run_jp(1, cap)
            rounds += r1
            if done and nc < self.n_colors:
                self.n_colors, self.jp_mode = nc, 1
            else:
                _, r2, self.n_colors = run_jp(0, 0)
                rounds += r2
        self.jp_rounds = rounds
        # visit colours in increasing order of their smallest global variable id (same rule as the
        # single-GPU build, decided globally so that every rank relabels identically)
        mins = np.full(max(self.n_colors, 1), np.iinfo(np.int64).max, np.int64)
        _lib.check(L.nb_color_min_ids(g, self.n_colors, _lib.ptr(mins)))
        tm = torch.from_numpy(mins).to(self.dev)
        if world > 1:
            dist.all_reduce(tm, op=dist.ReduceOp.MIN, group=group)
        order = np.argsort(tm.cpu().numpy()[:self.n_colors], kind="stable")
        cmap = np.empty(self.n_colors, np.int32)
        cmap[order] = np.arange(self.n_colors, dtype=np.int32)
        _lib.check(L.nb_relabel_colors(g, _lib.ptr(cmap), self.n_colors))
        # Split every colour into a boundary phase (2c: the owned variables other ranks hold copies
        # of, a few rows) and an interior phase (2c + 1: variables that never read a ghost), so the
        # halo push of a colour travels while its interior is still being sampled.  Variables of
        # one colour are independent, so the samples do not change.
        import os
        self.split = world > 1 and os.environ.get("NUMBSKULL_B200_SPLIT", "1") != "0"
        if self.split:
            sends = [ids for ids in self.plan.send_ids if len(ids)]
            bnd = np.unique(np.concatenate(sends)).astype(np.int32) if sends else np.zeros(0, np.int32)
            _lib.check(L.nb_split_colors(g, _lib.ptr(bnd) if len(bnd) else None, len(bnd)))
        self.n_phases = self.n_colors * (2 if self.split else 1)
        _lib.check(L.nb_graph_finalize(g))
        phases = fg.colors()
        self.phases = phases
        self.colors = phases >> 1 if self.split else phases
        colors = phases

        # ---- per-phase halo exchanges (uint8 values); interior phases have none ----
        self.halo = []
        for c in range(self.n_phases):
            send, recv = self.plan.restrict(colors == c)
            assert not (self.split and c % 2 == 1 and (sum(map(len, send)) or sum(map(len, recv))))
            self.halo.append(Exchange(send, recv, rank, world, torch.uint8, self.dev, group))
        self.halo_bytes_per_sweep = sum(h.n_send for h in self.halo)
        # blocks without any ghost on any rank (independent sub-graphs that only share weights, e.g. the
        # candidates of the labelling-function model): no exchange, whole epochs in single launches
        t = torch.tensor([len(self.global_vid) - self.n_owned], device=self.dev, dtype=torch.int64)
        if world > 1:
            dist.all_reduce(t, group=group)
        self.any_halo = int(t.item()) > 0
        self.p2p = False
        self.p2p_nowait = 16 if os.environ.get("NUMBSKULL_B200_P2P_NOWAIT", "1") != "0" else 0
        if (world > 1 and dist.get_backend(group) == "nccl" and os.environ.get("NUMBSKULL_B200_P2P", "1") != "0"):
            # every rank must end up on the same transport: fall back to NCCL point-to-point
            # everywhere if any rank could not map its neighbours' memory
            ok = 1 if self._setup_p2p(colors) else 0
            t = torch.tensor([ok], device=self.dev, dtype=torch.int64)
            dist.all_reduce(t, op=dist.ReduceOp.MIN, group=group)
            self.p2p = bool(int(t.item()))

    def _setup_p2p(self, colors):
        """Peer-to-peer halo: owners store boundary values straight into the neighbours' ghost
        slots over NVLink (CUDA IPC mappings) and synchronise with a flag barrier in the kernel.
        Returns False (after taking part in every collective) if this rank cannot set it up."""
        L, lib, dist, g = self.lib.lib(), self.lib, self.dist, self.fg._g
        world, rank = self.world, self.rank
        handles = np.zeros(3 * 64, np.uint8)
        my_slots, ok = [np.zeros(0, np.int64)] * world, 1
        try:
            lib.check(L.nb_p2p_export(g, world, rank, lib.ptr(handles)))
            # slots (new ids) of my ghosts, per owner, in the order the owner sends them
            my_slots = []
            for p in range(world):
                ids = np.ascontiguousarray(self.plan.recv_ids[p], dtype=np.int32)
                out = np.zeros(len(ids), np.int32)
                if len(ids):
                    lib.check(L.nb_p2p_local_slots(g, lib.ptr(ids), len(ids), lib.ptr(out)))
                my_slots.append(out.astype(np.int64))
        except Exception as exc:  # noqa: BLE001
            self.p2p_error = str(exc)
            ok = 0
        th = self.torch.from_numpy(np.concatenate((handles, np.array([ok], np.uint8)))).to(self.dev)
        allh = [self.torch.zeros_like(th) for _ in range(world)]
        dist.all_gather(allh, th, group=self.group)
        allh = np.stack([t.cpu().numpy() for t in allh])
        # p's slots for what I send it, in my send order (tensors: a rank can have 10^7 ghosts)
        remote_slots = exchange_arrays(my_slots, rank, world, self.dev, self.group)
        if not allh[:, -1].all():
            return False
        try:
            neigh = [p for p in range(world)
                     if p != rank and (len(self.plan.send_ids[p]) or len(self.plan.recv_ids[p]))]
            hs = np.ascontiguousarray(allh[:, :3 * 64])
            nb_arr = np.asarray(neigh, np.int32)
            lib.check(L.nb_p2p_open(g, lib.ptr(hs), lib.ptr(nb_arr) if len(neigh) else None, len(neigh)))
            # plan entries grouped by phase: (owned local variable, peer rank, slot in the peer's value array)
            src = np.concatenate([self.plan.send_ids[p] for p in range(world)] + [np.zeros(0, np.int64)]).astype(np.int64)
            peer = np.concatenate([np.full(len(self.plan.send_ids[p]), p, np.int64) for p in range(world)] + [np.zeros(0, np.int64)])
            dst = np.concatenate([np.asarray(remote_slots[p], np.int64) for p in range(world)] + [np.zeros(0, np.int64)])
            assert len(src) == len(dst)
            phase = colors[src] if len(src) else np.zeros(0, np.int64)
            order = np.argsort(phase, kind="stable")
            ptr = np.zeros(self.n_phases + 1, np.int64)
            np.cumsum(np.bincount(phase, minlength=self.n_phases)[:self.n_phases], out=ptr[1:])
            cat = lambda x: np.ascontiguousarray(x[order], dtype=np.int32)  # noqa: E731
            src, peer, dst = cat(src), cat(peer), cat(dst)
            lib.check(L.nb_p2p_set_plan(g, self.n_phases, lib.ptr(ptr), lib.ptr(src), lib.ptr(peer), lib.ptr(dst)))
        except Exception as exc:  # noqa: BLE001  (CUDA IPC unavailable, peer access denied, ...)
            self.p2p_error = str(exc)
            return False
        return True

    # -- device helpers
    def _has_halo(self, c):
        """Interior phases (odd, split mode) exchange nothing on any rank."""
        return not (self.split and c % 2 == 1)

    def _exchange(self, c, chain):
        L, g, lib = self.lib.lib(), self.fg._g, self.lib
        if self.p2p:
            lib.check(L.nb_p2p_exchange(g, c, 1 << chain))
            return
        self.halo[c].run(
            lambda ids, out: lib.check(L.nb_gather_values_dev(g, chain, ids.data_ptr(), ids.numel(), out.data_ptr())),
            lambda ids, buf: lib.check(L.nb_scatter_values_dev(g, chain, ids.data_ptr(), ids.numel(), buf.data_ptr())))

    def sweeps(self, n, burnin, sample_evidence):
        """n chromatic Gibbs sweeps; after each colour the owners' new values reach the ghosts."""
        L, g, lib = self.lib.lib(), self.fg._g, self.lib
        if not self.any_halo:
            if n > 0:
                lib.check(L.nb_gibbs_sweeps(g, int(n), int(bool(burnin)), int(bool(sample_evidence)), self.fg.seed))
            return
        if self.world > 1 and self.p2p:
            # the whole launch sequence (colour kernels + halo pushes) is issued from C
            mode = (1 if self.p2p_nowait else 0) | (2 if self.split and self.p2p_nowait else 0)
            lib.check(L.nb_gibbs_sweeps_p2p(g, int(n), int(bool(burnin)), int(bool(sample_evidence)), self.fg.seed,
                                            self.n_phases, mode))
            return
        for _ in range(n):
            ep = C.c_int64(0)
            lib.check(L.nb_begin_epoch(g, C.byref(ep)))
            for c in range(self.n_phases):
                lib.check(L.nb_gibbs_color_phase(g, c, int(bool(burnin)), int(bool(sample_evidence)),
                                                 self.fg.seed, ep.value))
                if self.world > 1 and self._has_halo(c):
                    if self.p2p:
                        # push + signal only; the next colour's kernels wait for the neighbours' signal
                        lib.check(L.nb_p2p_exchange(g, c, 1 | self.p2p_nowait))
                    else:
                        self._exchange(c, 0)
        if self.world > 1 and self.p2p and n > 0:
            lib.check(L.nb_p2p_wait(g))

    def inference(self, burnin_epochs, epochs, sample_evidence=True):
        """FactorGraph.inference for the owned block; returns the owned marginals."""
        fg, L = self.fg, self.lib.lib()
        fg._sync_device(0, 0, evid=False, counts=True)
        self.sweeps(burnin_epochs, True, sample_evidence)
        self.sweeps(epochs, False, sample_evidence)
        self.torch.cuda.synchronize()
        if self.p2p:
            self.lib.check(L.nb_p2p_check(fg._g))
        fg._marg_epochs = epochs
        fg._mark_device_newer("var_value", "count", "marginals")
        return fg.marginals[:fg.cstart[self.n_owned]]

    def close(self):
        """Tear the rank's graph down: unmap the peers' arrays, synchronise, then free."""
        if self.fg._g is not None:
            self.torch.cuda.synchronize()
            if self.p2p:
                self.lib.check(self.lib.lib().nb_p2p_close(self.fg._g))
            if self.world > 1:
                self.dist.barrier(group=self.group)
            self.fg.clear()

    def inference_e2e(self, epochs):
        return self.inference(0, epochs, True)

    def learn(self, burnin_epochs, epochs, stepsize, decay, regularization, reg_param, truncation,
              learn_non_evidence=False, weight_sync="sum"):
        """FactorGraph.learn across the ranks: per colour both chains' boundary values are
        exchanged; per epoch the ranks' weight deltas are combined.  ``weight_sync="sum"`` is the
        reference master's rule (numbskull_master.py:223-224: ``weight_value += dw`` for every
        minion): to first order the move of one sequential pass over all ranks' variables, and right
        when a weight's factors live mostly on one rank.  ``"mean"`` averages the deltas (parameter
        averaging): the stable rule for data-parallel cuts of a model whose weights are tied across
        ALL ranks (the labelling-function model cut by candidate) -- there every rank's epoch already
        moves a weight most of the way to its optimum, and the sum of N such moves overshoots N-fold
        and diverges (505 M variables on 8 GPUs: |w| ~ 460 after 4 epochs)."""
        if weight_sync not in ("sum", "mean"):
            raise ValueError("weight_sync must be 'sum' or 'mean'")
        scale = 1.0 / self.world if weight_sync == "mean" else 1.0
        fg, L, lib, torch = self.fg, self.lib.lib(), self.lib, self.torch
        g = fg._device_graph()
        fg._sync_device(0, 0)
        self.sweeps(burnin_epochs, True, True)
        w_prev = torch.from_numpy(fg._host("weight_value", expose=False)[0].copy()).to(self.dev)
        w_now = torch.empty_like(w_prev)      # the deltas never leave the devices (nb_get/set_weights_dev + NCCL)
        for _ in range(epochs):
            if not self.any_halo:
                # one persistent launch per epoch (nb_learn_sweeps), then the ranks' deltas are summed
                s_ = C.c_double(float(stepsize))
                lib.check(L.nb_learn_sweeps(g, 1, C.byref(s_), 1.0, int(regularization), float(reg_param), float(truncation),
                                            int(bool(learn_non_evidence)), fg.seed, int(fg.batch_visits)))
                if self.world > 1:
                    lib.check(L.nb_get_weights_dev(g, C.c_void_p(w_now.data_ptr())))
                    delta = w_now - w_prev
                    if delta.is_cuda and self.dist.get_backend(self.group) == "gloo":
                        d = delta.cpu()
                        self.dist.all_reduce(d, group=self.group)
                        delta = d.to(self.dev)
                    else:
                        self.dist.all_reduce(delta, group=self.group)
                    w_prev = w_prev + delta * scale
                    lib.check(L.nb_set_weights_dev(g, C.c_void_p(w_prev.data_ptr())))
                stepsize *= decay
                continue
            ep = C.c_int64(0)
            lib.check(L.nb_begin_epoch(g, C.byref(ep)))
            nb = C.c_int(1)
            lib.check(L.nb_learn_blocks(g, float(stepsize), int(bool(learn_non_evidence)), int(fg.batch_visits),
                                        C.byref(nb)))
            n_blocks = nb.value
            if self.world > 1:
                t = torch.tensor([n_blocks], device=self.dev, dtype=torch.int64)
                self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX, group=self.group)
                n_blocks = int(t.item())
            for b in range(n_blocks):
                for c in range(self.n_phases):
                    lib.check(L.nb_learn_color_phase(g, c, b, n_blocks, float(stepsize), int(regularization),
                                                     float(reg_param), float(truncation),
                                                     int(bool(learn_non_evidence)), fg.seed, ep.value))
                    if self.world > 1 and self._has_halo(c):
                        if self.p2p:
                            lib.check(L.nb_p2p_exchange(g, c, 3))
                        else:
                            self._exchange(c, 0)
                            self._exchange(c, 1)
            if self.world > 1:
                lib.check(L.nb_get_weights_dev(g, C.c_void_p(w_now.data_ptr())))
                delta = w_now - w_prev
                if delta.is_cuda and self.dist.get_backend(self.group) == "gloo":   # 1-GPU tests: gloo moves host memory
                    d = delta.cpu()
                    self.dist.all_reduce(d, group=self.group)
                    delta = d.to(self.dev)
                else:
                    self.dist.all_reduce(delta, group=self.group)
                w_prev = w_prev + delta * scale
                lib.check(L.nb_set_weights_dev(g, C.c_void_p(w_prev.data_ptr())))
            stepsize *= decay
        torch.cuda.synchronize()
        fg._mark_device_newer("var_value", "var_value_evid")
        fg._stale.add("weight_value")
        fg._fetch("weight_value")
        return stepsize


def partition_graph(weight, variable, factor, fmap, rank, world, device, seed, group=None, color_seed=0x5EED,
                    owner=None):
    """Partition a global graph (every rank passes the same arrays): contiguous owner blocks, or
    the placement ``owner[v]`` -- e.g. :func:`owners_from_salt_keys` (the reference's partition
    keys) or :func:`locality_owners`.  Samples do not depend on the placement: colours and Philox
    streams are functions of the global ids."""
    _check_single_byte(variable)
    if owner is None:
        # contiguous blocks: the same cut as extract_local (the tests compare them), made by host threads
        bounds = block_bounds(len(variable), world)
        owner = (np.searchsorted(bounds, np.arange(len(variable), dtype=np.int64), side="right") - 1).astype(np.int32)
    local = extract_local_by_owner(weight, variable, factor, fmap, owner, rank)
    return PartitionedGibbs(local, len(variable), rank, world, device, seed, color_seed, group)


def lf_block(copies_total, n_lf, rank, world, seed=1003):
    """Rank ``rank``'s candidates of the labelling-function model (BASELINE config 3; full size:
    10 M candidates x 100 labelling functions = 1.01 B variables, beyond one GPU's 2^31 ids, so it
    exists only in partitioned form).  Candidates are independent given the weights: the block has
    no ghosts, the ranks only meet in the per-epoch weight-delta all-reduce.  Built locally; the
    labelling-function accuracies are a function of ``seed`` alone, the votes of (seed, rank)."""
    from . import synth
    per = 1 + n_lf
    c_lo, c_hi = copies_total * rank // world, copies_total * (rank + 1) // world
    acc = np.random.default_rng(seed).uniform(0.55, 0.95, n_lf)
    w, v, f, fm, dm, e = synth.lf_model(c_hi - c_lo, n_lf, np.random.default_rng([seed, rank]), accuracy=acc)
    gv = np.arange(c_lo * per, c_hi * per, dtype=np.int64)
    return dict(weight=w, variable=v, factor=f, fmap=fm, domain_mask=dm, global_vid=gv, n_owned=len(v)), copies_total * per


def ising_strip_runner(rows, cols, rank, world, device, seed):
    local, n_global = ising_strip(rows, cols, rank, world)
    return PartitionedGibbs(local, n_global, rank, world, device, seed)
