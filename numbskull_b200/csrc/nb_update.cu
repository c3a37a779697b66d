// In-place edits of the record fields that do not change the layout of a built graph:
// variable.isEvidence / initialValue (plus a chain value) and weight.isFixed.  The sort key of a
// variable (row class, colour, id window, row length) depends on none of them, so patching the few
// words that carry them leaves the device graph byte for byte what a rebuild from the edited
// records would produce -- nb_graph_digest makes that checkable.
#include <algorithm>
#include <cstring>

#include "nb_eval.cuh"

static inline unsigned grid_for(int64_t n, int block = 256) { return (unsigned)std::max<int64_t>(1, (n + block - 1) / block); }
static inline size_t align16(size_t x) { return (x + 15) & ~(size_t)15; }

// Ids validated against [0, bound), then one entry per id in increasing id order: the LAST
// occurrence of a duplicated id, as numpy's a[ids] = x.  Resolved here so that the device scatter
// never sees two writes to one place.
static int last_wins(const int64_t *ids, int64_t n, int64_t bound, const char *what, std::vector<int64_t> &pick)
{
    bool increasing = true;
    for (int64_t i = 0; i < n; i++) {
        if (ids[i] < 0 || ids[i] >= bound)
            NB_FAIL(NB_ERR_INVALID, "%s id %lld out of range [0, %lld)", what, (long long)ids[i], (long long)bound);
        if (i && ids[i] <= ids[i - 1]) increasing = false;
    }
    pick.clear();
    if (increasing) {
        pick.resize((size_t)n);
        for (int64_t i = 0; i < n; i++) pick[(size_t)i] = i;
        return NB_OK;
    }
    if (n >= (1ll << 33)) NB_FAIL(NB_ERR_INVALID, "more than 2^33 entries in one update");
    std::vector<uint64_t> key((size_t)n);   // id:31 | entry index:33
    for (int64_t i = 0; i < n; i++) key[(size_t)i] = ((uint64_t)ids[i] << 33) | (uint64_t)i;
    std::sort(key.begin(), key.end());
    for (int64_t k = 0; k < n; k++)
        if (k + 1 == n || (key[(size_t)k + 1] >> 33) != (key[(size_t)k] >> 33))
            pick.push_back((int64_t)(key[(size_t)k] & ((1ull << 33) - 1)));
    return NB_OK;
}

// ---------------------------------------------------------------------------
// variables
// ---------------------------------------------------------------------------
// error key: kind:32 | variable id (the smallest id of the first kind wins: deterministic message)
#define NB_UPD_GHOST 0ull
#define NB_UPD_EVID_INIT 1ull
#define NB_UPD_VALUE 2ull

__global__ void k_update_vars_check(int64_t m, const int32_t *ids, const int8_t *evid, const int64_t *init, const int64_t *value,
                                    const int8_t *v_evid, const int32_t *v_card, const int32_t *v_init,
                                    unsigned long long *err)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= m) return;
    const int v = ids[i];
    const int cur = v_evid[v], card = v_card[v];
    unsigned long long bad = ~0ull;
    if (cur == 4) bad = (NB_UPD_GHOST << 32) | (unsigned)v;
    else {
        const int e = evid ? evid[i] : cur;
        // without a new initialValue the stored one counts (the build stores an out-of-domain one as 0)
        const int64_t x = init ? init[i] : (int64_t)v_init[v];
        if (e == 1 && (x < 0 || x >= card)) bad = (NB_UPD_EVID_INIT << 32) | (unsigned)v;
        else if (value && (value[i] < 0 || value[i] >= card)) bad = (NB_UPD_VALUE << 32) | (unsigned)v;
    }
    if (bad != ~0ull) atomicMin(err, bad);
}

// the build's packing (k_assign_ids / extract_and_upload): isEvidence & 0xF into vmeta, the raw
// byte into v_evid; initialValue where it lies in [0, card), else 0
template <class T>
__global__ void k_update_vars(int64_t m, const int32_t *ids, const int8_t *evid, const int64_t *init, const int64_t *value,
                              const int32_t *old2new, const int32_t *v_card, int8_t *v_evid, int32_t *v_init, uint32_t *vmeta,
                              T *vinit, T *val0, T *val1)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= m) return;
    const int v = ids[i];
    const int64_t nid = old2new[v];
    if (evid) {
        v_evid[v] = evid[i];
        vmeta[nid] = (vmeta[nid] & ~(0xFu << 8)) | ((uint32_t)(evid[i] & 0xF) << 8);
    }
    if (init) {
        const int64_t x = init[i];
        const int32_t s = (x >= 0 && x < v_card[v]) ? (int32_t)x : 0;
        v_init[v] = s;
        vinit[nid] = (T)s;
    }
    if (value) {
        val0[nid] = (T)value[i];
        val1[nid] = (T)value[i];
    }
}

extern "C" int nb_update_variables(nb_graph *g, const int64_t *var_ids, int64_t n, const int8_t *is_evidence,
                                   const int64_t *initial_value, const int64_t *value)
{
    if (!g->finalized) NB_FAIL(NB_ERR_INVALID, "graph not finalized");
    if (n < 0) NB_FAIL(NB_ERR_INVALID, "negative entry count");
    if (n == 0 || (!is_evidence && !initial_value && !value)) return NB_OK;
    if (!var_ids) NB_FAIL(NB_ERR_INVALID, "null variable ids");
    NB_CUDA(cudaSetDevice(g->device));
    std::vector<int64_t> pick;
    NB_TRY(last_wins(var_ids, n, g->V, "variable", pick));
    if (is_evidence)
        for (int64_t i : pick)
            if (is_evidence[i] == 4)
                NB_FAIL(NB_ERR_INVALID, "isEvidence 4 marks a ghost, which only the partitioner creates (variable %lld)",
                        (long long)var_ids[i]);
    const int64_t m = (int64_t)pick.size();
    // staging: ids int32 | isEvidence int8 | initialValue int64 | value int64 | error word
    const size_t o_ev = align16((size_t)m * 4), o_in = align16(o_ev + (is_evidence ? (size_t)m : 0));
    const size_t o_va = align16(o_in + (initial_value ? (size_t)m * 8 : 0));
    const size_t o_err = align16(o_va + (value ? (size_t)m * 8 : 0));
    NB_TRY(nb_ensure_pinned(g, o_err + 16));
    NB_TRY(nb_ensure_xfer(g, o_err + 16));
    char *h = (char *)g->h_pinned, *d = (char *)g->d_xfer;
    for (int64_t k = 0; k < m; k++) {
        const int64_t i = pick[(size_t)k];
        ((int32_t *)h)[k] = (int32_t)var_ids[i];
        if (is_evidence) ((int8_t *)(h + o_ev))[k] = is_evidence[i];
        if (initial_value) ((int64_t *)(h + o_in))[k] = initial_value[i];
        if (value) ((int64_t *)(h + o_va))[k] = value[i];
    }
    NB_CUDA(cudaMemcpyAsync(d, h, o_err, cudaMemcpyHostToDevice, g->stream));
    unsigned long long *d_err = (unsigned long long *)(d + o_err);
    NB_CUDA(cudaMemsetAsync(d_err, 0xFF, 8, g->stream));
    const int32_t *ids = (const int32_t *)d;
    const int8_t *ev = is_evidence ? (const int8_t *)(d + o_ev) : nullptr;
    const int64_t *in = initial_value ? (const int64_t *)(d + o_in) : nullptr;
    const int64_t *va = value ? (const int64_t *)(d + o_va) : nullptr;
    k_update_vars_check<<<grid_for(m), 256, 0, g->stream>>>(m, ids, ev, in, va, g->d_v_evid, g->d_v_card, g->d_v_init, d_err);
    unsigned long long err = 0;
    NB_CUDA(cudaMemcpyAsync(&err, d_err, 8, cudaMemcpyDeviceToHost, g->stream));
    NB_CUDA(cudaStreamSynchronize(g->stream));
    if (err != ~0ull) {
        const long long v = (long long)(err & 0xFFFFFFFFull);
        switch (err >> 32) {
        case NB_UPD_GHOST: NB_FAIL(NB_ERR_INVALID, "variable %lld is a ghost (isEvidence 4): the partitioner owns it", v);
        case NB_UPD_EVID_INIT:
            NB_FAIL(NB_ERR_INVALID, "invalid factor graph: evidence variable with initialValue outside [0, cardinality) (index %lld)", v);
        default: NB_FAIL(NB_ERR_INVALID, "value of variable %lld lies outside [0, cardinality)", v);
        }
    }
    if (g->value_bytes == 1)
        k_update_vars<nb_val_t><<<grid_for(m), 256, 0, g->stream>>>(m, ids, ev, in, va, g->d_old2new, g->d_v_card, g->d_v_evid,
                                                                    g->d_v_init, g->d_vmeta, (nb_val_t *)g->d_vinit,
                                                                    nb_vals<nb_val_t>(g, 0), nb_vals<nb_val_t>(g, 1));
    else
        k_update_vars<nb_val16_t><<<grid_for(m), 256, 0, g->stream>>>(m, ids, ev, in, va, g->d_old2new, g->d_v_card, g->d_v_evid,
                                                                       g->d_v_init, g->d_vmeta, (nb_val16_t *)g->d_vinit,
                                                                       nb_vals<nb_val16_t>(g, 0), nb_vals<nb_val16_t>(g, 1));
    NB_CUDA(cudaGetLastError());
    NB_CUDA(cudaStreamSynchronize(g->stream));
    // the per-colour visit bounds of learning count the evidence rows only (k_visit_histogram)
    if (is_evidence) g->learn_vmax_flag = -1;
    return NB_OK;
}

// ---------------------------------------------------------------------------
// weight.isFixed
// ---------------------------------------------------------------------------
// Every kernel sets the fixed bit of the records whose weight is marked in `chg` to wfixed[wid].
// Padding records (wid 0, fixed bit set) lie past a row's incidence count and are never touched.
__device__ __forceinline__ uint32_t nb_with_bit(uint32_t w, uint32_t bit, int on) { return on ? (w | bit) : (w & ~bit); }

__global__ void k_mark_weights(int64_t k, const int32_t *wids, const uint8_t *fixed, uint8_t *chg, uint8_t *wfixed)
{
    const int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (j < k) { chg[wids[j]] = 1; wfixed[wids[j]] = fixed[j]; }
}

// generic headers of the thread rows (SELL-32 words; compact bit 25 of the header, wide bit 25 of its second word)
template <bool WIDE>
__global__ void k_fix_thread_rows(int64_t n_trows, const int32_t *new2old, const uint32_t *rowlen, const int64_t *slice_ptr,
                                  uint32_t *twords, const uint8_t *chg, const uint8_t *wfixed)
{
    const int64_t nid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (nid >= n_trows) return;
    const int v = new2old[nid];
    if (v < 0) return;
    const int len = (int)rowlen[v];
    const NbRow r = nb_thread_row(twords, slice_ptr, nid);
    for (int pos = 0; pos < len;) {
        const NbHdr h = nb_read_hdr<WIDE>(r, pos);
        if (h.code != C_MARK && chg[h.wid]) {
            uint32_t *w = nb_thread_row_word(twords, slice_ptr, nid, WIDE ? pos + 1 : pos);
            *w = nb_with_bit(*w, 1u << 25, wfixed[h.wid]);
        }
        pos += nb_inc_words<WIDE>(h);
    }
}

// generic headers of the warp rows: one thread per incidence (d_inc holds its offset in the row)
template <bool WIDE>
__global__ void k_fix_warp_rows(int64_t n_inc, int64_t n_wrows, const int64_t *inc_ptr, const uint2 *inc, const int64_t *wrow_ptr,
                                uint32_t *wwords, const uint8_t *chg, const uint8_t *wfixed)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n_inc) return;
    int64_t lo = 0, hi = n_wrows - 1;   // the row r with inc_ptr[r] <= i < inc_ptr[r + 1]
    while (lo < hi) {
        const int64_t mid = (lo + hi + 1) >> 1;
        if (inc_ptr[mid] <= i) lo = mid;
        else hi = mid - 1;
    }
    uint32_t *p = wwords + wrow_ptr[lo] + inc[i].x;
    const uint32_t wid = WIDE ? p[0] : (p[0] & 0xFFFFFu);
    if (chg[wid]) {
        uint32_t *w = WIDE ? p + 1 : p;
        *w = nb_with_bit(*w, 1u << 25, wfixed[wid]);
    }
}

// truth-table quads of the PAIR + FAST rows (weight ids in tt_wid)
__global__ void k_fix_tt(int64_t n_frows, const int32_t *new2old, const uint32_t *ninc, const int64_t *tt_ptr, uint4 *tt,
                         const uint32_t *tt_wid, const uint8_t *chg, const uint8_t *wfixed)
{
    const int64_t nid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (nid >= n_frows) return;
    const int v = new2old[nid];
    if (v < 0) return;
    const int64_t base = tt_ptr[nid >> 5] + (nid & 31);
    for (uint32_t e = 0; e < ninc[v]; e++) {
        const int64_t q = base + (int64_t)e * 32;
        const uint32_t wid = tt_wid[q];
        if (chg[wid]) tt[q].z = nb_with_bit(tt[q].z, NB_TT_FIXED_BIT, wfixed[wid]);
    }
}

// pair stream: the 8-byte records of mixed slices (wid in the word), the hoisted word of uniform ones
__global__ void k_fix_tt2(int64_t n_prows, const int32_t *new2old, const uint32_t *ninc, const int64_t *tt2_ptr, uint4 *tt2,
                          uint32_t *tt2_common, const uint8_t *chg, const uint8_t *wfixed)
{
    const int64_t nid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (nid >= n_prows) return;
    const int64_t s = nid >> 5;
    const uint32_t common = tt2_common[s];
    if (common != NB_PAIR_NONE) {   // one weight for the whole slice: it stays uniform
        if ((nid & 31) == 0 && chg[common >> 10]) tt2_common[s] = nb_with_bit(common, NB_PAIR_FIXED_BIT, wfixed[common >> 10]);
        return;
    }
    const int v = new2old[nid];
    if (v < 0) return;
    uint4 *row = tt2 + tt2_ptr[s] + (nid & 31);
    for (uint32_t e = 0; e < ninc[v]; e++) {
        uint32_t *w = reinterpret_cast<uint32_t *>(row + (size_t)(e >> 1) * 32) + 2 * (e & 1) + 1;
        const uint32_t wid = *w >> 10;
        if (chg[wid]) *w = nb_with_bit(*w, NB_PAIR_FIXED_BIT, wfixed[wid]);
    }
}

// categorical records of the CAT rows (weight ids in cat_wid; fixed is bit 26 of the packed word)
__global__ void k_fix_cat(int64_t first_id, int64_t end_id, const int32_t *new2old, const uint32_t *ninc, const int64_t *cat_ptr,
                          uint4 *cat, const uint32_t *cat_wid, const uint8_t *chg, const uint8_t *wfixed)
{
    const int64_t nid = first_id + blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (nid >= end_id) return;
    const int v = new2old[nid];
    if (v < 0) return;
    const int64_t base = cat_ptr[(nid - first_id) >> 5] + (nid & 31);
    for (uint32_t e = 0; e < ninc[v]; e++) {
        const int64_t q = base + (int64_t)e * 32;
        const uint32_t wid = cat_wid[q];
        if (chg[wid]) cat[q].z = nb_with_bit(cat[q].z, 1u << 26, wfixed[wid]);
    }
}

extern "C" int nb_update_weights_fixed(nb_graph *g, const int64_t *weight_ids, int64_t n, const uint8_t *is_fixed)
{
    if (!g->finalized) NB_FAIL(NB_ERR_INVALID, "graph not finalized");
    if (n < 0) NB_FAIL(NB_ERR_INVALID, "negative entry count");
    if (n == 0) return NB_OK;
    if (!weight_ids || !is_fixed) NB_FAIL(NB_ERR_INVALID, "null weight ids or flags");
    for (int64_t i = 0; i < n; i++)
        if (weight_ids[i] < 0 || weight_ids[i] >= g->W)
            NB_FAIL(NB_ERR_INVALID, "weight id %lld out of range [0, %lld)", (long long)weight_ids[i], (long long)g->W);
    NB_CUDA(cudaSetDevice(g->device));
    const int64_t W = g->W;
    if ((int64_t)g->h_wfixed.size() != W) {   // host copy of d_wfixed: tells which flags actually change
        g->h_wfixed.assign((size_t)W, 0);
        NB_CUDA(cudaMemcpyAsync(g->h_wfixed.data(), g->d_wfixed, (size_t)W, cudaMemcpyDeviceToHost, g->stream));
        NB_CUDA(cudaStreamSynchronize(g->stream));
    }
    // apply in order (the last occurrence of an id wins), then list each weight whose flag changed once
    std::vector<uint8_t> next(g->h_wfixed);
    for (int64_t i = 0; i < n; i++) next[(size_t)weight_ids[i]] = is_fixed[i] ? 1 : 0;
    std::vector<int32_t> wids;
    for (int64_t i = 0; i < n; i++) {
        const size_t w = (size_t)weight_ids[i];
        if ((next[w] & 1) != g->h_wfixed[w] && !(next[w] & 2)) { wids.push_back((int32_t)w); next[w] |= 2; }
    }
    if (wids.empty()) return NB_OK;
    const int64_t k = (int64_t)wids.size();
    // device scratch: changed map (W bytes) | ids int32 | flags uint8
    const size_t o_ids = align16((size_t)W), o_fix = align16(o_ids + (size_t)k * 4), bytes = o_fix + (size_t)k;
    NB_TRY(nb_ensure_pinned(g, bytes - o_ids));
    NB_TRY(nb_ensure_xfer(g, bytes));
    char *h = (char *)g->h_pinned, *d = (char *)g->d_xfer;
    for (int64_t j = 0; j < k; j++) {
        ((int32_t *)h)[j] = wids[(size_t)j];
        (h + (o_fix - o_ids))[j] = next[(size_t)wids[(size_t)j]] & 1;
    }
    uint8_t *chg = (uint8_t *)d;
    NB_CUDA(cudaMemsetAsync(chg, 0, (size_t)W, g->stream));
    NB_CUDA(cudaMemcpyAsync(d + o_ids, h, bytes - o_ids, cudaMemcpyHostToDevice, g->stream));
    k_mark_weights<<<grid_for(k), 256, 0, g->stream>>>(k, (const int32_t *)(d + o_ids), (const uint8_t *)(d + o_fix), chg,
                                                                g->d_wfixed);
    const uint8_t *wf = g->d_wfixed;
    if (g->n_trows) {
        if (g->wide)
            k_fix_thread_rows<true><<<grid_for(g->n_trows), 256, 0, g->stream>>>(g->n_trows, g->d_new2old, g->d_rowlen0, g->d_slice_ptr,
                                                                                  g->d_twords, chg, wf);
        else
            k_fix_thread_rows<false><<<grid_for(g->n_trows), 256, 0, g->stream>>>(g->n_trows, g->d_new2old, g->d_rowlen0, g->d_slice_ptr,
                                                                                   g->d_twords, chg, wf);
    }
    if (g->n_inc) {
        if (g->wide)
            k_fix_warp_rows<true><<<grid_for(g->n_inc), 256, 0, g->stream>>>(g->n_inc, g->n_wrows, g->d_inc_ptr, g->d_inc, g->d_wrow_ptr,
                                                                             g->d_wwords, chg, wf);
        else
            k_fix_warp_rows<false><<<grid_for(g->n_inc), 256, 0, g->stream>>>(g->n_inc, g->n_wrows, g->d_inc_ptr, g->d_inc, g->d_wrow_ptr,
                                                                              g->d_wwords, chg, wf);
    }
    if (g->n_tt_quads)
        k_fix_tt<<<grid_for(g->n_frows), 256, 0, g->stream>>>(g->n_frows, g->d_new2old, g->d_ninc0, g->d_tt_ptr, g->d_tt, g->d_tt_wid,
                                                               chg, wf);
    if (g->n_prows)
        k_fix_tt2<<<grid_for(g->n_prows), 256, 0, g->stream>>>(g->n_prows, g->d_new2old, g->d_ninc0, g->d_tt2_ptr, g->d_tt2,
                                                               g->d_tt2_common, chg, wf);
    if (g->n_cat_quads)
        k_fix_cat<<<grid_for(g->n_crows - g->n_frows), 256, 0, g->stream>>>(g->n_frows, g->n_crows, g->d_new2old, g->d_ninc0,
                                                                            g->d_cat_ptr, g->d_cat, g->d_cat_wid, chg, wf);
    NB_CUDA(cudaGetLastError());
    NB_CUDA(cudaStreamSynchronize(g->stream));
    for (int32_t w : wids) g->h_wfixed[(size_t)w] = next[(size_t)w] & 1;
    // the per-colour visit bounds of learning skip fixed incidences (k_visit_histogram)
    g->learn_vmax_flag = -1;
    return NB_OK;
}

// ---------------------------------------------------------------------------
// digest
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint64_t nb_digest_mix(uint64_t x)
{
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

// sum over i of mix(mix(i) ^ x[i]) mod 2^64: keyed by position, independent of the summation order
template <class E>
__global__ void k_digest(const E *p, int64_t n, unsigned long long *out)
{
    uint64_t acc = 0;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        acc += nb_digest_mix(nb_digest_mix((uint64_t)i) ^ (uint64_t)p[i]);
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(0xFFFFFFFFu, acc, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(out, (unsigned long long)acc);
}

template <class E>
static void digest_launch(nb_graph *g, const void *p, int64_t n, unsigned long long *out)
{
    if (!p || n <= 0) return;   // absent arrays hash as 0
    const unsigned grid = (unsigned)std::min<int64_t>(grid_for(n), 148 * 16);
    k_digest<E><<<grid, 256, 0, g->stream>>>((const E *)p, n, out);
}

extern "C" int nb_graph_digest(const nb_graph *gc, uint64_t *digest, int n)
{
    nb_graph *g = const_cast<nb_graph *>(gc);
    if (!g->finalized) NB_FAIL(NB_ERR_INVALID, "graph not finalized");
    if (n < NB_DIGEST_ARRAYS) NB_FAIL(NB_ERR_INVALID, "digest needs room for %d words", NB_DIGEST_ARRAYS);
    NB_CUDA(cudaSetDevice(g->device));
    unsigned long long *d;
    NB_CUDA(cudaMalloc(&d, NB_DIGEST_ARRAYS * 8));
    cudaMemsetAsync(d, 0, NB_DIGEST_ARRAYS * 8, g->stream);
    const int64_t Vn = g->Vn, V = g->V;
    digest_launch<uint32_t>(g, g->d_vmeta, Vn, d + 0);
    if (g->value_bytes == 1) digest_launch<uint8_t>(g, g->d_vinit, Vn, d + 1);
    else digest_launch<uint16_t>(g, g->d_vinit, Vn, d + 1);
    digest_launch<uint16_t>(g, g->d_vcard, Vn, d + 2);
    digest_launch<uint8_t>(g, g->d_v_evid, V, d + 3);
    digest_launch<uint32_t>(g, g->d_v_init, V, d + 4);
    digest_launch<uint8_t>(g, g->d_wfixed, g->W, d + 5);
    digest_launch<uint32_t>(g, g->d_twords, g->n_twords, d + 6);
    digest_launch<uint32_t>(g, g->d_wwords, g->n_wwords, d + 7);
    digest_launch<uint32_t>(g, g->d_tt, 4 * g->n_tt_quads, d + 8);
    digest_launch<uint32_t>(g, g->d_tt_wid, g->n_tt_quads, d + 9);
    digest_launch<uint32_t>(g, g->d_tt2, 4 * g->n_tt2_quads, d + 10);
    digest_launch<uint32_t>(g, g->d_tt2_common, g->n_prows / 32, d + 11);
    digest_launch<uint32_t>(g, g->d_cat, 4 * g->n_cat_quads, d + 12);
    digest_launch<uint32_t>(g, g->d_cat_wid, g->n_cat_quads, d + 13);
    digest_launch<uint32_t>(g, g->d_new2old, Vn, d + 14);
    unsigned long long h[NB_DIGEST_ARRAYS];
    cudaMemcpyAsync(h, d, sizeof(h), cudaMemcpyDeviceToHost, g->stream);
    cudaError_t e = cudaStreamSynchronize(g->stream);
    cudaFree(d);
    NB_CUDA(e);
    NB_CUDA(cudaGetLastError());
    for (int i = 0; i < NB_DIGEST_ARRAYS; i++) digest[i] = (uint64_t)h[i];
    return NB_OK;
}
