// Device-graph construction: AoS records -> SoA upload -> Jones-Plassmann
// colouring -> (colour, window, row length) ordering -> SELL-32 / contiguous
// incidence streams resident in HBM.
#include <algorithm>
#include <atomic>
#include <cstdlib>
#include <cstring>
#include <thread>
#include <cub/cub.cuh>

#include "nb_eval.cuh"

// ---------------------------------------------------------------------------
// small host helpers
// ---------------------------------------------------------------------------
template <class F>
static void parallel_for(int64_t n, F fn)
{
    int nt = (int)std::min<int64_t>(std::max(1u, std::thread::hardware_concurrency()), 64);
    if (n < (1 << 16)) nt = 1;
    if (nt == 1) { fn(0, n); return; }
    std::vector<std::thread> th;
    int64_t chunk = (n + nt - 1) / nt;
    for (int t = 0; t < nt; t++) {
        int64_t a = t * chunk, b = std::min(n, a + chunk);
        if (a >= b) break;
        th.emplace_back([=] { fn(a, b); });
    }
    for (auto &t : th) t.join();
}

int nb_dev_alloc(nb_graph *g, void **p, size_t bytes, bool zero)
{
    *p = nullptr;
    if (bytes == 0) bytes = 16;
    cudaError_t e = cudaMalloc(p, bytes);
    if (e != cudaSuccess) {
        nb_set_error("cudaMalloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
        return e == cudaErrorMemoryAllocation ? NB_ERR_NOMEM : NB_ERR_CUDA;
    }
    g->allocs.push_back(*p);
    g->device_bytes += (int64_t)bytes;
    if (zero) NB_CUDA(cudaMemsetAsync(*p, 0, bytes, g->stream));
    return NB_OK;
}

int nb_ensure_xfer(nb_graph *g, size_t bytes)
{
    if (g->xfer_bytes >= bytes) return NB_OK;
    if (g->d_xfer) cudaFree(g->d_xfer);
    g->d_xfer = nullptr;
    g->xfer_bytes = 0;
    cudaError_t e = cudaMalloc(&g->d_xfer, bytes);
    if (e != cudaSuccess) NB_FAIL(NB_ERR_NOMEM, "cudaMalloc(xfer %zu) failed: %s", bytes, cudaGetErrorString(e));
    g->xfer_bytes = bytes;
    return NB_OK;
}

int nb_ensure_pinned(nb_graph *g, size_t bytes)
{
    if (g->pinned_bytes >= bytes) return NB_OK;
    if (g->h_pinned) cudaFreeHost(g->h_pinned);
    g->h_pinned = nullptr;
    g->pinned_bytes = 0;
    cudaError_t e = cudaMallocHost(&g->h_pinned, bytes);
    if (e != cudaSuccess) NB_FAIL(NB_ERR_NOMEM, "cudaMallocHost(%zu) failed: %s", bytes, cudaGetErrorString(e));
    g->pinned_bytes = bytes;
    return NB_OK;
}

template <class T>
static int upload(nb_graph *g, T **dst, const std::vector<T> &src)
{
    NB_TRY(nb_alloc(g, dst, src.size(), false));
    if (!src.empty())
        NB_CUDA(cudaMemcpyAsync(*dst, src.data(), src.size() * sizeof(T), cudaMemcpyHostToDevice, g->stream));
    NB_CUDA(cudaStreamSynchronize(g->stream));
    return NB_OK;
}

// ---------------------------------------------------------------------------
// kernels
// ---------------------------------------------------------------------------
struct RawGraph {
    int64_t V;
    const int8_t *v_evid;
    const int32_t *v_card;
    const int8_t *v_dtype;
    const int64_t *v_vtf;
    const int64_t *b_off;
    const int32_t *b_len;
    const int32_t *fi;
    const uint8_t *f_code;
    const int32_t *f_wid;
    const double *f_feat;
    const int32_t *f_arity;
    const int64_t *f_off;
    const int32_t *m_vid;
    const int32_t *m_eq;
    const int64_t *gid;
    bool wide;
    bool val16;     // 2-byte value graph (some cardinality above 255)
};

__device__ __forceinline__ int nbuckets(const RawGraph &G, int64_t v) { return G.v_dtype[v] == 0 ? 1 : G.v_card[v]; }

// words and incidences of every row (ghost rows are empty: they are never sampled), and whether
// the row qualifies for the single-pass Boolean kernel (NB_CLASS_FAST)
__global__ void k_row_size(RawGraph G, uint32_t *rowlen, uint32_t *ninc, uint8_t *fast, int *overflow)
{
    int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (v >= G.V) return;
    if (G.v_evid[v] == 4) { rowlen[v] = 0; ninc[v] = 0; fast[v] = 0; return; }
    uint64_t words = 0, inc = 0;
    int nb = nbuckets(G, v);
    bool ok = G.v_dtype[v] == 0 && G.v_card[v] == 2;
    bool pair = true;
    bool catok = G.v_dtype[v] == 1 && G.v_card[v] <= NB_CAT_MAX_CARD;
    for (int b = 0; b < nb; b++) {
        int64_t off = G.b_off[G.v_vtf[v] + b];
        int len = G.b_len[G.v_vtf[v] + b];
        if (G.v_dtype[v] == 1 && len > 0) words += G.wide ? 2 : 1;
        for (int e = 0; e < len; e++) {
            int f = G.fi[off + e];
            int code = G.f_code[f], a = G.f_arity[f];
            words += nb_incidence_words(G.wide, code, a, G.f_feat[f] != 1.0);
            if (catok) catok = (code == C_AND_CAT || code == C_EQUAL_CAT_CONST) && a <= 3 && G.f_feat[f] == 1.0;
            // the records hold the other members' dense_equal_to in 8 bits; on a 2-byte graph a member
            // value of 255 or more would compare against a truncated one: such rows stay generic
            if (catok && G.val16)
                for (int j = 0; j < a; j++)
                    catok &= G.m_vid[G.f_off[f] + j] == v || (uint32_t)G.m_eq[G.f_off[f] + j] <= 0xFFu;
            if (ok) {   // truth-table class: arity <= 3, integer-valued function, small member domains
                if (!nb_code_tt_ok(code) || a > 3 || G.f_feat[f] != 1.0) ok = false;
                else if (!nb_code_tt_const_compare(code))
                    for (int j = 0; j < a; j++) ok &= G.v_card[G.m_vid[G.f_off[f] + j]] <= 3;
                int others = 0;
                for (int j = 0; j < a && j < 3; j++) others += G.m_vid[G.f_off[f] + j] != v;
                pair &= others <= 1 && (uint32_t)G.f_wid[f] <= NB_PAIR_MAX_WID;
            }
        }
        inc += len;
    }
    if (words > 0x7FFFFFFFull || inc > 0x7FFFFFFFull) { *overflow = 1; words = 0; inc = 0; }
    rowlen[v] = (uint32_t)words;
    ninc[v] = (uint32_t)inc;
    fast[v] = ok ? (pair ? 2 : 1) : (catok ? 3 : 0);
}

__host__ __device__ inline uint64_t nb_mix64(uint64_t x)
{
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}
// Jones-Plassmann priority: a pure function of the GLOBAL variable id
__host__ __device__ inline uint64_t nb_jp_priority(uint64_t gid, uint64_t seed)
{
    return (nb_mix64(gid ^ nb_mix64(seed)) & 0xFFFFFFFF00000000ull) | (gid & 0xFFFFFFFFull);
}

// One Jones-Plassmann round.  A variable takes the smallest colour unused by its
// neighbours once every neighbour of higher priority is coloured; the outcome
// equals a sequential greedy colouring in priority order, whatever the schedule.
// Colours are searched in windows of 64 (cbase); a full window defers to the next round.
// `remaining` is only a flag (non-zero iff some variable is still uncoloured).  A blocked variable
// remembers the neighbour that blocked it and looks at that one first in the next round: in the
// natural order nearly every variable is blocked for thousands of rounds, and this keeps a round at
// three coalesced loads per variable instead of a walk over its factors.
// returns true iff v is still uncoloured after this round
__device__ __forceinline__ bool jp_visit(const RawGraph &G, int64_t v, uint64_t seed, int32_t *color, int32_t *cbase,
                                         int32_t *cround, int32_t *blocker, int round, int mode)
{
    if (color[v] != -1) return false;     // already coloured
    if (G.v_evid[v] == 4) return false;   // ghosts are coloured by their owner
    {
        const int bl = blocker[v];
        if (bl >= 0) {
            int cb = ((volatile int32_t *)color)[bl];
            if (mode == 1 && cb >= 0 && ((volatile int32_t *)cround)[bl] >= round) cb = -1;
            if (cb == -1) return true;
        }
    }
    const uint64_t gv = G.gid ? (uint64_t)G.gid[v] : (uint64_t)v;
    const uint64_t pv = nb_jp_priority(gv, seed);
    const int base = cbase[v];
    uint64_t used = 0;
    bool ready = true;
    int nb = nbuckets(G, v);
    for (int b = 0; b < nb && ready; b++) {
        int64_t off = G.b_off[G.v_vtf[v] + b];
        int len = G.b_len[G.v_vtf[v] + b];
        for (int e = 0; e < len && ready; e++) {
            int f = G.fi[off + e];
            int64_t mo = G.f_off[f];
            int a = G.f_arity[f];
            for (int j = 0; j < a; j++) {
                int u = G.m_vid[mo + j];
                if (u == v) continue;
                int cu = ((volatile int32_t *)color)[u];
                if (cu == -2) continue;
                // natural-order mode counts rounds exactly (a colour taken in this round is not
                // visible before the next one), so that the round cap means the same thing on one
                // GPU and on a partitioned graph
                if (mode == 1 && cu >= 0 && ((volatile int32_t *)cround)[u] >= round) cu = -1;
                if (cu == -1) {
                    const uint64_t gu = G.gid ? (uint64_t)G.gid[u] : (uint64_t)u;
                    const bool higher = mode == 1 ? gu < gv : nb_jp_priority(gu, seed) > pv;
                    if (higher) { ready = false; blocker[v] = u; break; }
                } else if (cu >= base && cu < base + 64) {
                    used |= 1ull << (cu - base);
                }
            }
        }
    }
    if (!ready) return true;
    if (used == ~0ull) { cbase[v] = base + 64; return true; }
    if (mode == 1) { ((volatile int32_t *)cround)[v] = round; __threadfence(); }
    ((volatile int32_t *)color)[v] = base + (__ffsll((long long)~used) - 1);
    return false;
}

__global__ void __launch_bounds__(256) k_jp_round(RawGraph G, uint64_t seed, int32_t *color, int32_t *cbase, int32_t *cround,
                                                  int32_t *blocker, int round, int mode, unsigned long long *remaining)
{
    const int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const bool open = v < G.V && jp_visit(G, v, seed, color, cbase, cround, blocker, round, mode);
    // one (L1-cached) look at the flag per block: a load per thread of the same word serialises in L2
    if (__syncthreads_or(open) && threadIdx.x == 0 && *remaining == 0) *remaining = 1;
}

// single-GPU graphs ignore ghosts (-2); partitioned graphs wait for the owner's colour (-1)
__global__ void k_init_color(int64_t V, const int8_t *v_evid, int32_t *color, int32_t *cbase, int32_t *cround,
                             int32_t *blocker, int deferred)
{
    int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (v >= V) return;
    color[v] = (v_evid[v] == 4 && !deferred) ? -2 : -1;
    cbase[v] = 0;
    blocker[v] = -1;
    cround[v] = v_evid[v] == 4 ? -1 : 0x7FFFFFFF;   // ghost colours arrive between rounds: always visible
}

// conflicts = ordered pairs (v, u) of owned variables that share a factor and a colour
__global__ void k_check_coloring(RawGraph G, const int32_t *color, unsigned long long *conflicts)
{
    int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (v >= G.V || color[v] < 0) return;
    unsigned long long bad = 0;
    int nb = nbuckets(G, v);
    for (int b = 0; b < nb; b++) {
        int64_t off = G.b_off[G.v_vtf[v] + b];
        int len = G.b_len[G.v_vtf[v] + b];
        for (int e = 0; e < len; e++) {
            int f = G.fi[off + e];
            for (int j = 0; j < G.f_arity[f]; j++) {
                int u = G.m_vid[G.f_off[f] + j];
                if (u != v && color[u] == color[v]) bad++;
            }
        }
    }
    if (bad) atomicAdd(conflicts, bad);
}

// smallest GLOBAL id of the owned variables of each colour
__global__ void k_color_min_id(RawGraph G, const int32_t *color, int n_colors, unsigned long long *min_id)
{
    int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (v >= G.V || G.v_evid[v] == 4) return;
    int c = color[v];
    if (c < 0 || c >= n_colors) return;
    atomicMin(&min_id[c], (unsigned long long)(G.gid ? G.gid[v] : v));
}

__global__ void k_relabel_colors(int64_t V, int32_t *color, const int32_t *map, int n)
{
    int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (v < V && color[v] >= 0 && color[v] < n) color[v] = map[color[v]];
}

__global__ void k_max_color(int64_t V, const int32_t *color, int *maxc)
{
    int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (v < V && color[v] >= 0) atomicMax(maxc, color[v]);
}

// sort key: class(3) | colour(14) | window(27) | row length(20); ghosts use colour = n_colors
__global__ void k_sort_keys(int64_t V, const int32_t *color, const int8_t *v_evid, const uint32_t *rowlen, const uint8_t *fast, int n_colors,
                            int warp_row_words, int sigma_shift, uint64_t *keys, int32_t *ids,
                            unsigned long long *group_count, unsigned long long *color_edges,
                            const uint32_t *ninc)
{
    int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (v >= V) return;
    const bool ghost = v_evid[v] == 4 || color[v] < 0;
    int c = ghost ? n_colors : color[v];
    uint32_t len = rowlen[v];
    int cls = len > (uint32_t)warp_row_words
                  ? NB_CLASS_WARP
                  : (fast[v] == 2 ? NB_CLASS_PAIR : (fast[v] == 1 ? NB_CLASS_FAST : (fast[v] == 3 ? NB_CLASS_CAT : NB_CLASS_GEN)));
    if (ghost) cls = NB_CLASS_GEN;
    uint64_t window = ((uint64_t)v >> sigma_shift) & ((1ull << 27) - 1);
    uint64_t l = len < (1u << 20) ? len : (1u << 20) - 1;
    keys[v] = ((uint64_t)cls << 61) | ((uint64_t)c << 47) | (window << 20) | l;
    ids[v] = (int32_t)v;
    atomicAdd(&group_count[cls * (n_colors + 1) + c], 1ull);
    if (!ghost) atomicAdd(&color_edges[c], (unsigned long long)ninc[v]);
}

// sorted position -> new id, plus all per-variable arrays in the new order (T: value element type;
// vcard: cardinalities of a 2-byte graph, whose vmeta card field is 0 above 255)
template <class T>
__global__ void k_assign_ids(int64_t V, const uint64_t *keys, const int32_t *sorted_ids, int n_colors,
                             const int64_t *group_start, const int64_t *group_base, RawGraph G,
                             const int32_t *v_init, const uint32_t *rowlen, const uint8_t *fast, int32_t *old2new,
                             int32_t *new2old, uint32_t *vmeta, uint32_t *rowlen_new, T *vinit,
                             uint32_t *rng_id, T *val0, T *val1, uint16_t *vcard)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= V) return;
    uint64_t key = keys[i];
    int cls = NB_KEY_CLASS(key);
    int c = NB_KEY_COLOR(key);
    int g = cls * (n_colors + 1) + c;
    int64_t nid = group_base[g] + (i - group_start[g]);
    int v = sorted_ids[i];
    old2new[v] = (int32_t)nid;
    new2old[nid] = v;
    const int card = G.v_card[v];
    vmeta[nid] = nb_pack_meta(card <= NB_MAX_CARD ? card : 0, G.v_evid[v], G.v_dtype[v], 1, cls <= NB_CLASS_FAST, rowlen[v]);
    if (vcard) vcard[nid] = (uint16_t)card;
    rowlen_new[nid] = rowlen[v];
    T init = (T)v_init[v];
    vinit[nid] = init;
    val0[nid] = init;
    val1[nid] = init;
    rng_id[nid] = (uint32_t)(G.gid ? (uint64_t)G.gid[v] : (uint64_t)v);
}

// first new id of every (group, id-window) run of the sorted order (-1 where a window is empty)
__global__ void k_window_starts(int64_t V, const uint64_t *keys, int n_colors, const int64_t *group_start,
                                const int64_t *group_base, int64_t n_win, int32_t *win_start)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= V) return;
    const uint64_t key = keys[i];
    const int g = NB_KEY_CLASS(key) * (n_colors + 1) + NB_KEY_COLOR(key);
    const int64_t w = NB_KEY_WINDOW(key);
    if (i > 0) {
        const uint64_t prev = keys[i - 1];
        if (NB_KEY_GROUP_BITS(prev) == NB_KEY_GROUP_BITS(key) && NB_KEY_WINDOW(prev) == w) return;
    }
    win_start[(size_t)g * (size_t)(n_win + 1) + (size_t)w] = (int32_t)(group_base[g] + (i - group_start[g]));
}

template <class T>
__global__ void k_count_entries(int64_t Vn, const uint32_t *vmeta, const uint16_t *vcard, uint32_t *entries)
{
    int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (n >= Vn) return;
    uint32_t m = vmeta[n];
    int card = NbCardOf<T>(vcard).card(m, (uint32_t)n);
    entries[n] = NB_META_VALID(m) ? (card == 2 ? 1u : (uint32_t)card) : 0u;
}

__global__ void k_count_entries_old(int64_t V, const int32_t *v_card, int64_t *entries)
{
    int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (v < V) entries[v] = v_card[v] == 2 ? 1 : v_card[v];
}

// SELL-32 slice size in quads (16 B): 32 lanes x ceil(longest row / 4)
__global__ void k_slice_width(int64_t n_slices, const uint32_t *rowlen_new, int64_t *quads)
{
    int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (s >= n_slices) return;
    uint32_t w = 0;
    for (int l = 0; l < 32; l++) w = max(w, rowlen_new[s * 32 + l]);
    quads[s] = (int64_t)((w + 3) / 4) * 32;
}

__global__ void k_warp_row_sizes(int64_t n_wrows, int64_t n_trows, const uint32_t *rowlen_new,
                                 const int32_t *new2old, const uint32_t *ninc, int64_t *wlen, int64_t *winc)
{
    int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (r >= n_wrows) return;
    wlen[r] = rowlen_new[n_trows + r];
    winc[r] = ninc[new2old[n_trows + r]];
}

// Write every row's incidence stream (member ids translated to new ids).
__global__ void k_fill_rows(RawGraph G, const int32_t *old2new, int64_t n_trows, const int64_t *slice_ptr,
                            uint32_t *twords, const int64_t *wrow_ptr, uint32_t *wwords,
                            const int64_t *inc_ptr, uint2 *inc, const uint8_t *wfixed)
{
    int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (v >= G.V || G.v_evid[v] == 4) return;
    int64_t nid = old2new[v];
    uint32_t *base;
    bool quad;
    uint2 *incp = nullptr;
    if (nid < n_trows) {
        base = twords + ((slice_ptr[nid >> 5] + (nid & 31)) << 2);
        quad = true;
    } else {
        base = wwords + wrow_ptr[nid - n_trows];
        quad = false;
        incp = inc + inc_ptr[nid - n_trows];
    }
#define ROW_W(i) base[quad ? ((((i) >> 2) << 7) + ((i) & 3)) : (i)]
    int64_t pos = 0;
    int nb = nbuckets(G, v);
    const bool cat = G.v_dtype[v] == 1;
    for (int b = 0; b < nb; b++) {
        int64_t off = G.b_off[G.v_vtf[v] + b];
        int len = G.b_len[G.v_vtf[v] + b];
        if (cat && len > 0) {
            if (G.wide) { ROW_W(pos) = (uint32_t)b; ROW_W(pos + 1) = nb_pack_wide_b(C_MARK, 0, 0, 0); pos += 2; }
            else { ROW_W(pos) = nb_pack_mark_compact((uint32_t)b); pos += 1; }
        }
        for (int e = 0; e < len; e++) {
            int f = G.fi[off + e];
            int code = G.f_code[f], a = G.f_arity[f];
            uint32_t wid = (uint32_t)G.f_wid[f];
            double feat = G.f_feat[f];
            int hasfeat = feat != 1.0;
            int fixed = wfixed[wid];
            if (incp) { *incp++ = make_uint2((uint32_t)pos, (uint32_t)b); }
            if (G.wide) {
                ROW_W(pos) = wid;
                ROW_W(pos + 1) = nb_pack_wide_b(code, hasfeat, fixed, a);
                pos += 2;
            } else {
                ROW_W(pos) = nb_pack_compact(code, hasfeat, fixed, a, wid);
                pos += 1;
            }
            int64_t mo = G.f_off[f];
            bool eq = nb_code_has_eq(code);
            for (int j = 0; j < a; j++) {
                ROW_W(pos) = (uint32_t)old2new[G.m_vid[mo + j]];
                pos++;
                if (eq) { ROW_W(pos) = (uint32_t)G.m_eq[mo + j]; pos++; }
            }
            if (nb_code_has_extra(code)) {
                uint32_t x;
                if (code == C_IMPLY_MLN || code == C_IMPLY_NATURAL_CAT || code == C_IMPLY_MLN_CAT) {
                    // the reference reads var_value[fmap slot of the head] (inference.py:243,277,292)
                    int64_t slot = mo + a - 1;
                    x = (a > 0 && slot < G.V) ? (uint32_t)old2new[slot] : 0xFFFFFFFFu;
                } else {
                    int m = nb_code_abstain_member(code);
                    x = m < a ? (uint32_t)(G.v_card[G.m_vid[mo + m]] - 1) : 0u;
                }
                ROW_W(pos) = x;
                pos++;
            }
            if (hasfeat) {
                ROW_W(pos) = (uint32_t)__double2loint(feat);
                ROW_W(pos + 1) = (uint32_t)__double2hiint(feat);
                pos += 2;
            }
        }
    }
#undef ROW_W
}

// ---- truth-table stream of the FAST rows --------------------------------------------------
__global__ void k_tt_slice_width(int64_t n_slices, const int32_t *new2old, const uint32_t *ninc, int64_t *quads)
{
    int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (s >= n_slices) return;
    uint32_t w = 0;
    for (int l = 0; l < 32; l++) {
        int v = new2old[s * 32 + l];
        if (v >= 0) w = max(w, ninc[v]);
    }
    quads[s] = (int64_t)w * 32;
}

__global__ void k_tt_pad(uint4 *tt, uint32_t *base, uint32_t *wid, int64_t n)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) { tt[i] = make_uint4(0u, 0u, NB_TT_NEUTRAL | NB_TT_FIXED_BIT, 0u); base[i] = NB_TT_BASE_NEUTRAL; wid[i] = 0u; }
}

// The tables are produced by nb_tabulate (nb_eval.cuh), i.e. by nb_eval_incidence_v run on the
// variable's own generic row with the other members' values forced: one source of truth for
// factor semantics.  k_fill_rows must have run.
template <bool WIDE>
__global__ void k_fill_tt(RawGraph G, const int32_t *old2new, int64_t n_frows, const int64_t *slice_ptr,
                          const uint32_t *twords, const int64_t *tt_ptr, uint4 *tt, uint32_t *tt_base, uint32_t *tt_wid,
                          const uint8_t *wfixed, const double *weight)
{
    int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (v >= G.V || G.v_evid[v] == 4) return;
    const int64_t nid = old2new[v];
    if (nid >= n_frows) return;
    uint4 *row = tt + tt_ptr[nid >> 5] + (nid & 31);
    uint32_t *brow = tt_base + tt_ptr[nid >> 5] + (nid & 31);
    uint32_t *wrow = tt_wid + tt_ptr[nid >> 5] + (nid & 31);
    const int len = G.b_len[G.v_vtf[v]];
    const NbRow r = nb_thread_row(twords, slice_ptr, nid);
    int pos = 0;
    for (int e = 0; e < len; e++) {
        uint32_t other[2], table, base;
        const NbHdr h = nb_tabulate<WIDE>(r, pos, (uint32_t)nid, other, table, base);
        if (wfixed[h.wid]) table |= NB_TT_FIXED_BIT;
        row[(size_t)e * 32] = make_uint4(other[0], other[1], table, __float_as_uint((float)weight[h.wid]));
        brow[(size_t)e * 32] = base;
        wrow[(size_t)e * 32] = h.wid;
        pos += nb_inc_words<WIDE>(h);
    }
}

// (re)inline the current weight values into the quads
__global__ void k_tt_refresh(int64_t n, uint4 *tt, const uint32_t *tt_wid, const double *weight)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) reinterpret_cast<uint32_t *>(tt + i)[3] = __float_as_uint((float)__ldg(weight + tt_wid[i]));
}

int nb_refresh_inlined_weights(nb_graph *g)
{
    if (g->tt_weights_version == g->weights_version) return NB_OK;
    if (g->n_tt_quads)
        k_tt_refresh<<<(unsigned)((g->n_tt_quads + 255) / 256), 256, 0, g->stream>>>(g->n_tt_quads, g->d_tt, g->d_tt_wid, g->d_weight);
    if (g->n_cat_quads)
        k_tt_refresh<<<(unsigned)((g->n_cat_quads + 255) / 256), 256, 0, g->stream>>>(g->n_cat_quads, g->d_cat, g->d_cat_wid, g->d_weight);
    NB_CUDA(cudaGetLastError());
    g->tt_weights_version = g->weights_version;
    return NB_OK;
}

// ---- pair stream of the PAIR rows -----------------------------------------------------------
// second word {table:9 | fixed:1 | wid:22} of the PAIR incidence at `pos`, and its other member
template <bool WIDE>
__device__ inline uint32_t nb_pair_word(const NbRow &r, int &pos, uint32_t self, const uint8_t *wfixed, uint32_t &other)
{
    uint32_t o2[2], table, base;
    const NbHdr h = nb_tabulate<WIDE>(r, pos, self, o2, table, base);
    // only xb = 0 matters: a PAIR incidence has at most one other member (slot A)
    uint32_t t3 = 0;
    for (int x = 0; x < 3; x++) t3 |= ((table >> (3 * (3 * x))) & 7u) << (3 * x);
    other = o2[0];
    pos += nb_inc_words<WIDE>(h);
    return nb_pack_pair(t3, wfixed[h.wid], h.wid);
}

// per PAIR row: the second word shared by all its records (NB_PAIR_ANY: no record, NB_PAIR_NONE: mixed)
template <bool WIDE>
__global__ void k_tt2_row_word(RawGraph G, const int32_t *old2new, int64_t n_prows, const int64_t *slice_ptr,
                               const uint32_t *twords, const uint8_t *wfixed, uint32_t *row_word)
{
    int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (v >= G.V || G.v_evid[v] == 4) return;
    const int64_t nid = old2new[v];
    if (nid >= n_prows) return;
    const int len = G.b_len[G.v_vtf[v]];
    const NbRow r = nb_thread_row(twords, slice_ptr, nid);
    uint32_t common = NB_PAIR_ANY;
    int pos = 0;
    for (int e = 0; e < len; e++) {
        uint32_t other;
        const uint32_t w = nb_pair_word<WIDE>(r, pos, (uint32_t)nid, wfixed, other);
        if (common == NB_PAIR_ANY) common = w;
        else if (common != w) common = NB_PAIR_NONE;
    }
    row_word[nid] = common;
}

// slice width in quads and the slice's common word (NB_PAIR_NONE = two 8-byte records per quad)
__global__ void k_tt2_slice_width(int64_t n_slices, const int32_t *new2old, const uint32_t *ninc, const uint32_t *row_word,
                                  int64_t *quads, uint32_t *common_out)
{
    int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (s >= n_slices) return;
    uint32_t w = 0, common = NB_PAIR_ANY;
    for (int l = 0; l < 32; l++) {
        int v = new2old[s * 32 + l];
        if (v < 0) continue;
        w = max(w, ninc[v]);
        const uint32_t rw = row_word[s * 32 + l];
        if (rw == NB_PAIR_ANY) continue;
        if (common == NB_PAIR_ANY) common = rw;
        else if (common != rw) common = NB_PAIR_NONE;
    }
    if (common == NB_PAIR_ANY) common = NB_PAIR_NONE;
    common_out[s] = common;
    quads[s] = (common != NB_PAIR_NONE ? (int64_t)((w + 3) / 4) : (int64_t)((w + 1) / 2)) * 32;
}

__global__ void k_tt2_pad(uint4 *tt2, const int64_t *tt2_ptr, const uint32_t *common, int64_t n_slices)
{
    const int64_t s = blockIdx.x;
    if (s >= n_slices) return;
    const uint32_t w = nb_pack_pair(NB_PAIR_NEUTRAL, 1, 0u);
    const uint4 pad = common[s] != NB_PAIR_NONE ? make_uint4(NB_PAIR_NONE, NB_PAIR_NONE, NB_PAIR_NONE, NB_PAIR_NONE)
                                               : make_uint4(0u, w, 0u, w);
    for (int64_t i = tt2_ptr[s] + threadIdx.x; i < tt2_ptr[s + 1]; i += blockDim.x) tt2[i] = pad;
}

template <bool WIDE>
__global__ void k_fill_tt2(RawGraph G, const int32_t *old2new, int64_t n_prows, const int64_t *slice_ptr,
                           const uint32_t *twords, const int64_t *tt2_ptr, const uint32_t *tt2_common, uint4 *tt2,
                           const uint8_t *wfixed)
{
    int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (v >= G.V || G.v_evid[v] == 4) return;
    const int64_t nid = old2new[v];
    if (nid >= n_prows) return;
    uint4 *row = tt2 + tt2_ptr[nid >> 5] + (nid & 31);
    const bool uniform = tt2_common[nid >> 5] != NB_PAIR_NONE;
    const int len = G.b_len[G.v_vtf[v]];
    const NbRow r = nb_thread_row(twords, slice_ptr, nid);
    int pos = 0;
    for (int e = 0; e < len; e++) {
        uint32_t other;
        const uint32_t w = nb_pair_word<WIDE>(r, pos, (uint32_t)nid, wfixed, other);
        if (uniform) reinterpret_cast<uint32_t *>(row + (size_t)(e >> 2) * 32)[e & 3] = other;
        else reinterpret_cast<uint2 *>(row + (size_t)(e >> 1) * 32)[e & 1] = make_uint2(other, w);
    }
}

// ---- categorical records of the CAT rows ------------------------------------------------------
__global__ void k_cat_slice_width(int64_t n_slices, int64_t first_id, const int32_t *new2old, const uint32_t *ninc, int64_t *quads)
{
    int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (s >= n_slices) return;
    uint32_t w = 0;
    for (int l = 0; l < 32; l++) {
        int v = new2old[first_id + s * 32 + l];
        if (v >= 0) w = max(w, ninc[v]);
    }
    quads[s] = (int64_t)w * 32;
}

__global__ void k_cat_pad(uint4 *cat, uint32_t *wid, int64_t n)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) { cat[i] = make_uint4(0u, 0u, nb_pack_cat(0, 0, 0, 3, 1), 0u); wid[i] = 0u; }
}

__global__ void k_fill_cat(RawGraph G, const int32_t *old2new, int64_t first_id, int64_t end_id, const int64_t *cat_ptr,
                           uint4 *cat, uint32_t *cat_wid, const uint8_t *wfixed, const double *weight)
{
    int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (v >= G.V || G.v_evid[v] == 4) return;
    const int64_t nid = old2new[v];
    if (nid < first_id || nid >= end_id) return;
    uint4 *row = cat + cat_ptr[(nid - first_id) >> 5] + (nid & 31);
    uint32_t *wrow = cat_wid + cat_ptr[(nid - first_id) >> 5] + (nid & 31);
    int e_out = 0;
    const int card = G.v_card[v];
    for (int k = 0; k < card; k++) {
        const int64_t off = G.b_off[G.v_vtf[v] + k];
        const int len = G.b_len[G.v_vtf[v] + k];
        for (int e = 0; e < len; e++) {
            const int f = G.fi[off + e];
            const int a = G.f_arity[f];
            const int64_t mo = G.f_off[f];
            uint32_t other[2] = {(uint32_t)nid, (uint32_t)nid};
            int eq[2] = {0, 0}, n_other = 0;
            bool never = false;
            for (int j = 0; j < a; j++) {
                int u = G.m_vid[mo + j];
                if (u == v) { never |= G.m_eq[mo + j] != k; continue; }   // v forced to k must equal every one of its own slots
                if (n_other < 2) { other[n_other] = (uint32_t)old2new[u]; eq[n_other] = G.m_eq[mo + j] & 0xFF; }
                n_other++;
            }
            const uint32_t wid = (uint32_t)G.f_wid[f];
            row[(size_t)e_out * 32] = make_uint4(other[0], other[1], nb_pack_cat(k, eq[0], eq[1], never ? 3 : n_other, wfixed[wid]),
                                                 __float_as_uint((float)weight[wid]));
            wrow[(size_t)e_out * 32] = wid;
            e_out++;
        }
    }
}

// ---------------------------------------------------------------------------
// host driver
// ---------------------------------------------------------------------------
static RawGraph raw_view(const nb_graph *g)
{
    RawGraph G;
    G.V = g->V;
    G.v_evid = g->d_v_evid; G.v_card = g->d_v_card; G.v_dtype = g->d_v_dtype; G.v_vtf = g->d_v_vtf;
    G.b_off = g->d_b_off; G.b_len = g->d_b_len; G.fi = g->d_fi;
    G.f_code = g->d_f_code; G.f_wid = g->d_f_wid; G.f_feat = g->d_f_feat; G.f_arity = g->d_f_arity;
    G.f_off = g->d_f_off; G.m_vid = g->d_m_vid; G.m_eq = g->d_m_eq; G.gid = g->d_gid; G.wide = g->wide;
    G.val16 = g->value_bytes == 2;
    return G;
}

static inline unsigned grid_for(int64_t n, int block = 256) { return (unsigned)std::max<int64_t>(1, (n + block - 1) / block); }

template <class T>
static int exclusive_scan(nb_graph *g, const T *in, T *out, int64_t n)
{
    size_t tmp = 0;
    NB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp, in, out, n, g->stream));
    NB_TRY(nb_ensure_xfer(g, tmp));
    NB_CUDA(cub::DeviceScan::ExclusiveSum(g->d_xfer, tmp, in, out, n, g->stream));
    return NB_OK;
}

static int extract_and_upload(nb_graph *g, const nb_graph_desc *d)
{
    const int64_t V = d->n_variable, F = d->n_factor, W = d->n_weight;
    const int64_t NF = d->n_fmap, NV = d->n_vmap, NFI = d->n_factor_index;
    if (V < 0 || F < 0 || W < 0 || NF < 0 || NV < 0 || NFI < 0) NB_FAIL(NB_ERR_INVALID, "negative array length");
    if (V >= (1ll << 31) - 64 || F >= (1ll << 31) || W >= (1ll << 31))
        NB_FAIL(NB_ERR_UNSUPPORTED, "variables/factors/weights must stay below 2^31 per GPU (partition the graph)");
    g->V = V; g->F = F; g->W = W; g->NFMAP = NF; g->NVMAP = NV; g->NFI = NFI;

    std::atomic<int> bad(0);
    std::atomic<int> maxcard(1), maxarity(0), anycat(0);
    std::atomic<int64_t> unknown(-1);
    char msg[256] = "";
    auto fail = [&](const char *what, int64_t idx) {
        int expected = 0;
        if (bad.compare_exchange_strong(expected, 1)) snprintf(msg, sizeof(msg), "%s (index %lld)", what, (long long)idx);
    };

    // Each section is validated, narrowed into SoA columns by host threads, uploaded and
    // freed before the next one starts, so the host peak stays at one section.
    // ---- variables ----
    {
        std::vector<int8_t> v_evid(V), v_dtype(V);
        std::vector<int32_t> v_card(V), v_init(V);
        std::vector<int64_t> v_vtf(V);
        parallel_for(V, [&](int64_t a, int64_t b) {
            int mc = 1, cat = 0;
            for (int64_t i = a; i < b; i++) {
                const nb_variable_rec &r = d->variable[i];
                if (r.dataType != 0 && r.dataType != 1) { fail("variable dataType must be 0 or 1", i); continue; }
                if (r.cardinality < 1 || r.cardinality > NB_MAX_CARD_WIDE) { fail("variable cardinality outside [1, 65535]", i); continue; }
                // the reference accepts such graphs: a sampled variable's value is overwritten at its first
                // sample (load_domains can leave a raw initialValue that is not in the domain)
                const bool init_ok = r.initialValue >= 0 && r.initialValue < r.cardinality;
                if (!init_ok && r.isEvidence == 1) { fail("evidence variable with initialValue outside [0, cardinality)", i); continue; }
                int64_t nb = r.dataType == 0 ? 1 : r.cardinality;
                if (r.vtf_offset < 0 || r.vtf_offset + nb > NV) { fail("variable vtf_offset out of range", i); continue; }
                v_evid[i] = r.isEvidence; v_dtype[i] = (int8_t)r.dataType;
                v_card[i] = (int32_t)r.cardinality; v_init[i] = init_ok ? (int32_t)r.initialValue : 0; v_vtf[i] = r.vtf_offset;
                mc = std::max(mc, (int)r.cardinality);
                cat |= r.dataType == 1;
            }
            int cur = maxcard.load();
            while (mc > cur && !maxcard.compare_exchange_weak(cur, mc)) {}
            if (cat) anycat.store(1);
        });
        if (bad.load()) NB_FAIL(NB_ERR_INVALID, "invalid factor graph: %s", msg);
        NB_TRY(upload(g, &g->d_v_evid, v_evid));
        NB_TRY(upload(g, &g->d_v_dtype, v_dtype));
        NB_TRY(upload(g, &g->d_v_card, v_card));
        NB_TRY(upload(g, &g->d_v_init, v_init));
        NB_TRY(upload(g, &g->d_v_vtf, v_vtf));
    }
    // ---- buckets ----
    std::atomic<int64_t> edges(0);
    {
        std::vector<int64_t> b_off(NV);
        std::vector<int32_t> b_len(NV);
        parallel_for(NV, [&](int64_t a, int64_t b) {
            int64_t sum = 0;
            for (int64_t i = a; i < b; i++) {
                const nb_vtf_rec &r = d->vmap[i];
                if (r.factor_index_length < 0 || r.factor_index_offset < 0 ||
                    r.factor_index_offset + r.factor_index_length > NFI || r.factor_index_length > 0x7FFFFFFF) {
                    fail("vmap bucket outside factor_index", i);
                    continue;
                }
                b_off[i] = r.factor_index_offset;
                b_len[i] = (int32_t)r.factor_index_length;
                sum += r.factor_index_length;
            }
            edges += sum;
        });
        if (bad.load()) NB_FAIL(NB_ERR_INVALID, "invalid factor graph: %s", msg);
        NB_TRY(upload(g, &g->d_b_off, b_off));
        NB_TRY(upload(g, &g->d_b_len, b_len));
    }
    {
        std::vector<int32_t> fi(NFI);
        parallel_for(NFI, [&](int64_t a, int64_t b) {
            for (int64_t i = a; i < b; i++) {
                int64_t f = d->factor_index[i];
                // entries beyond a bucket's de-duplicated length are scratch; clamp instead of failing
                fi[i] = (f >= 0 && f < F) ? (int32_t)f : 0;
            }
        });
        NB_TRY(upload(g, &g->d_fi, fi));
    }
    // ---- factors ----
    {
        std::vector<uint8_t> f_code(F);
        std::vector<int32_t> f_wid(F), f_arity(F);
        std::vector<double> f_feat(F);
        std::vector<int64_t> f_off(F);
        parallel_for(F, [&](int64_t a, int64_t b) {
            int ma = 0, cat = 0;
            for (int64_t i = a; i < b; i++) {
                const nb_factor_rec &r = d->factor[i];
                int code = nb_code_of_func(r.factorFunction);
                if (code == C_UNKNOWN) {
                    int64_t cur = unknown.load();
                    while ((cur < 0 || i < cur) && !unknown.compare_exchange_weak(cur, i)) {}
                }
                if (r.weightId < 0 || r.weightId >= W) { fail("factor weightId out of range", i); continue; }
                if (r.arity < 0 || r.arity >= (1 << 24) || r.ftv_offset < 0 || r.ftv_offset + r.arity > NF) { fail("factor fmap range out of bounds", i); continue; }
                f_code[i] = (uint8_t)code; f_wid[i] = (int32_t)r.weightId; f_arity[i] = (int32_t)r.arity;
                f_feat[i] = r.featureValue; f_off[i] = r.ftv_offset;
                ma = std::max(ma, (int)r.arity);
                cat |= nb_code_has_eq(code);
            }
            int cur = maxarity.load();
            while (ma > cur && !maxarity.compare_exchange_weak(cur, ma)) {}
            if (cat) anycat.store(1);
        });
        if (bad.load()) NB_FAIL(NB_ERR_INVALID, "invalid factor graph: %s", msg);
        NB_TRY(upload(g, &g->d_f_code, f_code));
        NB_TRY(upload(g, &g->d_f_wid, f_wid));
        NB_TRY(upload(g, &g->d_f_arity, f_arity));
        NB_TRY(upload(g, &g->d_f_feat, f_feat));
        NB_TRY(upload(g, &g->d_f_off, f_off));
    }
    // ---- members ----
    const bool need_eq = anycat.load() != 0;
    {
        std::vector<int32_t> m_vid(NF), m_eq;
        if (need_eq) m_eq.resize(NF);
        parallel_for(NF, [&](int64_t a, int64_t b) {
            for (int64_t i = a; i < b; i++) {
                const nb_ftv_rec &r = d->fmap[i];
                if (r.vid < 0 || r.vid >= V) { fail("fmap vid out of range", i); continue; }
                m_vid[i] = (int32_t)r.vid;
                if (need_eq) m_eq[i] = (int32_t)std::min<int64_t>(std::max<int64_t>(r.dense_equal_to, -1), 0x7FFFFFFF);
            }
        });
        if (bad.load()) NB_FAIL(NB_ERR_INVALID, "invalid factor graph: %s", msg);
        NB_TRY(upload(g, &g->d_m_vid, m_vid));
        if (need_eq) NB_TRY(upload(g, &g->d_m_eq, m_eq));
    }

    g->n_edges = edges.load();
    g->max_card = maxcard.load();
    g->value_bytes = g->max_card > NB_MAX_CARD ? 2 : 1;   // 1-byte values unless some cardinality needs 2
    g->max_arity = maxarity.load();
    g->any_categorical = need_eq;
    g->wide = (W > (int64_t)NB_COMPACT_MAX_WID + 1) || (maxarity.load() > NB_COMPACT_MAX_ARITY);
    if (unknown.load() >= 0) {
        g->has_unknown_func = true;
        g->unknown_func_factor = unknown.load();
        g->unknown_func_id = d->factor[unknown.load()].factorFunction;
    }
    if (d->global_vid) {
        std::vector<int64_t> gid(d->global_vid, d->global_vid + V);
        NB_TRY(upload(g, &g->d_gid, gid));
    }
    // weights
    std::vector<double> w(W);
    std::vector<uint8_t> wf(W);
    for (int64_t i = 0; i < W; i++) { w[i] = d->weight[i].initialValue; wf[i] = d->weight[i].isFixed ? 1 : 0; }
    NB_TRY(upload(g, &g->d_weight, w));
    NB_TRY(upload(g, &g->d_wfixed, wf));
    return NB_OK;
}

void nb_release_color_scratch(nb_graph *g)
{
    if (g->d_cbase) cudaFree(g->d_cbase);
    g->d_cbase = g->d_cround = g->d_blocker = nullptr;
}

// n_rounds (<= NB_JP_BATCH) rounds back to back, one host round trip; *remaining is the flag of the
// last one.  Rounds after the last variable took its colour change nothing.
#define NB_JP_BATCH 8
static int color_rounds(nb_graph *g, int n_rounds, int64_t *remaining)
{
    if (!g->d_cbase) NB_FAIL(NB_ERR_INVALID, "the graph is already coloured");
    RawGraph G = raw_view(g);
    NB_CUDA(cudaMemsetAsync(g->d_jpcnt, 0, 8 * NB_JP_BATCH, g->stream));
    for (int i = 0; i < n_rounds; i++) {
        k_jp_round<<<grid_for(g->V), 256, 0, g->stream>>>(G, g->color_seed, g->d_color, g->d_cbase, g->d_cround, g->d_blocker,
                                                          g->jp_round_no, g->jp_mode, g->d_jpcnt + i);
        g->jp_rounds++;
        g->jp_round_no++;
    }
    unsigned long long rem = 0;
    NB_CUDA(cudaMemcpyAsync(&rem, g->d_jpcnt + (n_rounds - 1), 8, cudaMemcpyDeviceToHost, g->stream));
    NB_CUDA(cudaStreamSynchronize(g->stream));
    *remaining = (int64_t)rem;
    return NB_OK;
}

int nb_build_color_round(nb_graph *g, int64_t *remaining) { return color_rounds(g, 1, remaining); }

// (re)start the colouring: mode 0 = hashed priorities (few rounds), 1 = natural order (smaller
// global id first: the sequential greedy colouring in id order; 2 colours on grids and other
// bipartite structured graphs, but as many rounds as the longest increasing-id path)
int nb_build_color_restart(nb_graph *g, int mode)
{
    if (g->finalized) NB_FAIL(NB_ERR_INVALID, "graph already finalized");
    g->jp_mode = mode;
    g->jp_round_no = 0;
    k_init_color<<<grid_for(g->V), 256, 0, g->stream>>>(g->V, g->d_v_evid, g->d_color, g->d_cbase, g->d_cround,
                                                        g->d_blocker, g->deferred ? 1 : 0);
    NB_CUDA(cudaGetLastError());
    return NB_OK;
}

static int count_colors(nb_graph *g, int *n_colors)
{
    int *d_max;
    NB_CUDA(cudaMalloc(&d_max, 4));
    cudaMemsetAsync(d_max, 0xFF, 4, g->stream);  // -1
    k_max_color<<<grid_for(g->V), 256, 0, g->stream>>>(g->V, g->d_color, d_max);
    int maxc = -1;
    cudaMemcpyAsync(&maxc, d_max, 4, cudaMemcpyDeviceToHost, g->stream);
    cudaError_t e = cudaStreamSynchronize(g->stream);
    cudaFree(d_max);
    NB_CUDA(e);
    *n_colors = maxc + 1;
    return NB_OK;
}

int nb_natural_round_cap(void)
{
    const char *env = getenv("NUMBSKULL_B200_NATURAL_ROUNDS");
    return env ? atoi(env) : 65536;
}

static int run_jp(nb_graph *g, int mode, int64_t cap, bool *finished)
{
    NB_TRY(nb_build_color_restart(g, mode));
    *finished = false;
    for (int64_t r = 0; cap <= 0 || r < cap;) {
        // the natural order needs thousands of cheap rounds: look at the flag once per batch
        const int n = (int)std::min<int64_t>(mode == 1 ? NB_JP_BATCH : 1, cap <= 0 ? NB_JP_BATCH : cap - r);
        int64_t rem = 0;
        NB_TRY(color_rounds(g, n, &rem));
        r += n;
        if (rem == 0) { *finished = true; break; }
        if (r > 4000000) NB_FAIL(NB_ERR_CUDA, "Jones-Plassmann colouring did not converge");
    }
    return NB_OK;
}

static int color_graph(nb_graph *g, const nb_graph_desc *d)
{
    const int64_t V = g->V;
    RawGraph G = raw_view(g);
    NB_TRY(nb_alloc(g, &g->d_color, (size_t)V, false));
    NB_TRY(nb_alloc(g, &g->d_jpcnt, 2 * NB_JP_BATCH));
    // colouring scratch (released by nb_build_finalize): colour window, round stamp, last blocker
    NB_CUDA(cudaMalloc(&g->d_cbase, (size_t)std::max<int64_t>(V, 1) * 12));
    g->d_cround = g->d_cbase + std::max<int64_t>(V, 1);
    g->d_blocker = g->d_cround + std::max<int64_t>(V, 1);
    g->color_seed = d->color_seed;
    if (d->preset_color) {
        NB_CUDA(cudaMemcpyAsync(g->d_color, d->preset_color, (size_t)V * 4, cudaMemcpyHostToDevice, g->stream));
        k_check_coloring<<<grid_for(V), 256, 0, g->stream>>>(G, g->d_color, g->d_jpcnt);
        unsigned long long bad = 0;
        NB_CUDA(cudaMemcpyAsync(&bad, g->d_jpcnt, 8, cudaMemcpyDeviceToHost, g->stream));
        NB_CUDA(cudaStreamSynchronize(g->stream));
        if (bad) NB_FAIL(NB_ERR_INVALID, "preset colouring has %llu conflicts", bad);
        return NB_OK;
    }
    if (g->deferred) return nb_build_color_restart(g, 0);   // the caller drives nb_color_round + the ghost exchange
    // hashed priorities first (a dozen rounds); if that needs more than two colours, try the
    // natural order under a round cap and keep whichever colouring is smaller
    bool done = false;
    NB_TRY(run_jp(g, 0, 0, &done));
    int nc_hash = 0;
    NB_TRY(count_colors(g, &nc_hash));
    // (a factor with three or more members is a clique of the conflict graph: the natural order
    // then needs as many rounds as the longest increasing-id path and gains little -- not tried)
    const int cap = nb_natural_round_cap();
    if (nc_hash > 2 && cap > 0 && g->max_arity <= 2) {
        int32_t *d_saved;
        NB_CUDA(cudaMalloc(&d_saved, (size_t)std::max<int64_t>(V, 1) * 4));
        cudaMemcpyAsync(d_saved, g->d_color, (size_t)V * 4, cudaMemcpyDeviceToDevice, g->stream);
        int rc = run_jp(g, 1, cap, &done);
        int nc_nat = 0;
        if (rc == NB_OK && done) rc = count_colors(g, &nc_nat);
        if (rc != NB_OK || !done || nc_nat >= nc_hash) {
            cudaMemcpyAsync(g->d_color, d_saved, (size_t)V * 4, cudaMemcpyDeviceToDevice, g->stream);
            g->jp_mode = 0;
        }
        cudaStreamSynchronize(g->stream);
        cudaFree(d_saved);
        NB_TRY(rc);
    }
    return NB_OK;
}

// Colours are visited in increasing order of the smallest (global) variable id they contain:
// the chromatic analogue of the reference's ascending-id scan (inference.py:16-20,
// learning.py:20-23).  It matters for learning, whose first sweep otherwise computes a whole
// colour's gradients against neighbours that still hold their initial values.
int nb_build_color_min_ids(nb_graph *g, int n_colors, int64_t *min_ids)
{
    if (n_colors <= 0) return NB_OK;
    unsigned long long *d_min;
    NB_CUDA(cudaMalloc(&d_min, (size_t)n_colors * 8));
    cudaMemsetAsync(d_min, 0xFF, (size_t)n_colors * 8, g->stream);
    k_color_min_id<<<grid_for(g->V), 256, 0, g->stream>>>(raw_view(g), g->d_color, n_colors, d_min);
    std::vector<unsigned long long> h((size_t)n_colors);
    cudaMemcpyAsync(h.data(), d_min, (size_t)n_colors * 8, cudaMemcpyDeviceToHost, g->stream);
    cudaError_t e = cudaStreamSynchronize(g->stream);
    cudaFree(d_min);
    NB_CUDA(e);
    for (int c = 0; c < n_colors; c++) min_ids[c] = h[(size_t)c] > 0x7FFFFFFFFFFFFFFFull ? INT64_MAX : (int64_t)h[(size_t)c];
    return NB_OK;
}

int nb_build_relabel_colors(nb_graph *g, const int32_t *map, int n)
{
    if (g->finalized) NB_FAIL(NB_ERR_INVALID, "colours cannot be relabelled after nb_graph_finalize");
    if (n <= 0) return NB_OK;
    int32_t *d_map;
    NB_CUDA(cudaMalloc(&d_map, (size_t)n * 4));
    cudaMemcpyAsync(d_map, map, (size_t)n * 4, cudaMemcpyHostToDevice, g->stream);
    k_relabel_colors<<<grid_for(g->V), 256, 0, g->stream>>>(g->V, g->d_color, d_map, n);
    cudaError_t e = cudaStreamSynchronize(g->stream);
    cudaFree(d_map);
    NB_CUDA(e);
    return NB_OK;
}

static int order_colors_by_min_id(nb_graph *g, int n_colors)
{
    std::vector<int64_t> mins((size_t)n_colors);
    NB_TRY(nb_build_color_min_ids(g, n_colors, mins.data()));
    std::vector<int32_t> order((size_t)n_colors), map((size_t)n_colors);
    for (int c = 0; c < n_colors; c++) order[(size_t)c] = c;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return mins[(size_t)a] < mins[(size_t)b]; });
    for (int i = 0; i < n_colors; i++) map[(size_t)order[(size_t)i]] = i;
    return nb_build_relabel_colors(g, map.data(), n_colors);
}

int nb_build_device_graph(nb_graph *g, const nb_graph_desc *d)
{
    // thread rows take their length from the 17-bit vmeta field: anything longer must be a warp row
    if (d->warp_row_words > 0) g->warp_row_words = (int)std::min<uint32_t>((uint32_t)d->warp_row_words, NB_META_MAX_ROWLEN);
    g->deferred = d->deferred_coloring != 0;
    NB_TRY(extract_and_upload(g, d));
    if (d->sigma_shift > 0) g->sigma_shift = d->sigma_shift;
    else {
        // id windows: 4096 ids on large graphs (gather locality of the SELL order), finer on small ones so
        // that learning still has ~1000 windows to cut its mini-batches from
        int lg = 0;
        while ((1ll << (lg + 1)) <= std::max<int64_t>(g->V, 1)) lg++;
        g->sigma_shift = std::min(12, std::max(5, lg - 10));
    }
    const int64_t V = g->V;
    RawGraph G = raw_view(g);

    // ---- row sizes ----
    int *d_overflow;
    NB_TRY(nb_alloc(g, &g->d_rowlen0, (size_t)V));
    NB_TRY(nb_alloc(g, &g->d_ninc0, (size_t)V));
    NB_TRY(nb_alloc(g, &g->d_fast0, (size_t)V));
    NB_TRY(nb_alloc(g, &d_overflow, 1));
    k_row_size<<<grid_for(V), 256, 0, g->stream>>>(G, g->d_rowlen0, g->d_ninc0, g->d_fast0, d_overflow);
    int overflow = 0;
    NB_CUDA(cudaMemcpyAsync(&overflow, d_overflow, 4, cudaMemcpyDeviceToHost, g->stream));
    NB_CUDA(cudaStreamSynchronize(g->stream));
    if (overflow) NB_FAIL(NB_ERR_UNSUPPORTED, "a variable's incidence row exceeds 2^31 words");

    // ---- colouring ----
    NB_TRY(color_graph(g, d));
    if (g->deferred) return NB_OK;
    return nb_build_finalize(g);
}

int nb_build_finalize(nb_graph *g)
{
    if (g->finalized) return NB_OK;
    const int64_t V = g->V;
    RawGraph G = raw_view(g);
    uint32_t *d_rowlen = g->d_rowlen0, *d_ninc = g->d_ninc0;
    uint8_t *d_fast = g->d_fast0;
    {
        int *d_max;
        NB_TRY(nb_alloc(g, &d_max, 1));
        NB_CUDA(cudaMemsetAsync(d_max, 0xFF, 4, g->stream));  // -1
        k_max_color<<<grid_for(V), 256, 0, g->stream>>>(V, g->d_color, d_max);
        int maxc = -1;
        NB_CUDA(cudaMemcpyAsync(&maxc, d_max, 4, cudaMemcpyDeviceToHost, g->stream));
        NB_CUDA(cudaStreamSynchronize(g->stream));
        g->n_colors = maxc + 1;
    }
    if (!g->deferred) NB_TRY(order_colors_by_min_id(g, g->n_colors));   // partitioned graphs: done by the caller, globally
    const int nc = g->n_colors, ng = NB_N_CLASSES * (nc + 1);
    if (nc >= 0x3FFF) NB_FAIL(NB_ERR_UNSUPPORTED, "colouring needs %d colours (limit 16382)", nc);

    // ---- ordering ----
    uint64_t *d_keys, *d_keys_sorted;
    int32_t *d_ids, *d_ids_sorted;
    unsigned long long *d_group_count, *d_color_edges;
    NB_TRY(nb_alloc(g, &d_keys, (size_t)V, false));
    NB_TRY(nb_alloc(g, &d_keys_sorted, (size_t)V, false));
    NB_TRY(nb_alloc(g, &d_ids, (size_t)V, false));
    NB_TRY(nb_alloc(g, &d_ids_sorted, (size_t)V, false));
    NB_TRY(nb_alloc(g, &d_group_count, (size_t)ng));
    NB_TRY(nb_alloc(g, &d_color_edges, (size_t)nc + 1));
    k_sort_keys<<<grid_for(V), 256, 0, g->stream>>>(V, g->d_color, g->d_v_evid, d_rowlen, d_fast, nc, g->warp_row_words, g->sigma_shift,
                                                    d_keys, d_ids, d_group_count, d_color_edges, d_ninc);
    {
        size_t tmp = 0;
        NB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp, d_keys, d_keys_sorted, d_ids, d_ids_sorted, V, 0, 64, g->stream));
        NB_TRY(nb_ensure_xfer(g, tmp));
        NB_CUDA(cub::DeviceRadixSort::SortPairs(g->d_xfer, tmp, d_keys, d_keys_sorted, d_ids, d_ids_sorted, V, 0, 64, g->stream));
    }
    std::vector<unsigned long long> gcount((size_t)ng), cedges((size_t)nc + 1);
    NB_CUDA(cudaMemcpyAsync(gcount.data(), d_group_count, (size_t)ng * 8, cudaMemcpyDeviceToHost, g->stream));
    NB_CUDA(cudaMemcpyAsync(cedges.data(), d_color_edges, ((size_t)nc + 1) * 8, cudaMemcpyDeviceToHost, g->stream));
    NB_CUDA(cudaStreamSynchronize(g->stream));

    // groups in sorted order: PAIR, FAST, CAT, GEN (colours 0..nc each, nc = ghosts), then WARP
    std::vector<int64_t> gstart((size_t)ng), gbase((size_t)ng);
    g->colors.assign((size_t)nc, NbColorRange());
    int64_t pos = 0, nid = 0;
    for (int cls = 0; cls < NB_CLASS_WARP; cls++) {
        for (int c = 0; c <= nc; c++) {
            size_t gi = (size_t)(cls * (nc + 1) + c);
            gstart[gi] = pos;
            nid = (nid + 31) & ~31ll;
            gbase[gi] = nid;
            if (c < nc) {
                NbColorRange &cr = g->colors[(size_t)c];
                int32_t b = (int32_t)nid, e = (int32_t)(nid + (int64_t)gcount[gi]);
                if (cls == NB_CLASS_PAIR) { cr.p_beg = b; cr.p_end = e; }
                else if (cls == NB_CLASS_FAST) { cr.f_beg = b; cr.f_end = e; }
                else if (cls == NB_CLASS_CAT) { cr.c_beg = b; cr.c_end = e; }
                else { cr.t_beg = b; cr.t_end = e; }
            }
            pos += (int64_t)gcount[gi];
            nid += (int64_t)gcount[gi];
        }
        if (cls == NB_CLASS_PAIR) { nid = (nid + 31) & ~31ll; g->n_prows = nid; }
        if (cls == NB_CLASS_FAST) { nid = (nid + 31) & ~31ll; g->n_frows = nid; }
        if (cls == NB_CLASS_CAT) { nid = (nid + 31) & ~31ll; g->n_crows = nid; }
    }
    g->n_trows = (nid + 31) & ~31ll;
    int64_t wr = 0;
    for (int c = 0; c <= nc; c++) {
        size_t gi = (size_t)(NB_CLASS_WARP * (nc + 1) + c);
        gstart[gi] = pos;
        gbase[gi] = g->n_trows + wr;
        if (c < nc) { g->colors[(size_t)c].w_beg = (int32_t)wr; g->colors[(size_t)c].w_end = (int32_t)(wr + (int64_t)gcount[gi]); g->colors[(size_t)c].edges = (int64_t)cedges[(size_t)c]; }
        pos += (int64_t)gcount[gi];
        wr += (int64_t)gcount[gi];
    }
    g->n_wrows = wr;
    g->Vn = g->n_trows + g->n_wrows;
    if (g->Vn >= (1ll << 31)) NB_FAIL(NB_ERR_UNSUPPORTED, "padded variable id space exceeds 2^31");
    const int64_t Vn = g->Vn;

    int64_t *d_gstart, *d_gbase;
    NB_TRY(upload(g, &d_gstart, gstart));
    NB_TRY(upload(g, &d_gbase, gbase));
    NB_TRY(nb_alloc(g, &g->d_old2new, (size_t)V, false));
    NB_TRY(nb_alloc(g, &g->d_new2old, (size_t)Vn, false));
    NB_CUDA(cudaMemsetAsync(g->d_new2old, 0xFF, (size_t)Vn * 4, g->stream));
    NB_TRY(nb_alloc(g, &g->d_vmeta, (size_t)Vn));
    uint32_t *d_rowlen_new;
    NB_TRY(nb_alloc(g, &d_rowlen_new, (size_t)Vn));
    NB_TRY(nb_dev_alloc(g, &g->d_vinit, (size_t)Vn * g->value_bytes, true));
    NB_TRY(nb_alloc(g, &g->d_rng_id, (size_t)Vn));
    // both chains in one allocation, val_stride elements apart (d_val[1] is not an allocation of its own)
    g->val_stride = ((size_t)Vn + 255) & ~(size_t)255;
    NB_TRY(nb_dev_alloc(g, &g->d_val[0], 2 * g->val_stride * g->value_bytes, true));
    g->d_val[1] = (char *)g->d_val[0] + g->val_stride * g->value_bytes;
    if (g->value_bytes == 1) {
        k_assign_ids<<<grid_for(V), 256, 0, g->stream>>>(V, d_keys_sorted, d_ids_sorted, nc, d_gstart, d_gbase, G,
                                                         g->d_v_init, d_rowlen, d_fast, g->d_old2new, g->d_new2old, g->d_vmeta,
                                                         d_rowlen_new, (nb_val_t *)g->d_vinit, g->d_rng_id, nb_vals<nb_val_t>(g, 0),
                                                         nb_vals<nb_val_t>(g, 1), (uint16_t *)nullptr);
    } else {
        NB_TRY(nb_alloc(g, &g->d_vcard, (size_t)Vn));
        k_assign_ids<<<grid_for(V), 256, 0, g->stream>>>(V, d_keys_sorted, d_ids_sorted, nc, d_gstart, d_gbase, G,
                                                         g->d_v_init, d_rowlen, d_fast, g->d_old2new, g->d_new2old, g->d_vmeta,
                                                         d_rowlen_new, (nb_val16_t *)g->d_vinit, g->d_rng_id,
                                                         nb_vals<nb_val16_t>(g, 0), nb_vals<nb_val16_t>(g, 1), g->d_vcard);
    }

    // ---- id windows of every (class, colour) group: learning walks the graph window by window ----
    {
        g->n_win = (V >> g->sigma_shift) + 1;
        const size_t row = (size_t)g->n_win + 1, total = (size_t)ng * row;
        int32_t *d_ws;
        NB_TRY(nb_alloc(g, &d_ws, total, false));
        NB_CUDA(cudaMemsetAsync(d_ws, 0xFF, total * 4, g->stream));
        k_window_starts<<<grid_for(V), 256, 0, g->stream>>>(V, d_keys_sorted, nc, d_gstart, d_gbase, g->n_win, d_ws);
        g->win_start.assign(total, -1);
        NB_CUDA(cudaMemcpyAsync(g->win_start.data(), d_ws, total * 4, cudaMemcpyDeviceToHost, g->stream));
        NB_CUDA(cudaStreamSynchronize(g->stream));
        for (int gi = 0; gi < ng; gi++) {
            int32_t *ws = g->win_start.data() + (size_t)gi * row;
            // end of the group in its own id space (thread classes: new ids; warp class: new ids too)
            ws[g->n_win] = (int32_t)(gbase[(size_t)gi] + (int64_t)gcount[(size_t)gi]);
            for (int64_t w = g->n_win - 1; w >= 0; w--) if (ws[w] < 0) ws[w] = ws[w + 1];
        }
        // the filled-in table goes back to the device for the persistent learning kernel
        NB_CUDA(cudaMemcpyAsync(d_ws, g->win_start.data(), total * 4, cudaMemcpyHostToDevice, g->stream));
        g->d_win_start = d_ws;
    }

    // ---- count layouts ----
    {
        uint32_t *d_entries;
        NB_TRY(nb_alloc(g, &d_entries, (size_t)Vn + 1));
        NB_TRY(nb_alloc(g, &g->d_cstart, (size_t)Vn + 1));
        if (g->value_bytes == 1) k_count_entries<nb_val_t><<<grid_for(Vn), 256, 0, g->stream>>>(Vn, g->d_vmeta, nullptr, d_entries);
        else k_count_entries<nb_val16_t><<<grid_for(Vn), 256, 0, g->stream>>>(Vn, g->d_vmeta, g->d_vcard, d_entries);
        NB_TRY(exclusive_scan(g, d_entries, g->d_cstart, Vn + 1));
        int64_t *d_entries_old;
        NB_TRY(nb_alloc(g, &d_entries_old, (size_t)V + 1));
        NB_TRY(nb_alloc(g, &g->d_cstart_old, (size_t)V + 1));
        k_count_entries_old<<<grid_for(V), 256, 0, g->stream>>>(V, g->d_v_card, d_entries_old);
        NB_TRY(exclusive_scan(g, d_entries_old, g->d_cstart_old, V + 1));
        int64_t total = 0;
        uint32_t total_new = 0;
        NB_CUDA(cudaMemcpyAsync(&total, g->d_cstart_old + V, 8, cudaMemcpyDeviceToHost, g->stream));
        NB_CUDA(cudaMemcpyAsync(&total_new, g->d_cstart + Vn, 4, cudaMemcpyDeviceToHost, g->stream));
        NB_CUDA(cudaStreamSynchronize(g->stream));
        if (total >= (1ll << 32) - 1 || total != (int64_t)total_new)
            NB_FAIL(NB_ERR_UNSUPPORTED, "count array of %lld entries unsupported (new layout %u)", (long long)total, total_new);
        g->count_entries = total;
        NB_TRY(nb_alloc(g, &g->d_count, (size_t)total));
        NB_TRY(nb_alloc(g, &g->d_count_b, (size_t)Vn));
    }

    // ---- SELL-32 slices (thread path) ----
    const int64_t n_slices = g->n_trows / 32;
    {
        int64_t *d_width;
        NB_TRY(nb_alloc(g, &d_width, (size_t)n_slices + 1));
        NB_TRY(nb_alloc(g, &g->d_slice_ptr, (size_t)n_slices + 1));
        if (n_slices) k_slice_width<<<grid_for(n_slices), 256, 0, g->stream>>>(n_slices, d_rowlen_new, d_width);
        NB_TRY(exclusive_scan(g, d_width, g->d_slice_ptr, n_slices + 1));
        int64_t n_quads = 0;
        NB_CUDA(cudaMemcpyAsync(&n_quads, g->d_slice_ptr + n_slices, 8, cudaMemcpyDeviceToHost, g->stream));
        NB_CUDA(cudaStreamSynchronize(g->stream));
        g->n_twords = n_quads * 4;
        NB_TRY(nb_alloc(g, &g->d_twords, (size_t)g->n_twords + 4));
    }
    // ---- contiguous rows (warp path) ----
    {
        const int64_t nw = g->n_wrows;
        int64_t *d_wlen, *d_winc;
        NB_TRY(nb_alloc(g, &d_wlen, (size_t)nw + 1));
        NB_TRY(nb_alloc(g, &d_winc, (size_t)nw + 1));
        NB_TRY(nb_alloc(g, &g->d_wrow_ptr, (size_t)nw + 1));
        NB_TRY(nb_alloc(g, &g->d_inc_ptr, (size_t)nw + 1));
        if (nw) k_warp_row_sizes<<<grid_for(nw), 256, 0, g->stream>>>(nw, g->n_trows, d_rowlen_new, g->d_new2old, d_ninc, d_wlen, d_winc);
        NB_TRY(exclusive_scan(g, d_wlen, g->d_wrow_ptr, nw + 1));
        NB_TRY(exclusive_scan(g, d_winc, g->d_inc_ptr, nw + 1));
        NB_CUDA(cudaMemcpyAsync(&g->n_wwords, g->d_wrow_ptr + nw, 8, cudaMemcpyDeviceToHost, g->stream));
        NB_CUDA(cudaMemcpyAsync(&g->n_inc, g->d_inc_ptr + nw, 8, cudaMemcpyDeviceToHost, g->stream));
        NB_CUDA(cudaStreamSynchronize(g->stream));
        NB_TRY(nb_alloc(g, &g->d_wwords, (size_t)g->n_wwords));
        NB_TRY(nb_alloc(g, &g->d_inc, (size_t)g->n_inc));
        // tasks: at most NB_WARP_TASK incidences of one row each
        std::vector<int64_t> inc_ptr((size_t)nw + 1), task_ptr((size_t)nw + 1, 0);
        NB_CUDA(cudaMemcpyAsync(inc_ptr.data(), g->d_inc_ptr, ((size_t)nw + 1) * 8, cudaMemcpyDeviceToHost, g->stream));
        NB_CUDA(cudaStreamSynchronize(g->stream));
        std::vector<int32_t> task_row, task_beg;
        for (int64_t r = 0; r < nw; r++) {
            int64_t n = inc_ptr[(size_t)r + 1] - inc_ptr[(size_t)r];
            task_ptr[(size_t)r] = (int64_t)task_row.size();
            for (int64_t b = 0; b < std::max<int64_t>(n, 1); b += NB_WARP_TASK) {
                task_row.push_back((int32_t)r);
                task_beg.push_back((int32_t)b);
            }
        }
        task_ptr[(size_t)nw] = (int64_t)task_row.size();
        g->n_wtasks = (int64_t)task_row.size();
        // (rows above NB_MAX_CARD -- 2-byte graphs -- write no task partials: nb_warp_sample_wide)
        const int part_card = std::min(g->max_card, NB_MAX_CARD);
        g->wpart_stride = part_card > 4 ? ((part_card + 3) & ~3) : 4;
        NB_TRY(upload(g, &g->d_wtask_row, task_row));
        NB_TRY(upload(g, &g->d_wtask_beg, task_beg));
        NB_TRY(upload(g, &g->d_wtask_ptr, task_ptr));
        NB_TRY(nb_alloc(g, &g->d_wpart, (size_t)g->n_wtasks * (size_t)g->wpart_stride));
        for (int c = 0; c < nc; c++) {
            NbColorRange &cr = g->colors[(size_t)c];
            cr.k_beg = (int32_t)task_ptr[(size_t)cr.w_beg];
            cr.k_end = (int32_t)task_ptr[(size_t)cr.w_end];
        }
    }
    k_fill_rows<<<grid_for(V), 256, 0, g->stream>>>(G, g->d_old2new, g->n_trows, g->d_slice_ptr, g->d_twords,
                                                    g->d_wrow_ptr, g->d_wwords, g->d_inc_ptr, g->d_inc, g->d_wfixed);
    NB_CUDA(cudaGetLastError());
    // ---- truth-table stream (FAST rows = new ids [0, n_frows)) ----
    {
        const int64_t nfs = g->n_frows / 32;
        int64_t *d_q;
        NB_TRY(nb_alloc(g, &d_q, (size_t)nfs + 1));
        NB_TRY(nb_alloc(g, &g->d_tt_ptr, (size_t)nfs + 1));
        if (nfs) k_tt_slice_width<<<grid_for(nfs), 256, 0, g->stream>>>(nfs, g->d_new2old, d_ninc, d_q);
        NB_TRY(exclusive_scan(g, d_q, g->d_tt_ptr, nfs + 1));
        NB_CUDA(cudaMemcpyAsync(&g->n_tt_quads, g->d_tt_ptr + nfs, 8, cudaMemcpyDeviceToHost, g->stream));
        NB_CUDA(cudaStreamSynchronize(g->stream));
        NB_TRY(nb_alloc(g, &g->d_tt, (size_t)g->n_tt_quads + 1, false));
        NB_TRY(nb_alloc(g, &g->d_tt_base, (size_t)g->n_tt_quads + 1, false));
        NB_TRY(nb_alloc(g, &g->d_tt_wid, (size_t)g->n_tt_quads + 1, false));
        if (g->n_tt_quads) {
            k_tt_pad<<<grid_for(g->n_tt_quads), 256, 0, g->stream>>>(g->d_tt, g->d_tt_base, g->d_tt_wid, g->n_tt_quads);
            if (g->wide)
                k_fill_tt<true><<<grid_for(V), 256, 0, g->stream>>>(G, g->d_old2new, g->n_frows, g->d_slice_ptr, g->d_twords, g->d_tt_ptr,
                                                                    g->d_tt, g->d_tt_base, g->d_tt_wid, g->d_wfixed, g->d_weight);
            else
                k_fill_tt<false><<<grid_for(V), 256, 0, g->stream>>>(G, g->d_old2new, g->n_frows, g->d_slice_ptr, g->d_twords, g->d_tt_ptr,
                                                                     g->d_tt, g->d_tt_base, g->d_tt_wid, g->d_wfixed, g->d_weight);
        }
        g->tt_weights_version = g->weights_version;
    }
    // ---- pair stream (PAIR rows = new ids [0, n_prows)) ----
    {
        const int64_t nps = g->n_prows / 32;
        int64_t *d_q;
        uint32_t *d_row_word;
        NB_TRY(nb_alloc(g, &d_q, (size_t)nps + 1));
        NB_TRY(nb_alloc(g, &g->d_tt2_ptr, (size_t)nps + 1));
        NB_TRY(nb_alloc(g, &g->d_tt2_common, (size_t)nps + 1, false));
        NB_TRY(nb_alloc(g, &d_row_word, (size_t)g->n_prows + 1, false));
        if (nps) {
            if (g->wide)
                k_tt2_row_word<true><<<grid_for(V), 256, 0, g->stream>>>(G, g->d_old2new, g->n_prows, g->d_slice_ptr, g->d_twords,
                                                                         g->d_wfixed, d_row_word);
            else
                k_tt2_row_word<false><<<grid_for(V), 256, 0, g->stream>>>(G, g->d_old2new, g->n_prows, g->d_slice_ptr, g->d_twords,
                                                                          g->d_wfixed, d_row_word);
            k_tt2_slice_width<<<grid_for(nps), 256, 0, g->stream>>>(nps, g->d_new2old, d_ninc, d_row_word, d_q, g->d_tt2_common);
        }
        NB_TRY(exclusive_scan(g, d_q, g->d_tt2_ptr, nps + 1));
        NB_CUDA(cudaMemcpyAsync(&g->n_tt2_quads, g->d_tt2_ptr + nps, 8, cudaMemcpyDeviceToHost, g->stream));
        NB_CUDA(cudaStreamSynchronize(g->stream));
        NB_TRY(nb_alloc(g, &g->d_tt2, (size_t)g->n_tt2_quads + 1, false));
        if (g->n_tt2_quads) {
            k_tt2_pad<<<(unsigned)nps, 128, 0, g->stream>>>(g->d_tt2, g->d_tt2_ptr, g->d_tt2_common, nps);
            if (g->wide)
                k_fill_tt2<true><<<grid_for(V), 256, 0, g->stream>>>(G, g->d_old2new, g->n_prows, g->d_slice_ptr, g->d_twords,
                                                                     g->d_tt2_ptr, g->d_tt2_common, g->d_tt2, g->d_wfixed);
            else
                k_fill_tt2<false><<<grid_for(V), 256, 0, g->stream>>>(G, g->d_old2new, g->n_prows, g->d_slice_ptr, g->d_twords,
                                                                      g->d_tt2_ptr, g->d_tt2_common, g->d_tt2, g->d_wfixed);
        }
    }
    // ---- categorical records (CAT rows = new ids [n_frows, n_crows)) ----
    {
        const int64_t ncs = (g->n_crows - g->n_frows) / 32;
        int64_t *d_q;
        NB_TRY(nb_alloc(g, &d_q, (size_t)ncs + 1));
        NB_TRY(nb_alloc(g, &g->d_cat_ptr, (size_t)ncs + 1));
        if (ncs) k_cat_slice_width<<<grid_for(ncs), 256, 0, g->stream>>>(ncs, g->n_frows, g->d_new2old, d_ninc, d_q);
        NB_TRY(exclusive_scan(g, d_q, g->d_cat_ptr, ncs + 1));
        NB_CUDA(cudaMemcpyAsync(&g->n_cat_quads, g->d_cat_ptr + ncs, 8, cudaMemcpyDeviceToHost, g->stream));
        NB_CUDA(cudaStreamSynchronize(g->stream));
        NB_TRY(nb_alloc(g, &g->d_cat, (size_t)g->n_cat_quads + 1, false));
        NB_TRY(nb_alloc(g, &g->d_cat_wid, (size_t)g->n_cat_quads + 1, false));
        if (g->n_cat_quads) {
            k_cat_pad<<<grid_for(g->n_cat_quads), 256, 0, g->stream>>>(g->d_cat, g->d_cat_wid, g->n_cat_quads);
            k_fill_cat<<<grid_for(V), 256, 0, g->stream>>>(G, g->d_old2new, g->n_frows, g->n_crows, g->d_cat_ptr, g->d_cat,
                                                           g->d_cat_wid, g->d_wfixed, g->d_weight);
        }
    }
    NB_CUDA(cudaGetLastError());
    NB_CUDA(cudaStreamSynchronize(g->stream));
    // bit mirror of the values (nb_common.cuh): all-Boolean graphs made of record rows and hub rows
    g->bits_eligible = g->max_card <= 2 && g->n_crows == g->n_frows && g->n_trows == g->n_crows && g->n_frows > 0;
    if (g->bits_eligible) NB_TRY(nb_alloc(g, &g->d_valbits, (size_t)((g->n_trows + g->n_wrows + 31) / 32 + 1)));
    nb_release_color_scratch(g);
    g->finalized = true;
    return NB_OK;
}

extern "C" int nb_graph_check_coloring(nb_graph *g, int64_t *conflicts)
{
    NB_CUDA(cudaSetDevice(g->device));
    unsigned long long *d_cnt;
    NB_CUDA(cudaMalloc(&d_cnt, 8));
    cudaMemsetAsync(d_cnt, 0, 8, g->stream);
    k_check_coloring<<<grid_for(g->V), 256, 0, g->stream>>>(raw_view(g), g->d_color, d_cnt);
    unsigned long long bad = 0;
    cudaMemcpyAsync(&bad, d_cnt, 8, cudaMemcpyDeviceToHost, g->stream);
    cudaError_t e = cudaStreamSynchronize(g->stream);
    cudaFree(d_cnt);
    NB_CUDA(e);
    *conflicts = (int64_t)bad;
    return NB_OK;
}
