// C-ABI entry points: graph lifecycle, state exchange at call boundaries,
// sweep drivers and measurement helpers (include/numbskull_b200.h).
#include <algorithm>
#include <atomic>
#include <cstring>
#include <thread>

#include "nb_common.cuh"

static inline unsigned grid_for(int64_t n, int block = 256) { return (unsigned)std::max<int64_t>(1, (n + block - 1) / block); }

// ---------------------------------------------------------------------------
// lifecycle
// ---------------------------------------------------------------------------
extern "C" int nb_graph_create(const nb_graph_desc *desc, nb_graph **out)
{
    *out = nullptr;
    if (!desc) NB_FAIL(NB_ERR_INVALID, "null descriptor");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        NB_FAIL(NB_ERR_CUDA, "no CUDA device available (%s); numbskull_b200 has no CPU fallback",
                e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    if (desc->device < 0 || desc->device >= ndev) NB_FAIL(NB_ERR_INVALID, "device %d out of range [0, %d)", desc->device, ndev);
    NB_CUDA(cudaSetDevice(desc->device));
    nb_graph *g = new nb_graph();
    g->device = desc->device;
    int rc = NB_OK;
    do {
        if (cudaStreamCreateWithFlags(&g->stream, cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreate(&g->ev0) != cudaSuccess || cudaEventCreate(&g->ev1) != cudaSuccess) {
            nb_set_error("stream/event creation failed: %s", cudaGetErrorString(cudaGetLastError()));
            rc = NB_ERR_CUDA;
            break;
        }
        rc = nb_build_device_graph(g, desc);
    } while (0);
    if (rc != NB_OK) { nb_graph_destroy(g); return rc; }
    *out = g;
    return NB_OK;
}

extern "C" void nb_graph_destroy(nb_graph *g)
{
    if (!g) return;
    cudaSetDevice(g->device);
    if (g->stream) cudaStreamSynchronize(g->stream);
    nb_p2p_destroy(g);
    for (void *p : g->allocs) cudaFree(p);
    if (g->d_xfer) cudaFree(g->d_xfer);
    if (g->d_flush) cudaFree(g->d_flush);
    if (g->h_pinned) cudaFreeHost(g->h_pinned);
    for (cudaEvent_t e : g->xfer_events) cudaEventDestroy(e);
    nb_release_color_scratch(g);
    for (int i = 0; i < NB_AUX_STREAMS; i++) {
        if (g->aux[i]) { cudaStreamSynchronize(g->aux[i]); cudaStreamDestroy(g->aux[i]); }
        if (g->ev_join[i]) cudaEventDestroy(g->ev_join[i]);
    }
    if (g->ev_fork) cudaEventDestroy(g->ev_fork);
    if (g->ev0) cudaEventDestroy(g->ev0);
    if (g->ev1) cudaEventDestroy(g->ev1);
    if (g->stream && g->own_stream) cudaStreamDestroy(g->stream);
    delete g;
}

extern "C" int nb_graph_get_info(const nb_graph *g, nb_graph_info *info)
{
    memset(info, 0, sizeof(*info));
    info->n_variable = g->V; info->n_factor = g->F; info->n_weight = g->W; info->n_edges = g->n_edges;
    info->n_colors = g->n_colors; info->wide_headers = g->wide ? 1 : 0;
    info->n_thread_rows = g->n_trows; info->n_warp_rows = g->n_wrows;
    info->stream_words = g->n_twords + g->n_wwords;
    info->device_bytes = g->device_bytes; info->count_entries = g->count_entries; info->jp_rounds = g->jp_rounds;
    info->max_arity = g->max_arity; info->n_pair_rows = g->n_prows; info->n_fast_rows = g->n_frows - g->n_prows;
    info->n_cat_rows = g->n_crows - g->n_frows; info->tt_quads = g->n_tt_quads; info->tt2_quads = g->n_tt2_quads;
    info->value_bytes = g->value_bytes;
    return NB_OK;
}

extern "C" int nb_graph_get_colors(const nb_graph *g, int32_t *colors)
{
    NB_CUDA(cudaSetDevice(g->device));
    NB_CUDA(cudaMemcpyAsync(colors, g->d_color, (size_t)g->V * 4, cudaMemcpyDeviceToHost, g->stream));
    NB_CUDA(cudaStreamSynchronize(g->stream));
    for (int64_t i = 0; i < g->V; i++) if (colors[i] < 0) colors[i] = -1;   /* -2 (ignored ghost) -> -1 */
    return NB_OK;
}

extern "C" int nb_graph_color_edges(const nb_graph *g, int64_t *edges_per_color)
{
    for (int c = 0; c < g->n_colors; c++) edges_per_color[c] = g->colors[(size_t)c].edges;
    return NB_OK;
}

// ---------------------------------------------------------------------------
// state exchange
//
// The caller's arrays keep the reference's types (int64 values and counts,
// float64 weights).  They are narrowed / widened on the host by a few threads
// next to pinned staging buffers, so only 1 byte per variable (2 on graphs with
// cardinalities above 255) and 4 bytes per count entry cross PCIe.
// ---------------------------------------------------------------------------
// The host conversion runs chunk by chunk on a few threads and overlaps with the PCIe copies:
// uploads are copied as soon as a chunk is narrowed, downloads are widened as soon as the chunk's
// copy has landed (one event per chunk).
static const int64_t NB_XFER_CHUNK = 1 << 18;   // elements

// Conversion threads of one process: at most 32, and the box's cores are shared by the ranks of a
// torchrun launch (LOCAL_WORLD_SIZE) -- 8 ranks x 32 threads on a 32-core host was what made the
// end-to-end step collapse at N = 8.  NUMBSKULL_B200_HOST_THREADS overrides.
static int nb_host_threads()
{
    static const int n = [] {
        const char *e = getenv("NUMBSKULL_B200_HOST_THREADS");
        if (e && atoi(e) > 0) return atoi(e);
        int cores = (int)std::max(1u, std::thread::hardware_concurrency());
        const char *lw = getenv("LOCAL_WORLD_SIZE");
        int ranks = lw && atoi(lw) > 0 ? atoi(lw) : 1;
        return std::max(1, std::min(32, cores / ranks));
    }();
    return n;
}

template <class F>
static int host_chunks(nb_graph *g, int64_t n, F fn)   // fn(chunk index, begin, end) -> cudaError_t
{
    const int64_t nchunks = (n + NB_XFER_CHUNK - 1) / NB_XFER_CHUNK;
    int nt = (int)std::min<int64_t>(nchunks, nb_host_threads());
    std::atomic<int64_t> next(0);
    std::atomic<int> err(0);
    auto work = [&](bool worker) {
        if (worker && cudaSetDevice(g->device) != cudaSuccess) { err.store((int)cudaErrorInvalidDevice); return; }
        for (;;) {
            const int64_t k = next.fetch_add(1);
            if (k >= nchunks) break;
            cudaError_t e = fn(k, k * NB_XFER_CHUNK, std::min(n, (k + 1) * NB_XFER_CHUNK));
            if (e != cudaSuccess) err.store((int)e);
        }
    };
    if (nt <= 1) {
        work(false);
    } else {
        std::vector<std::thread> th;
        for (int t = 0; t < nt; t++) th.emplace_back(work, true);
        for (auto &t : th) t.join();
    }
    if (err.load()) NB_FAIL(NB_ERR_CUDA, "host <-> device transfer failed: %s", cudaGetErrorString((cudaError_t)err.load()));
    return NB_OK;
}

// Widening loops.  The int64 / float64 result arrays are written once and not read back here, so
// on x86 hosts with AVX2 they go out as 32-byte non-temporal stores (no read-for-ownership of
// 3 x 134 MB on the C2 graph); other hosts use the plain loops.
#if defined(__x86_64__)
#include <immintrin.h>
#define NB_HAVE_AVX2_PATH 1
static bool nb_use_nt()
{
    static const bool on = __builtin_cpu_supports("avx2");
    return on;
}
__attribute__((target("avx2"))) static void widen_u8_nt(const uint8_t *s, int64_t *d, int64_t a, int64_t b)
{
    int64_t i = a;
    for (; i < b && ((uintptr_t)(d + i) & 31); i++) d[i] = (int64_t)s[i];
    for (; i + 4 <= b; i += 4) {
        uint32_t w;
        memcpy(&w, s + i, 4);
        _mm256_stream_si256((__m256i *)(d + i), _mm256_cvtepu8_epi64(_mm_cvtsi32_si128((int)w)));
    }
    for (; i < b; i++) d[i] = (int64_t)s[i];
    _mm_sfence();
}
template <class T>
__attribute__((target("avx2"))) static void merge_nt(const T *s, int64_t *c, int accumulate, double *m, double div, int64_t a,
                                                     int64_t b)
{
    // counts are read-modify-write when accumulating (plain stores), marginals are write-only
    int64_t i = a;
    auto one = [&](int64_t k) {
        int64_t x = accumulate ? c[k] + (int64_t)s[k] : (int64_t)s[k];
        c[k] = x;
        m[k] = (double)x / div;
    };
    for (; i < b && ((uintptr_t)(m + i) & 31); i++) one(i);
    for (; i + 4 <= b; i += 4) {
        alignas(32) double t[4];
        for (int j = 0; j < 4; j++) {
            int64_t x = accumulate ? c[i + j] + (int64_t)s[i + j] : (int64_t)s[i + j];
            c[i + j] = x;
            t[j] = (double)x / div;
        }
        _mm256_stream_pd(m + i, _mm256_load_pd(t));
    }
    for (; i < b; i++) one(i);
    _mm_sfence();
}
template <class T>
__attribute__((target("avx2"))) static void marginals_nt(const T *s, double *m, double div, int64_t a, int64_t b)
{
    int64_t i = a;
    for (; i < b && ((uintptr_t)(m + i) & 31); i++) m[i] = (double)s[i] / div;
    const __m256d vdiv = _mm256_set1_pd(div);
    for (; i + 4 <= b; i += 4) {
        const __m256d x = _mm256_set_pd((double)s[i + 3], (double)s[i + 2], (double)s[i + 1], (double)s[i]);
        _mm256_stream_pd(m + i, _mm256_div_pd(x, vdiv));
    }
    for (; i < b; i++) m[i] = (double)s[i] / div;
    _mm_sfence();
}
#else
#define NB_HAVE_AVX2_PATH 0
static bool nb_use_nt() { return false; }
#endif

static int ensure_events(nb_graph *g, int64_t n)
{
    while ((int64_t)g->xfer_events.size() < n) {
        cudaEvent_t e;
        NB_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        g->xfer_events.push_back(e);
    }
    return NB_OK;
}

// device -> pinned staging in chunks, one event per chunk
static int download_chunks(nb_graph *g, const void *d_src, int64_t n, int elem)
{
    const int64_t nchunks = (n + NB_XFER_CHUNK - 1) / NB_XFER_CHUNK;
    NB_TRY(ensure_events(g, nchunks));
    for (int64_t k = 0; k < nchunks; k++) {
        const int64_t a = k * NB_XFER_CHUNK, b = std::min(n, a + NB_XFER_CHUNK);
        NB_CUDA(cudaMemcpyAsync((char *)g->h_pinned + a * elem, (const char *)d_src + a * elem, (size_t)(b - a) * elem,
                                cudaMemcpyDeviceToHost, g->stream));
        NB_CUDA(cudaEventRecord(g->xfer_events[(size_t)k], g->stream));
    }
    return NB_OK;
}

// An out-of-range value is an error for an evidence variable; for a variable that is sampled
// anyway (or a ghost, refreshed by its owner) the reference simply overwrites it at the first
// sample (load_domains leaves a raw initialValue that is not in the explicit domain): mapped to 0.
// (T = the graph's value element type; the staged values have the same width)
template <class T>
__global__ void k_scatter_values(int64_t V, const T *in, const int32_t *old2new, const int32_t *v_card,
                                 const int8_t *v_evid, T *val, int *bad)
{
    int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (v >= V) return;
    int x = in[v];
    if (x >= v_card[v]) { if (v_evid[v] == 1) *bad = 1; x = 0; }
    val[old2new[v]] = (T)x;
}

template <class T>
__global__ void k_gather_values(int64_t V, const T *val, const int32_t *old2new, T *out)
{
    int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (v < V) out[v] = val[old2new[v]];
}

// Narrow to the value width on the host: anything outside [0, max value] becomes the largest
// value, which is >= every cardinality of the graph, so the device judges it out of range.
template <class T>
static int stage_values(nb_graph *g, const int64_t *values)
{
    const int64_t V = g->V;
    const int64_t top = (int64_t)(T)~(T)0;   // 255 / 65535
    T *stage = (T *)g->h_pinned;
    return host_chunks(g, V, [&](int64_t, int64_t a, int64_t b) {
        for (int64_t i = a; i < b; i++) {
            int64_t x = values[i];
            stage[i] = (x < 0 || x > top) ? (T)top : (T)x;
        }
        return cudaMemcpyAsync((T *)g->d_xfer + a, stage + a, (size_t)(b - a) * sizeof(T), cudaMemcpyHostToDevice, g->stream);
    });
}

extern "C" int nb_set_var_values(nb_graph *g, int chain, const int64_t *values)
{
    if (chain < 0 || chain > 1) NB_FAIL(NB_ERR_INVALID, "chain must be 0 or 1");
    if (!g->finalized) NB_FAIL(NB_ERR_INVALID, "graph not finalized");
    NB_CUDA(cudaSetDevice(g->device));
    const int64_t V = g->V;
    if (V == 0) return NB_OK;
    const size_t vb = (size_t)g->value_bytes;
    NB_TRY(nb_ensure_pinned(g, (size_t)V * vb + 64));
    NB_TRY(nb_ensure_xfer(g, (size_t)V * vb + 64));
    int rc = vb == 1 ? stage_values<nb_val_t>(g, values) : stage_values<nb_val16_t>(g, values);
    if (rc != NB_OK) {
        cudaStreamSynchronize(g->stream);
        return rc;
    }
    int *d_bad = (int *)((char *)g->d_xfer + (((size_t)V * vb + 15) & ~(size_t)15));
    NB_CUDA(cudaMemsetAsync(d_bad, 0, 4, g->stream));
    if (vb == 1)
        k_scatter_values<<<grid_for(V), 256, 0, g->stream>>>(V, (const nb_val_t *)g->d_xfer, g->d_old2new, g->d_v_card,
                                                             g->d_v_evid, nb_vals<nb_val_t>(g, chain), d_bad);
    else
        k_scatter_values<<<grid_for(V), 256, 0, g->stream>>>(V, (const nb_val16_t *)g->d_xfer, g->d_old2new, g->d_v_card,
                                                             g->d_v_evid, nb_vals<nb_val16_t>(g, chain), d_bad);
    int bad = 0;
    NB_CUDA(cudaMemcpyAsync(&bad, d_bad, 4, cudaMemcpyDeviceToHost, g->stream));
    NB_CUDA(cudaStreamSynchronize(g->stream));
    if (bad) NB_FAIL(NB_ERR_INVALID, "var_value of an evidence variable lies outside [0, cardinality)");
    return NB_OK;
}

extern "C" int nb_get_var_values(nb_graph *g, int chain, int64_t *values)
{
    if (chain < 0 || chain > 1) NB_FAIL(NB_ERR_INVALID, "chain must be 0 or 1");
    if (!g->finalized) NB_FAIL(NB_ERR_INVALID, "graph not finalized");
    NB_CUDA(cudaSetDevice(g->device));
    const int64_t V = g->V;
    if (V == 0) return NB_OK;
    const int vb = g->value_bytes;
    NB_TRY(nb_ensure_pinned(g, (size_t)V * vb + 64));
    NB_TRY(nb_ensure_xfer(g, (size_t)V * vb + 64));
    if (vb == 1)
        k_gather_values<<<grid_for(V), 256, 0, g->stream>>>(V, nb_vals<nb_val_t>(g, chain), g->d_old2new, (nb_val_t *)g->d_xfer);
    else
        k_gather_values<<<grid_for(V), 256, 0, g->stream>>>(V, nb_vals<nb_val16_t>(g, chain), g->d_old2new, (nb_val16_t *)g->d_xfer);
    int rc = download_chunks(g, g->d_xfer, V, vb);
    if (rc != NB_OK) { cudaStreamSynchronize(g->stream); return rc; }
    rc = host_chunks(g, V, [&](int64_t k, int64_t a, int64_t b) {
        cudaError_t e = cudaEventSynchronize(g->xfer_events[(size_t)k]);
        if (e != cudaSuccess) return e;
        if (vb == 2) {
            const nb_val16_t *stage16 = (const nb_val16_t *)g->h_pinned;
            for (int64_t i = a; i < b; i++) values[i] = (int64_t)stage16[i];
            return cudaSuccess;
        }
        const uint8_t *stage = (const uint8_t *)g->h_pinned;
#if NB_HAVE_AVX2_PATH
        if (nb_use_nt()) { widen_u8_nt(stage, values, a, b); return cudaSuccess; }
#endif
        for (int64_t i = a; i < b; i++) values[i] = (int64_t)stage[i];
        return cudaSuccess;
    });
    NB_CUDA(cudaStreamSynchronize(g->stream));
    return rc;
}

extern "C" int nb_set_weights(nb_graph *g, const double *weights)
{
    NB_CUDA(cudaSetDevice(g->device));
    NB_CUDA(cudaMemcpyAsync(g->d_weight, weights, (size_t)g->W * 8, cudaMemcpyHostToDevice, g->stream));
    NB_CUDA(cudaStreamSynchronize(g->stream));
    g->weights_version++;
    return NB_OK;
}

extern "C" int nb_get_weights(nb_graph *g, double *weights)
{
    NB_CUDA(cudaSetDevice(g->device));
    NB_CUDA(cudaMemcpyAsync(weights, g->d_weight, (size_t)g->W * 8, cudaMemcpyDeviceToHost, g->stream));
    NB_CUDA(cudaStreamSynchronize(g->stream));
    return NB_OK;
}

extern "C" int nb_get_weights_dev(nb_graph *g, double *dev_weights)
{
    NB_CUDA(cudaSetDevice(g->device));
    NB_CUDA(cudaMemcpyAsync(dev_weights, g->d_weight, (size_t)g->W * 8, cudaMemcpyDeviceToDevice, g->stream));
    return NB_OK;
}

extern "C" int nb_set_weights_dev(nb_graph *g, const double *dev_weights)
{
    NB_CUDA(cudaSetDevice(g->device));
    NB_CUDA(cudaMemcpyAsync(g->d_weight, dev_weights, (size_t)g->W * 8, cudaMemcpyDeviceToDevice, g->stream));
    g->weights_version++;
    return NB_OK;
}

extern "C" int nb_reset_counts(nb_graph *g)
{
    if (!g->finalized) NB_FAIL(NB_ERR_INVALID, "graph not finalized");
    NB_CUDA(cudaSetDevice(g->device));
    NB_CUDA(cudaMemsetAsync(g->d_count, 0, (size_t)g->count_entries * 4, g->stream));
    NB_CUDA(cudaMemsetAsync(g->d_count_b, 0, (size_t)g->Vn * 4, g->stream));
    g->tally_bound = g->tally_base = 0;
    g->tally_launches.clear();
    return NB_OK;
}

// new-order tallies -> reference cstart layout, narrowed on the fly: no tally exceeds g->tally_bound
// (tallying launches per colour since the last reset, plus the largest installed count, tracked on the
// host), so a short call's tallies cross PCIe as one byte each (two up to 65535 sweeps).
// (Boolean rows sampled by the truth-table kernels tally into count_b[new id].)
template <class T>
__global__ void k_counts_to_old(int64_t V, const int32_t *count, const int32_t *count_b, const uint32_t *cstart_new,
                                const int64_t *cstart_old, const int32_t *old2new, const int32_t *v_card, T *out)
{
    int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (v >= V) return;
    int n = v_card[v] == 2 ? 1 : v_card[v];
    int nid = old2new[v];
    uint32_t s = cstart_new[nid];
    int64_t d = cstart_old[v];
    for (int j = 0; j < n; j++) {
        int c = count[s + j];
        if (j == 0 && v_card[v] == 2) c += count_b[nid];
        out[d + j] = (T)c;
    }
}

// reference cstart layout -> new-order tallies (nb_set_counts)
__global__ void k_counts_from_old(int64_t V, int32_t *count, int32_t *count_b, const uint32_t *cstart_new,
                                  const int64_t *cstart_old, const int32_t *old2new, const int32_t *v_card, const int32_t *in)
{
    int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (v >= V) return;
    int n = v_card[v] == 2 ? 1 : v_card[v];
    int nid = old2new[v];
    uint32_t s = cstart_new[nid];
    int64_t d = cstart_old[v];
    for (int j = 0; j < n; j++) count[s + j] = in[d + j];
    count_b[nid] = 0;
}

template <class T>
static int merge_counts(nb_graph *g, int64_t n, int64_t *counts, int accumulate, double *marginals, double divisor)
{
    const T *src = (const T *)g->h_pinned;
    return host_chunks(g, n, [&](int64_t k, int64_t a, int64_t b) {
        cudaError_t e = cudaEventSynchronize(g->xfer_events[(size_t)k]);
        if (e != cudaSuccess) return e;
        if (!counts) {      // marginals only: the int64 count array is not materialised
#if NB_HAVE_AVX2_PATH
            if (nb_use_nt()) { marginals_nt<T>(src, marginals, divisor, a, b); return cudaSuccess; }
#endif
            for (int64_t i = a; i < b; i++) marginals[i] = (double)src[i] / divisor;
            return cudaSuccess;
        }
#if NB_HAVE_AVX2_PATH
        if (marginals && nb_use_nt()) { merge_nt<T>(src, counts, accumulate, marginals, divisor, a, b); return cudaSuccess; }
#endif
        for (int64_t i = a; i < b; i++) {
            int64_t c = accumulate ? counts[i] + (int64_t)src[i] : (int64_t)src[i];
            counts[i] = c;
            if (marginals) marginals[i] = (double)c / divisor;
        }
        return cudaSuccess;
    });
}

// element width the tallies travel with
static int tally_bytes(const nb_graph *g) { return g->tally_bound <= 255 ? 1 : (g->tally_bound <= 65535 ? 2 : 4); }

static int stage_counts(nb_graph *g, int elem)
{
    const int64_t n = g->count_entries;
    NB_TRY(nb_ensure_xfer(g, (size_t)n * elem + 256));
    const unsigned grid = grid_for(g->V);
    if (elem == 1)
        k_counts_to_old<uint8_t><<<grid, 256, 0, g->stream>>>(g->V, g->d_count, g->d_count_b, g->d_cstart, g->d_cstart_old,
                                                               g->d_old2new, g->d_v_card, (uint8_t *)g->d_xfer);
    else if (elem == 2)
        k_counts_to_old<uint16_t><<<grid, 256, 0, g->stream>>>(g->V, g->d_count, g->d_count_b, g->d_cstart, g->d_cstart_old,
                                                                g->d_old2new, g->d_v_card, (uint16_t *)g->d_xfer);
    else
        k_counts_to_old<int32_t><<<grid, 256, 0, g->stream>>>(g->V, g->d_count, g->d_count_b, g->d_cstart, g->d_cstart_old,
                                                               g->d_old2new, g->d_v_card, (int32_t *)g->d_xfer);
    NB_CUDA(cudaGetLastError());
    return NB_OK;
}

static int fetch_counts(nb_graph *g, int64_t *counts, int accumulate, double *marginals, double divisor)
{
    if (!g->finalized) NB_FAIL(NB_ERR_INVALID, "graph not finalized");
    NB_CUDA(cudaSetDevice(g->device));
    const int64_t n = g->count_entries;
    if (n == 0) return NB_OK;
    const int elem = tally_bytes(g);
    NB_TRY(nb_ensure_pinned(g, (size_t)n * elem));
    NB_TRY(stage_counts(g, elem));
    int rc = download_chunks(g, g->d_xfer, n, elem);
    if (rc == NB_OK) {
        if (elem == 1) rc = merge_counts<uint8_t>(g, n, counts, accumulate, marginals, divisor);
        else if (elem == 2) rc = merge_counts<uint16_t>(g, n, counts, accumulate, marginals, divisor);
        else rc = merge_counts<int32_t>(g, n, counts, accumulate, marginals, divisor);
    }
    NB_CUDA(cudaStreamSynchronize(g->stream));
    return rc;
}

extern "C" int nb_get_counts(nb_graph *g, int64_t *counts, int accumulate)
{
    return fetch_counts(g, counts, accumulate, nullptr, 1.0);
}

extern "C" int nb_get_counts_marginals(nb_graph *g, int64_t *counts, int accumulate, double *marginals, double epochs)
{
    return fetch_counts(g, counts, accumulate, marginals, epochs);
}

extern "C" int nb_get_marginals(nb_graph *g, double *marginals, double epochs)
{
    if (!marginals) NB_FAIL(NB_ERR_INVALID, "null marginals");
    return fetch_counts(g, nullptr, 0, marginals, epochs);
}

extern "C" int nb_get_counts_compact(nb_graph *g, void *out, int64_t out_bytes, int32_t *elem_bytes)
{
    if (!g->finalized) NB_FAIL(NB_ERR_INVALID, "graph not finalized");
    NB_CUDA(cudaSetDevice(g->device));
    const int elem = tally_bytes(g);
    *elem_bytes = elem;
    const int64_t n = g->count_entries;
    if (n == 0) return NB_OK;
    if (out_bytes < n * elem) NB_FAIL(NB_ERR_INVALID, "buffer of %lld bytes is too small for %lld tallies of %d bytes", (long long)out_bytes, (long long)n, elem);
    NB_TRY(stage_counts(g, elem));
    NB_CUDA(cudaMemcpyAsync(out, g->d_xfer, (size_t)n * elem, cudaMemcpyDeviceToHost, g->stream));
    NB_CUDA(cudaStreamSynchronize(g->stream));
    return NB_OK;
}

extern "C" int nb_host_alloc(void **ptr, int64_t bytes)
{
    cudaError_t e = cudaMallocHost(ptr, (size_t)std::max<int64_t>(bytes, 16));
    if (e != cudaSuccess) NB_FAIL(NB_ERR_NOMEM, "cudaMallocHost(%lld) failed: %s", (long long)bytes, cudaGetErrorString(e));
    return NB_OK;
}

extern "C" int nb_host_free(void *ptr)
{
    if (ptr) cudaFreeHost(ptr);
    return NB_OK;
}

extern "C" int nb_set_counts(nb_graph *g, const int64_t *counts)
{
    if (!g->finalized) NB_FAIL(NB_ERR_INVALID, "graph not finalized");
    NB_CUDA(cudaSetDevice(g->device));
    const int64_t n = g->count_entries;
    if (n == 0) return NB_OK;
    NB_TRY(nb_ensure_pinned(g, (size_t)n * 4));
    NB_TRY(nb_ensure_xfer(g, (size_t)n * 4 + 256));
    int32_t *stage = (int32_t *)g->h_pinned;
    std::atomic<long long> mx(0);
    std::atomic<int> bad(0);
    int rc = host_chunks(g, n, [&](int64_t, int64_t a, int64_t b) {
        long long m = 0;
        for (int64_t i = a; i < b; i++) {
            const int64_t c = counts[i];
            if (c < 0 || c > 0x7FFFFFFF) bad.store(1);
            stage[i] = (int32_t)c;
            m = std::max<long long>(m, c);
        }
        long long cur = mx.load();
        while (m > cur && !mx.compare_exchange_weak(cur, m)) {}
        return cudaMemcpyAsync((int32_t *)g->d_xfer + a, stage + a, (size_t)(b - a) * 4, cudaMemcpyHostToDevice, g->stream);
    });
    if (rc != NB_OK || bad.load()) {
        cudaStreamSynchronize(g->stream);
        if (rc != NB_OK) return rc;
        NB_FAIL(NB_ERR_INVALID, "count holds entries outside [0, 2^31)");
    }
    k_counts_from_old<<<grid_for(g->V), 256, 0, g->stream>>>(g->V, g->d_count, g->d_count_b, g->d_cstart, g->d_cstart_old,
                                                              g->d_old2new, g->d_v_card, (const int32_t *)g->d_xfer);
    NB_CUDA(cudaGetLastError());
    NB_CUDA(cudaStreamSynchronize(g->stream));
    g->tally_bound = g->tally_base = mx.load();
    g->tally_launches.clear();
    return NB_OK;
}

// ---------------------------------------------------------------------------
// hot path drivers
// ---------------------------------------------------------------------------
static int check_runnable(const nb_graph *g)
{
    if (!g->finalized) NB_FAIL(NB_ERR_INVALID, "graph not finalized: colour it (nb_color_round) and call nb_graph_finalize first");
    if (g->has_unknown_func)
        NB_FAIL(NB_ERR_NOT_IMPLEMENTED, "Error: Factor Function %d ( used in factor %lld ) is not implemented.",
                g->unknown_func_id, (long long)g->unknown_func_factor);
    return NB_OK;
}

extern "C" int nb_potentials(nb_graph *g, int chain, const int64_t *var_ids, int64_t n, const int64_t *out_offsets,
                             double *out, int64_t n_out)
{
    NB_CUDA(cudaSetDevice(g->device));
    NB_TRY(check_runnable(g));
    return nb_run_potentials(g, chain, var_ids, n, out_offsets, out, n_out);
}

extern "C" int nb_potentials_records(nb_graph *g, int chain, const int64_t *var_ids, int64_t n, const int64_t *out_offsets,
                                     double *out, int64_t n_out, int32_t *row_class)
{
    NB_CUDA(cudaSetDevice(g->device));
    NB_TRY(check_runnable(g));
    return nb_run_potentials_records(g, chain, var_ids, n, out_offsets, out, n_out, row_class);
}

extern "C" int nb_begin_epoch(nb_graph *g, int64_t *epoch)
{
    *epoch = (int64_t)g->epoch_counter++;
    return NB_OK;
}

extern "C" int nb_gibbs_color_phase(nb_graph *g, int color, int burnin, int sample_evidence, uint64_t seed, int64_t epoch)
{
    NB_CUDA(cudaSetDevice(g->device));
    NB_TRY(check_runnable(g));
    return nb_launch_gibbs_color(g, color, burnin, sample_evidence, seed, (uint64_t)epoch);
}

extern "C" int nb_gibbs_sweeps(nb_graph *g, int64_t n_epochs, int burnin, int sample_evidence, uint64_t seed)
{
    NB_CUDA(cudaSetDevice(g->device));
    NB_TRY(check_runnable(g));
    NB_TRY(nb_check_tally_room(g, burnin, n_epochs));
    NB_TRY(nb_refresh_inlined_weights(g));
    static const bool fan = [] { const char *e = getenv("NUMBSKULL_B200_FAN_OUT"); return !e || atoi(e) != 0; }();
    g->fan_out = fan && g->p2p == nullptr;
    // member gathers from the bit mirror once the byte array outgrows L2 (NUMBSKULL_B200_BIT_MIRROR =
    // minimum number of variables, 0 = always, negative = never)
    const char *bits_env = getenv("NUMBSKULL_B200_BIT_MIRROR");          // (read per call: the tests toggle it)
    const long long bits_min = bits_env ? atoll(bits_env) : 100000000ll;
    g->use_bits = g->bits_eligible && g->p2p == nullptr && bits_min >= 0 && g->V >= bits_min;
    int rc = g->use_bits ? nb_pack_value_bits(g) : NB_OK;     // (no early return: the flags below are always reset)
    for (int64_t ep = 0; ep < n_epochs && rc == NB_OK; ep++) {
        uint64_t epoch = g->epoch_counter++;
        for (int c = 0; c < g->n_colors && rc == NB_OK; c++) rc = nb_launch_gibbs_color(g, c, burnin, sample_evidence, seed, epoch);
    }
    g->fan_out = false;
    g->use_bits = false;
    NB_TRY(rc);
    NB_CUDA(cudaStreamSynchronize(g->stream));
    return NB_OK;
}

extern "C" int nb_learn_sweeps(nb_graph *g, int64_t n_epochs, double *stepsize, double decay, int regularization,
                               double reg_param, double truncation, int learn_non_evidence, uint64_t seed,
                               int64_t batch_visits)
{
    NB_CUDA(cudaSetDevice(g->device));
    NB_TRY(check_runnable(g));
    NB_TRY(nb_run_learn(g, n_epochs, stepsize, decay, regularization, reg_param, truncation, learn_non_evidence, seed,
                        batch_visits));
    NB_CUDA(cudaStreamSynchronize(g->stream));
    return NB_OK;
}

// ---------------------------------------------------------------------------
// measurement helpers
// ---------------------------------------------------------------------------
extern "C" int nb_timer_start(nb_graph *g)
{
    NB_CUDA(cudaSetDevice(g->device));
    NB_CUDA(cudaEventRecord(g->ev0, g->stream));
    return NB_OK;
}

extern "C" int nb_timer_stop(nb_graph *g, float *ms)
{
    NB_CUDA(cudaSetDevice(g->device));
    NB_CUDA(cudaEventRecord(g->ev1, g->stream));
    NB_CUDA(cudaEventSynchronize(g->ev1));
    NB_CUDA(cudaEventElapsedTime(ms, g->ev0, g->ev1));
    return NB_OK;
}

extern "C" int nb_synchronize(nb_graph *g)
{
    NB_CUDA(cudaSetDevice(g->device));
    NB_CUDA(cudaStreamSynchronize(g->stream));
    return NB_OK;
}

extern "C" int nb_launch_count(const nb_graph *g, int64_t *launches)
{
    *launches = g->launches;
    return NB_OK;
}

__global__ void k_flush(uint4 *p, int64_t n, uint32_t tag)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) p[i] = make_uint4(tag, tag, tag, tag);
}

extern "C" int nb_flush_l2(nb_graph *g, int64_t bytes)
{
    NB_CUDA(cudaSetDevice(g->device));
    if ((size_t)bytes > g->flush_bytes) {
        if (g->d_flush) cudaFree(g->d_flush);
        g->d_flush = nullptr;
        g->flush_bytes = 0;
        NB_CUDA(cudaMalloc(&g->d_flush, (size_t)bytes));
        g->flush_bytes = (size_t)bytes;
    }
    k_flush<<<148 * 8, 256, 0, g->stream>>>((uint4 *)g->d_flush, bytes / 16, (uint32_t)g->launches);
    NB_CUDA(cudaGetLastError());
    return NB_OK;
}

// ---------------------------------------------------------------------------
// partitioned graphs: gather / scatter by original local id on device buffers
// ---------------------------------------------------------------------------
__global__ void k_gather_u8(int64_t n, const int32_t *ids, const int32_t *old2new, const nb_val_t *val, uint8_t *out)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) out[i] = val[old2new[ids[i]]];
}
__global__ void k_scatter_u8(int64_t n, const int32_t *ids, const int32_t *old2new, nb_val_t *val, const uint8_t *in)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) val[old2new[ids[i]]] = in[i];
}

extern "C" int nb_gather_values_dev(nb_graph *g, int chain, const int32_t *dev_local_ids, int64_t n, uint8_t *dev_out)
{
    if (chain < 0 || chain > 1) NB_FAIL(NB_ERR_INVALID, "chain must be 0 or 1");
    if (g->value_bytes != 1) NB_FAIL(NB_ERR_UNSUPPORTED, "byte-valued halo transfers need a graph whose cardinalities are all <= 255");
    if (n == 0) return NB_OK;
    NB_CUDA(cudaSetDevice(g->device));
    k_gather_u8<<<grid_for(n), 256, 0, g->stream>>>(n, dev_local_ids, g->d_old2new, nb_vals<nb_val_t>(g, chain), dev_out);
    g->launches++;
    NB_CUDA(cudaGetLastError());
    return NB_OK;
}

extern "C" int nb_scatter_values_dev(nb_graph *g, int chain, const int32_t *dev_local_ids, int64_t n, const uint8_t *dev_in)
{
    if (chain < 0 || chain > 1) NB_FAIL(NB_ERR_INVALID, "chain must be 0 or 1");
    if (g->value_bytes != 1) NB_FAIL(NB_ERR_UNSUPPORTED, "byte-valued halo transfers need a graph whose cardinalities are all <= 255");
    if (n == 0) return NB_OK;
    NB_CUDA(cudaSetDevice(g->device));
    k_scatter_u8<<<grid_for(n), 256, 0, g->stream>>>(n, dev_local_ids, g->d_old2new, nb_vals<nb_val_t>(g, chain), dev_in);
    g->launches++;
    NB_CUDA(cudaGetLastError());
    return NB_OK;
}

extern "C" int nb_learn_color_phase(nb_graph *g, int color, int block, int n_blocks, double stepsize, int regularization,
                                    double reg_param, double truncation, int learn_non_evidence, uint64_t seed,
                                    int64_t epoch)
{
    NB_CUDA(cudaSetDevice(g->device));
    NB_TRY(check_runnable(g));
    return nb_learn_color(g, color, block, n_blocks, stepsize, regularization, reg_param, truncation,
                          learn_non_evidence, seed, (uint64_t)epoch);
}

extern "C" int nb_learn_blocks(nb_graph *g, double stepsize, int learn_non_evidence, int64_t batch_visits, int *n_blocks)
{
    NB_CUDA(cudaSetDevice(g->device));
    NB_TRY(check_runnable(g));
    return nb_learn_block_count(g, stepsize, learn_non_evidence, batch_visits, n_blocks);
}

extern "C" int nb_learn_cell_ids(nb_graph *g, int color, int block, int n_blocks, int64_t *ids, int64_t *n)
{
    NB_CUDA(cudaSetDevice(g->device));
    NB_TRY(check_runnable(g));
    return nb_learn_cell_id_list(g, color, block, n_blocks, ids, n);
}

extern "C" int nb_color_round(nb_graph *g, int64_t *remaining)
{
    NB_CUDA(cudaSetDevice(g->device));
    if (g->finalized) { *remaining = 0; return NB_OK; }
    return nb_build_color_round(g, remaining);
}

extern "C" int nb_color_restart(nb_graph *g, int mode)
{
    NB_CUDA(cudaSetDevice(g->device));
    return nb_build_color_restart(g, mode);
}

extern "C" int nb_color_natural_round_cap(void) { return nb_natural_round_cap(); }

extern "C" int nb_color_min_ids(nb_graph *g, int n_colors, int64_t *min_ids)
{
    NB_CUDA(cudaSetDevice(g->device));
    return nb_build_color_min_ids(g, n_colors, min_ids);
}

extern "C" int nb_relabel_colors(nb_graph *g, const int32_t *map, int n)
{
    NB_CUDA(cudaSetDevice(g->device));
    return nb_build_relabel_colors(g, map, n);
}

// Split every colour c of a partitioned (deferred) graph into the phases 2c (ghosts and the owned
// variables some other rank holds a copy of: `boundary_ids`, local ids) and 2c + 1 (interior
// variables, which never read a ghost).  The boundary phase is tiny; its halo push then travels
// while the interior phase runs (nb_gibbs_sweeps_p2p mode 2).
__global__ void k_split_all(int64_t V, const int8_t *evid, int32_t *color)
{
    int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (v < V && color[v] >= 0) color[v] = 2 * color[v] + (evid[v] == 4 ? 0 : 1);
}
__global__ void k_split_boundary(int64_t n, const int32_t *ids, int32_t *color)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n && color[ids[i]] >= 0) color[ids[i]] &= ~1;
}

extern "C" int nb_split_colors(nb_graph *g, const int32_t *boundary_ids, int64_t n)
{
    NB_CUDA(cudaSetDevice(g->device));
    if (g->finalized || !g->deferred) NB_FAIL(NB_ERR_INVALID, "nb_split_colors needs a deferred graph before nb_graph_finalize");
    for (int64_t i = 0; i < n; i++)
        if (boundary_ids[i] < 0 || boundary_ids[i] >= g->V) NB_FAIL(NB_ERR_INVALID, "boundary id out of range");
    const unsigned grid = (unsigned)((std::max<int64_t>(g->V, 1) + 255) / 256);
    k_split_all<<<grid, 256, 0, g->stream>>>(g->V, g->d_v_evid, g->d_color);
    if (n) {
        int32_t *d_ids;
        NB_CUDA(cudaMalloc(&d_ids, (size_t)n * 4));
        cudaMemcpyAsync(d_ids, boundary_ids, (size_t)n * 4, cudaMemcpyHostToDevice, g->stream);
        k_split_boundary<<<(unsigned)((n + 255) / 256), 256, 0, g->stream>>>(n, d_ids, g->d_color);
        cudaError_t e = cudaStreamSynchronize(g->stream);
        cudaFree(d_ids);
        NB_CUDA(e);
    }
    NB_CUDA(cudaGetLastError());
    return NB_OK;
}

extern "C" int nb_graph_finalize(nb_graph *g)
{
    NB_CUDA(cudaSetDevice(g->device));
    return nb_build_finalize(g);
}

__global__ void k_gather_i32(int64_t n, const int32_t *ids, const int32_t *src, int32_t *out)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) out[i] = src[ids[i]];
}
__global__ void k_scatter_i32(int64_t n, const int32_t *ids, int32_t *dst, const int32_t *in)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) dst[ids[i]] = in[i];
}

extern "C" int nb_gather_colors_dev(nb_graph *g, const int32_t *dev_local_ids, int64_t n, int32_t *dev_out)
{
    if (n == 0) return NB_OK;
    NB_CUDA(cudaSetDevice(g->device));
    k_gather_i32<<<grid_for(n), 256, 0, g->stream>>>(n, dev_local_ids, g->d_color, dev_out);
    NB_CUDA(cudaGetLastError());
    return NB_OK;
}

extern "C" int nb_scatter_colors_dev(nb_graph *g, const int32_t *dev_local_ids, int64_t n, const int32_t *dev_in)
{
    if (n == 0) return NB_OK;
    NB_CUDA(cudaSetDevice(g->device));
    k_scatter_i32<<<grid_for(n), 256, 0, g->stream>>>(n, dev_local_ids, g->d_color, dev_in);
    NB_CUDA(cudaGetLastError());
    return NB_OK;
}

extern "C" int nb_set_stream(nb_graph *g, void *cuda_stream)
{
    NB_CUDA(cudaSetDevice(g->device));
    NB_CUDA(cudaStreamSynchronize(g->stream));
    if (g->own_stream && g->stream) cudaStreamDestroy(g->stream);
    g->stream = (cudaStream_t)cuda_stream;
    g->own_stream = false;
    return NB_OK;
}
