// Host-side integer work of the drop-in boundary: error strings, the DeepDive
// binary parsers and the (bit-exact) variable-to-factor index builder.
#include <algorithm>
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <thread>
#include <vector>

#include "nb_common.cuh"

static thread_local char g_err[1024] = "";

void nb_set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

extern "C" const char *nb_last_error(void) { return g_err; }
extern "C" int nb_abi_version(void) { return NB_ABI_VERSION; }

extern "C" int nb_device_count(int *count)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        *count = 0;
        NB_FAIL(NB_ERR_CUDA, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
    }
    *count = n;
    return NB_OK;
}

// ---------------------------------------------------------------------------
// numbskull.py:219-227 (and :309-317): vtf_offset = running count of
// VarToFactor records; Boolean (dataType 0) variables take one record,
// categorical ones `cardinality`.
// ---------------------------------------------------------------------------
extern "C" int nb_assign_vtf_offsets(nb_variable_rec *variable, int64_t n_variable, int64_t *n_vtf)
{
    int64_t n = 0;
    for (int64_t i = 0; i < n_variable; i++) {
        variable[i].vtf_offset = n;
        if (variable[i].dataType == 0) n += 1;
        else {
            if (variable[i].cardinality < 0) NB_FAIL(NB_ERR_INVALID, "variable %lld: negative cardinality", (long long)i);
            n += variable[i].cardinality;
        }
    }
    *n_vtf = n;
    return NB_OK;
}

// ---------------------------------------------------------------------------
// dataloading.py:16-81 compute_var_map.  Same outputs as the reference's four
// steps: (1) bucket lengths from every fmap entry, (2) exclusive scan ->
// offsets, (3) factor ids scattered into the buckets (skipping factors_to_skip),
// (4) per bucket sort + unique with the length shrunk and the offsets left alone.
// The reference scatters in factor order, so its buckets come out ascending and
// step 4 only removes duplicates; here steps 1, 3 and 4 run on host threads
// (atomic bucket cursors, then each bucket is sorted), which yields the same
// ascending, de-duplicated buckets whatever the thread interleaving.
// ---------------------------------------------------------------------------
static inline int64_t bucket_of(const nb_variable_rec *variable, const nb_ftv_rec &m)
{
    const nb_variable_rec &v = variable[m.vid];
    return v.vtf_offset + (v.dataType == 1 ? m.dense_equal_to : 0);
}

template <class F>
static void host_threads(int64_t n, F fn)
{
    int nt = n > (1 << 16) ? (int)std::min(32u, std::max(1u, std::thread::hardware_concurrency())) : 1;
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

static inline int64_t atomic_fetch_add_i64(int64_t *p, int64_t x) { return __atomic_fetch_add(p, x, __ATOMIC_RELAXED); }

// ---------------------------------------------------------------------------
// Atomics-free index build for the usual layout (factors tile fmap in order, nothing skipped):
// the variable ids are cut into one range per thread with about the same number of fmap entries;
// every thread stages the (bucket, factor) pairs of its contiguous factor chunk per destination
// range (8 bytes each, factor order kept), then every thread owns one range and counts / fills
// its buckets from the staged pairs alone -- local writes, no shared cursors, buckets come out
// ascending.  Returns false (nothing written) when the layout or the sizes do not qualify; the
// caller then takes the general path.  Identical output to the general path by construction.
// ---------------------------------------------------------------------------
struct NbStaged { uint32_t bucket_rel, fid; };

template <class F>
static void run_threads(int nt, F fn)
{
    if (nt == 1) { fn(0); return; }
    std::vector<std::thread> th;
    for (int t = 0; t < nt; t++) th.emplace_back([=] { fn(t); });
    for (auto &t : th) t.join();
}

static bool var_map_partitioned(const nb_variable_rec *variable, int64_t n_variable, const nb_factor_rec *factor,
                                int64_t n_factor, const nb_ftv_rec *fmap, int64_t n_fmap, nb_vtf_rec *vmap, int64_t n_vmap,
                                int64_t *factor_index, int64_t n_factor_index, int *bad_out, char *msg, size_t msg_len)
{
    if (n_fmap < (1 << 20) || n_factor >= (1ll << 32) || n_variable < 64 || n_factor_index < n_fmap) return false;
    const char *nt_env = getenv("NUMBSKULL_B200_HOST_THREADS");
    const int nt = nt_env ? std::max(1, std::min(64, atoi(nt_env)))
                          : (int)std::min<int64_t>(32, std::max(1u, std::thread::hardware_concurrency()));
    if (nt < 2) return false;
    // contiguous factor chunks and the fmap positions they start at
    std::vector<int64_t> fbeg((size_t)nt + 1), ebeg((size_t)nt + 1, 0), esum((size_t)nt, 0);
    for (int t = 0; t <= nt; t++) fbeg[(size_t)t] = n_factor * t / nt;
    run_threads(nt, [&](int t) {
        int64_t s = 0;
        for (int64_t f = fbeg[(size_t)t]; f < fbeg[(size_t)t + 1]; f++) s += factor[f].arity;
        esum[(size_t)t] = s;
    });
    for (int t = 0; t < nt; t++) ebeg[(size_t)t + 1] = ebeg[(size_t)t] + esum[(size_t)t];
    if (ebeg[(size_t)nt] != n_fmap) return false;
    std::atomic<int> canonical(1), bad(0);
    auto fail = [&](const char *what, int64_t idx) {
        int expected = 0;
        if (bad.compare_exchange_strong(expected, 1)) snprintf(msg, msg_len, "%s (index %lld)", what, (long long)idx);
    };
    // coarse histogram of the variable ids (also: layout check, vid validation)
    int shift = 0;
    while ((n_variable >> shift) > 65536) shift++;
    const int64_t nbins = ((n_variable - 1) >> shift) + 1;
    std::vector<std::vector<int64_t>> hist((size_t)nt);
    run_threads(nt, [&](int t) {
        std::vector<int64_t> &h = hist[(size_t)t];
        h.assign((size_t)nbins, 0);
        int64_t e = ebeg[(size_t)t];
        for (int64_t f = fbeg[(size_t)t]; f < fbeg[(size_t)t + 1]; f++) {
            if (factor[f].ftv_offset != e) { canonical.store(0); return; }
            e += factor[f].arity;
        }
        for (int64_t j = ebeg[(size_t)t]; j < ebeg[(size_t)t + 1]; j++) {
            const int64_t vid = fmap[j].vid;
            if (vid < 0 || vid >= n_variable) { fail("fmap vid out of range", j); return; }
            h[(size_t)(vid >> shift)]++;
        }
    });
    if (!canonical.load()) return false;
    if (bad.load()) { *bad_out = 1; return true; }
    // ranges of whole bins with ~n_fmap / nt entries each
    std::vector<int64_t> total((size_t)nbins, 0);
    for (int t = 0; t < nt; t++)
        for (int64_t b = 0; b < nbins; b++) total[(size_t)b] += hist[(size_t)t][(size_t)b];
    std::vector<int32_t> range_of_bin((size_t)nbins);
    std::vector<int64_t> range_first_bin((size_t)nt + 1, nbins);
    {
        int64_t acc = 0;
        int r = 0;
        range_first_bin[0] = 0;
        for (int64_t b = 0; b < nbins; b++) {
            while (r + 1 < nt && acc >= n_fmap * (int64_t)(r + 1) / nt) range_first_bin[(size_t)++r] = b;
            range_of_bin[(size_t)b] = r;
            acc += total[(size_t)b];
        }
        for (int q = r + 1; q <= nt; q++) range_first_bin[(size_t)q] = nbins;
    }
    // bucket span of every range (vtf_offset is increasing in the variable id; the caller checked the bounds)
    std::vector<int64_t> bucket_base((size_t)nt + 1);
    for (int r = 0; r <= nt; r++) {
        const int64_t v0 = std::min(n_variable, range_first_bin[(size_t)r] << shift);
        bucket_base[(size_t)r] = v0 < n_variable ? variable[v0].vtf_offset : n_vmap;
    }
    for (int r = 0; r < nt; r++) {
        if (bucket_base[(size_t)r + 1] < bucket_base[(size_t)r]) return false;          // offsets not monotone: general path
        if (bucket_base[(size_t)r + 1] - bucket_base[(size_t)r] >= (1ll << 32)) return false;
    }
    // staging positions: range-major, then source thread (= factor order inside a range)
    std::vector<int64_t> pos((size_t)nt * nt), range_beg((size_t)nt + 1, 0);
    for (int r = 0; r < nt; r++) {
        int64_t acc = range_beg[(size_t)r];
        for (int t = 0; t < nt; t++) {
            int64_t c = 0;
            for (int64_t b = range_first_bin[(size_t)r]; b < range_first_bin[(size_t)r + 1]; b++) c += hist[(size_t)t][(size_t)b];
            pos[(size_t)t * nt + r] = acc;
            acc += c;
        }
        range_beg[(size_t)r + 1] = acc;
    }
    NbStaged *staged = (NbStaged *)malloc((size_t)n_fmap * sizeof(NbStaged));
    if (!staged) return false;
    run_threads(nt, [&](int t) {
        std::vector<int64_t> cur(pos.begin() + (size_t)t * nt, pos.begin() + (size_t)(t + 1) * nt);
        for (int64_t f = fbeg[(size_t)t]; f < fbeg[(size_t)t + 1]; f++) {
            const int64_t a = factor[f].ftv_offset, n = factor[f].arity;
            for (int64_t j = a; j < a + n; j++) {
                const nb_ftv_rec &m = fmap[j];
                const nb_variable_rec &v = variable[m.vid];
                if (v.dataType == 1 && (m.dense_equal_to < 0 || m.dense_equal_to >= v.cardinality)) {
                    fail("fmap dense_equal_to outside the variable's cardinality", j);
                    return;
                }
                const int r = range_of_bin[(size_t)(m.vid >> shift)];
                const int64_t bucket = v.vtf_offset + (v.dataType == 1 ? m.dense_equal_to : 0);
                if (bucket < bucket_base[(size_t)r] || bucket >= bucket_base[(size_t)r + 1]) { canonical.store(0); return; }
                staged[cur[(size_t)r]++] = NbStaged{(uint32_t)(bucket - bucket_base[(size_t)r]), (uint32_t)f};
            }
        }
    });
    if (bad.load() || !canonical.load()) {
        free(staged);
        if (bad.load()) { *bad_out = 1; return true; }
        return false;   // (nothing was written to vmap / factor_index yet)
    }
    // bucket lengths, per range
    run_threads(nt, [&](int r) {
        const int64_t base = bucket_base[(size_t)r];
        for (int64_t i = range_beg[(size_t)r]; i < range_beg[(size_t)r + 1]; i++)
            vmap[base + staged[i].bucket_rel].factor_index_length += 1;
    });
    int64_t last_len = 0, last_off = 0;
    for (int64_t i = 0; i < n_vmap; i++) {
        vmap[i].factor_index_offset = last_off + last_len;
        last_len = vmap[i].factor_index_length;
        last_off = vmap[i].factor_index_offset;
    }
    // fill (ascending factor ids per bucket) and drop duplicates in place, like dataloading.py:67-81
    run_threads(nt, [&](int r) {
        const int64_t base = bucket_base[(size_t)r], nb = bucket_base[(size_t)r + 1] - base;
        std::vector<uint32_t> filled((size_t)nb, 0);
        for (int64_t i = range_beg[(size_t)r]; i < range_beg[(size_t)r + 1]; i++) {
            const NbStaged e = staged[i];
            factor_index[vmap[base + e.bucket_rel].factor_index_offset + filled[e.bucket_rel]++] = (int64_t)e.fid;
        }
        for (int64_t b = base; b < base + nb; b++) {
            int64_t *p = factor_index + vmap[b].factor_index_offset;
            const int64_t len = vmap[b].factor_index_length;
            int64_t n = 0, last = -1;
            for (int64_t k = 0; k < len; k++) {
                if (p[k] == last) continue;
                last = p[k];
                p[n++] = last;
            }
            vmap[b].factor_index_length = n;
        }
    });
    free(staged);
    return true;
}

extern "C" int nb_compute_var_map(nb_variable_rec *variable, int64_t n_variable,
                                  const nb_factor_rec *factor, int64_t n_factor,
                                  const nb_ftv_rec *fmap, int64_t n_fmap, nb_vtf_rec *vmap,
                                  int64_t n_vmap, int64_t *factor_index, int64_t n_factor_index,
                                  const uint8_t *domain_mask, const int64_t *factors_to_skip,
                                  int64_t n_skip)
{
    std::atomic<int> bad(0);
    char msg[200] = "";
    auto fail = [&](const char *what, int64_t idx) {
        int expected = 0;
        if (bad.compare_exchange_strong(expected, 1)) snprintf(msg, sizeof(msg), "%s (index %lld)", what, (long long)idx);
    };
    // :20-30 implicit domains
    for (int64_t i = 0; i < n_variable; i++) {
        const nb_variable_rec &v = variable[i];
        if (v.dataType == 0) {
            if (v.vtf_offset < 0 || v.vtf_offset >= n_vmap) NB_FAIL(NB_ERR_INVALID, "variable %lld: vmap offset out of bounds", (long long)i);
            continue;
        }
        if (v.vtf_offset < 0 || v.cardinality < 0 || v.vtf_offset + v.cardinality > n_vmap)
            NB_FAIL(NB_ERR_INVALID, "variable %lld: vmap range out of bounds", (long long)i);
        if (domain_mask && domain_mask[i]) continue;
        for (int64_t k = 0; k < v.cardinality; k++) vmap[v.vtf_offset + k].value = k;
    }
    // skip list -> flag per factor
    std::vector<uint8_t> skip;
    if (n_skip > 0) {
        skip.assign((size_t)n_factor, 0);
        for (int64_t s = 0; s < n_skip; s++) {
            int64_t i = factors_to_skip[s];
            if (i < 0 || i >= n_factor || (s > 0 && factors_to_skip[s - 1] >= i))
                NB_FAIL(NB_ERR_INVALID, "factors_to_skip must be sorted, unique and in range");
            skip[(size_t)i] = 1;
        }
    }
    // :33-38 bucket lengths.  The reference also counts the entries of skipped factors and then
    // never writes their slots, which leaves stale ids in the buckets (and overruns factor_index);
    // here skipped factors simply occupy no bucket space.  With an empty skip list the result is
    // identical to the reference's.
    for (int64_t f = 0; f < n_factor; f++)
        if (factor[f].ftv_offset < 0 || factor[f].arity < 0 || factor[f].ftv_offset + factor[f].arity > n_fmap)
            NB_FAIL(NB_ERR_INVALID, "factor %lld: fmap range out of bounds", (long long)f);
    if (n_skip == 0 && !getenv("NUMBSKULL_B200_VARMAP_GENERAL")) {
        int bad_graph = 0;
        if (var_map_partitioned(variable, n_variable, factor, n_factor, fmap, n_fmap, vmap, n_vmap, factor_index,
                                n_factor_index, &bad_graph, msg, sizeof(msg))) {
            if (bad_graph) NB_FAIL(NB_ERR_INVALID, "invalid factor graph: %s", msg);
            return NB_OK;
        }
    }
    host_threads(n_fmap, [&](int64_t a, int64_t b) {
        for (int64_t j = a; j < b; j++) {
            const nb_ftv_rec &m = fmap[j];
            if (m.vid < 0 || m.vid >= n_variable) { fail("fmap vid out of range", j); continue; }
            const nb_variable_rec &v = variable[m.vid];
            if (v.dataType == 1 && (m.dense_equal_to < 0 || m.dense_equal_to >= v.cardinality)) {
                fail("fmap dense_equal_to outside the variable's cardinality", j);
                continue;
            }
            atomic_fetch_add_i64(&vmap[bucket_of(variable, m)].factor_index_length, 1);
        }
    });
    if (bad.load()) NB_FAIL(NB_ERR_INVALID, "invalid factor graph: %s", msg);
    if (n_skip > 0)
        for (int64_t s = 0; s < n_skip; s++) {
            const nb_factor_rec &f = factor[factors_to_skip[s]];
            for (int64_t j = f.ftv_offset; j < f.ftv_offset + f.arity; j++)
                vmap[bucket_of(variable, fmap[j])].factor_index_length -= 1;
        }
    // :40-46 exclusive scan
    int64_t last_len = 0, last_off = 0;
    for (int64_t i = 0; i < n_vmap; i++) {
        vmap[i].factor_index_offset = last_off + last_len;
        last_len = vmap[i].factor_index_length;
        last_off = vmap[i].factor_index_offset;
    }
    if (last_off + last_len > n_factor_index)
        NB_FAIL(NB_ERR_INVALID,
                "factor_index holds %lld entries but the buckets need %lld (the reference overruns "
                "here when factors_to_skip is non-empty)",
                (long long)n_factor_index, (long long)(last_off + last_len));
    // :48-65 scatter (bucket cursors advanced atomically; order inside a bucket is fixed by the sort below)
    std::vector<int64_t> cursor((size_t)n_vmap);
    for (int64_t i = 0; i < n_vmap; i++) cursor[(size_t)i] = vmap[i].factor_index_offset;
    host_threads(n_factor, [&](int64_t a, int64_t b) {
        for (int64_t i = a; i < b; i++) {
            if (!skip.empty() && skip[(size_t)i]) continue;
            const nb_factor_rec &f = factor[i];
            for (int64_t j = f.ftv_offset; j < f.ftv_offset + f.arity; j++)
                factor_index[atomic_fetch_add_i64(&cursor[(size_t)bucket_of(variable, fmap[j])], 1)] = i;
        }
    });
    // :67-81 sort + unique each bucket; offsets are not compacted
    host_threads(n_vmap, [&](int64_t a, int64_t b) {
        for (int64_t i = a; i < b; i++) {
            int64_t off = vmap[i].factor_index_offset, len = vmap[i].factor_index_length;
            int64_t *p = factor_index + off;
            if (!std::is_sorted(p, p + len)) std::sort(p, p + len);
            int64_t n = 0, last = -1;
            for (int64_t k = 0; k < len; k++) {
                if (p[k] == last) continue;
                last = p[k];
                p[n++] = last;
            }
            vmap[i].factor_index_length = n;
        }
    });
    return NB_OK;
}

// ---------------------------------------------------------------------------
// Big-endian readers for the DeepDive binary graph files.
// ---------------------------------------------------------------------------
static inline uint64_t be64(const uint8_t *p)
{
    uint64_t x;
    memcpy(&x, p, 8);
    return __builtin_bswap64(x);
}
static inline uint16_t be16(const uint8_t *p) { return (uint16_t)((p[0] << 8) | p[1]); }
static inline double be_f64(const uint8_t *p)
{
    uint64_t x = be64(p);
    double d;
    memcpy(&d, &x, 8);
    return d;
}

// dataloading.py:103-123: 17-byte records (int64 weightId, u8 isFixed, f64 initialValue).
// Fixed-width records: parsed by host threads (every id occurs once, so the writes do not collide).
extern "C" int nb_load_weights(const uint8_t *data, int64_t n_bytes, int64_t n_weight, nb_weight_rec *out)
{
    if (n_bytes < 17 * n_weight) NB_FAIL(NB_ERR_INVALID, "graph.weights: %lld bytes < %lld records", (long long)n_bytes, (long long)n_weight);
    std::atomic<int64_t> bad(-1);
    host_threads(n_weight, [&](int64_t a, int64_t b) {
        for (int64_t i = a; i < b; i++) {
            const uint8_t *r = data + 17 * i;
            int64_t id = (int64_t)be64(r);
            if (id < 0 || id >= n_weight) { bad.store(id); continue; }
            out[id].isFixed = r[8];
            out[id].initialValue = be_f64(r + 9);
        }
    });
    if (bad.load() != -1) NB_FAIL(NB_ERR_INVALID, "graph.weights: weightId %lld out of range", (long long)bad.load());
    return NB_OK;
}

// dataloading.py:126-156: 27-byte records (int64 id, i8 isEvidence, int64 initialValue,
// int16 dataType, int64 cardinality)
extern "C" int nb_load_variables(const uint8_t *data, int64_t n_bytes, int64_t n_variable, nb_variable_rec *out)
{
    if (n_bytes < 27 * n_variable) NB_FAIL(NB_ERR_INVALID, "graph.variables: %lld bytes < %lld records", (long long)n_bytes, (long long)n_variable);
    std::atomic<int64_t> bad(-1);
    host_threads(n_variable, [&](int64_t a, int64_t b) {
        for (int64_t i = a; i < b; i++) {
            const uint8_t *r = data + 27 * i;
            int64_t id = (int64_t)be64(r);
            if (id < 0 || id >= n_variable) { bad.store(id); continue; }
            out[id].isEvidence = (int8_t)r[8];
            out[id].initialValue = (int64_t)be64(r + 9);
            out[id].dataType = (int16_t)be16(r + 17);
            out[id].cardinality = (int64_t)be64(r + 19);
        }
    });
    if (bad.load() != -1) NB_FAIL(NB_ERR_INVALID, "graph.variables: variableId %lld out of range", (long long)bad.load());
    return NB_OK;
}

// dataloading.py:159-187: (int64 variableId, int64 cardinality, cardinality x int64 value);
// marks the variable, stores the (sorted) domain in vmap[].value and rewrites
// initialValue to its dense index.
extern "C" int nb_load_domains(const uint8_t *data, int64_t n_bytes, uint8_t *domain_mask, nb_vtf_rec *vmap,
                               int64_t n_vmap, nb_variable_rec *variable, int64_t n_variable)
{
    int64_t idx = 0;
    while (idx < n_bytes) {
        if (idx + 16 > n_bytes) NB_FAIL(NB_ERR_INVALID, "graph.domains: truncated header");
        int64_t vid = (int64_t)be64(data + idx);
        int64_t card = (int64_t)be64(data + idx + 8);
        idx += 16;
        if (vid < 0 || vid >= n_variable) NB_FAIL(NB_ERR_INVALID, "graph.domains: variableId %lld out of range", (long long)vid);
        if (card < 0 || idx + 8 * card > n_bytes || variable[vid].vtf_offset + card > n_vmap)
            NB_FAIL(NB_ERR_INVALID, "graph.domains: bad cardinality for variable %lld", (long long)vid);
        domain_mask[vid] = 1;
        for (int64_t j = 0; j < card; j++) {
            int64_t val = (int64_t)be64(data + idx);
            idx += 8;
            vmap[variable[vid].vtf_offset + j].value = val;
            if (val == variable[vid].initialValue) variable[vid].initialValue = j;
        }
    }
    return NB_OK;
}

// dataloading.py:190-237: variable-length records
// (int16 func, int64 arity, arity x (int64 vid, int64 value), int64 weightId, f64 feature);
// values of variables with an explicit domain are translated to dense indices by
// binary search over vmap[].value (np.searchsorted, side='left').
// Two passes: a sequential scan that only reads the arity of every record (record start and
// ftv_offset are running sums: 26 + 16 arity bytes and arity entries per record), then the bodies
// are decoded by host threads.  Same output as the reference's one-pass loop.
extern "C" int nb_load_factors(const uint8_t *data, int64_t n_bytes, int64_t n_factor, nb_factor_rec *factor,
                               nb_ftv_rec *fmap, int64_t n_fmap, const uint8_t *domain_mask,
                               const nb_variable_rec *variable, int64_t n_variable, const nb_vtf_rec *vmap,
                               int64_t n_vmap)
{
    std::vector<int64_t> start((size_t)n_factor + 1);
    {
        int64_t idx = 0, e = 0;
        for (int64_t i = 0; i < n_factor; i++) {
            if (idx + 10 > n_bytes) NB_FAIL(NB_ERR_INVALID, "graph.factors: truncated at factor %lld", (long long)i);
            const int64_t arity = (int64_t)be64(data + idx + 2);
            if (arity < 0 || arity > n_fmap || idx + 26 + 16 * arity > n_bytes || e + arity > n_fmap)
                NB_FAIL(NB_ERR_INVALID, "graph.factors: factor %lld has bad arity %lld", (long long)i, (long long)arity);
            start[(size_t)i] = idx;
            factor[i].arity = arity;
            factor[i].ftv_offset = e;
            idx += 26 + 16 * arity;
            e += arity;
        }
        start[(size_t)n_factor] = idx;
    }
    std::atomic<int64_t> bad_factor(-1), bad_vid(0);
    std::atomic<int> bad_kind(0);
    host_threads(n_factor, [&](int64_t a, int64_t b) {
        for (int64_t i = a; i < b; i++) {
            const uint8_t *r = data + start[(size_t)i];
            const int64_t arity = factor[i].arity, e = factor[i].ftv_offset;
            factor[i].factorFunction = (int16_t)be16(r);
            r += 10;
            for (int64_t k = 0; k < arity; k++, r += 16) {
                int64_t vid = (int64_t)be64(r);
                int64_t val = (int64_t)be64(r + 8);
                if (vid < 0 || vid >= n_variable) { bad_factor.store(i); bad_vid.store(vid); bad_kind.store(1); vid = 0; val = 0; }
                else if (domain_mask && domain_mask[vid]) {
                    int64_t s = variable[vid].vtf_offset, n = variable[vid].cardinality;
                    if (s < 0 || s + n > n_vmap) { bad_factor.store(i); bad_vid.store(vid); bad_kind.store(2); n = 0; }
                    int64_t lo = 0, hi = n;
                    while (lo < hi) {
                        int64_t mid = (lo + hi) / 2;
                        if (vmap[s + mid].value < val) lo = mid + 1; else hi = mid;
                    }
                    val = lo;
                }
                fmap[e + k].vid = vid;
                fmap[e + k].dense_equal_to = val;
            }
            factor[i].weightId = (int64_t)be64(r);
            factor[i].featureValue = be_f64(r + 8);
        }
    });
    if (bad_kind.load() == 1)
        NB_FAIL(NB_ERR_INVALID, "graph.factors: factor %lld references variable %lld", (long long)bad_factor.load(), (long long)bad_vid.load());
    if (bad_kind.load() == 2)
        NB_FAIL(NB_ERR_INVALID, "graph.factors: domain of variable %lld out of range", (long long)bad_vid.load());
    return NB_OK;
}

// ---------------------------------------------------------------------------
// Benchmark input generator (BASELINE config 4, SURVEY.md section 8d): the KBC-style Boolean graph
// of numbskull_b200/synth.py kbc(), filled by host threads straight into the reference's packed
// record arrays.  Counter-based randomness (splitmix64 of (seed, stream, index)): the graph does
// not depend on the thread count, and any owner block of it can be generated on its own
// (nb_synth_kbc_block: partitioned runs never materialise the 1 B-edge graph).  Not part of the
// hot path: it only feeds it (the role ising/ising.cpp plays for the reference).
// ---------------------------------------------------------------------------
static inline uint64_t sm64(uint64_t x)
{
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}
static inline uint64_t rnd(uint64_t seed, uint64_t stream, uint64_t i) { return sm64(sm64(seed ^ (stream * 0xD1342543DE82EF95ull)) + i); }
static inline double unit(uint64_t r) { return (double)(r >> 11) * (1.0 / 9007199254740992.0); }

struct KbcShape {
    int64_t nvar, n_imp, n_and, n_or, nhub, window, n_weights;
    uint64_t seed;
    double far_frac, hub_frac, log1mp;
    int64_t n_factor() const { return nvar + n_imp + n_and + n_or; }
};

static KbcShape kbc_shape(int64_t nvar, uint64_t seed, int64_t n_weights, int64_t window, double far_frac, double hub_frac,
                          const double *mix3)
{
    KbcShape S;
    S.nvar = nvar; S.seed = seed; S.n_weights = n_weights; S.window = window; S.far_frac = far_frac; S.hub_frac = hub_frac;
    S.n_imp = (int64_t)(nvar * mix3[0]); S.n_and = (int64_t)(nvar * mix3[1]); S.n_or = (int64_t)(nvar * mix3[2]);
    S.nhub = std::max<int64_t>(1, (int64_t)(nvar * 1e-5));
    S.log1mp = std::log1p(-1.0 / std::max(2.0, (double)window / 8.0));
    return S;
}

// factor f: [0, nvar) ISTRUE(v = f); then IMPLY_NATURAL arity 3, AND arity 2, OR arity 3.  Members: an
// anchor plus geometric-window partners (local), uniform partners (far) or Zipf-like hubs.
static inline int kbc_factor(const KbcShape &S, int64_t f, int &func, int64_t m[3])
{
    int arity;
    if (f < S.nvar) { func = 4; m[0] = f; return 1; }
    else if (f < S.nvar + S.n_imp) { func = 0; arity = 3; }
    else if (f < S.nvar + S.n_imp + S.n_and) { func = 2; arity = 2; }
    else { func = 1; arity = 3; }
    const int64_t anchor = (int64_t)(rnd(S.seed, 6, (uint64_t)f) % (uint64_t)S.nvar);
    m[0] = anchor;
    for (int j = 1; j < arity; j++) {
        const uint64_t k = (uint64_t)f * 4 + (uint64_t)j;
        if (unit(rnd(S.seed, 7, k)) < S.hub_frac) {                 // P(rank >= x) = x^-(a-1), a = 1.5
            const double u = std::max(unit(rnd(S.seed, 8, k)), 1e-12);
            const int64_t rank = std::min<int64_t>(S.nhub - 1, (int64_t)(1.0 / (u * u)) - 1);
            m[j] = (int64_t)(rnd(S.seed, 9, (uint64_t)rank) % (uint64_t)S.nvar);
        } else if (unit(rnd(S.seed, 10, k)) < S.far_frac) {
            m[j] = (int64_t)(rnd(S.seed, 11, k) % (uint64_t)S.nvar);
        } else {
            const double u = std::max(unit(rnd(S.seed, 12, k)), 1e-300);
            int64_t d = std::min<int64_t>(S.window, 1 + (int64_t)(std::log(u) / S.log1mp));   // geometric, capped
            if (rnd(S.seed, 13, k) & 1u) d = -d;
            m[j] = ((anchor + d) % S.nvar + S.nvar) % S.nvar;
        }
    }
    return arity;
}

static inline void kbc_factor_rec(const KbcShape &S, int64_t f, int func, int arity, int64_t off, nb_factor_rec &r)
{
    r.factorFunction = (int16_t)func;
    r.weightId = (int64_t)((((uint64_t)f * 0x9E3779B97F4A7C15ull) >> 40) % (uint64_t)S.n_weights);
    r.featureValue = 1.0;
    r.arity = arity;
    r.ftv_offset = off;
}

static inline void kbc_variable_rec(uint64_t seed, double evidence_frac, int64_t gid, nb_variable_rec &v)
{
    const bool ev = unit(rnd(seed, 4, (uint64_t)gid)) < evidence_frac;
    v.isEvidence = ev ? 1 : 0;
    v.initialValue = ev ? (int64_t)(rnd(seed, 5, (uint64_t)gid) & 1u) : 0;
    v.dataType = 0;
    v.cardinality = 2;
    v.vtf_offset = 0;
}

extern "C" int nb_synth_kbc_weights(uint64_t seed, int64_t n_weights, double fixed_frac, nb_weight_rec *weight)
{
    host_threads(n_weights, [&](int64_t a, int64_t b) {
        for (int64_t i = a; i < b; i++) {
            weight[i].isFixed = unit(rnd(seed, 1, (uint64_t)i)) < fixed_frac;
            // N(0, 0.5) by Box-Muller
            const double u1 = std::max(unit(rnd(seed, 2, (uint64_t)i)), 1e-300), u2 = unit(rnd(seed, 3, (uint64_t)i));
            weight[i].initialValue = 0.5 * std::sqrt(-2.0 * std::log(u1)) * std::cos(6.283185307179586 * u2);
        }
    });
    return NB_OK;
}

// variable records of the listed global ids (gids == NULL: ids 0 .. n-1)
extern "C" int nb_synth_kbc_variables(uint64_t seed, double evidence_frac, const int64_t *gids, int64_t n,
                                      nb_variable_rec *variable)
{
    host_threads(n, [&](int64_t a, int64_t b) {
        for (int64_t i = a; i < b; i++) kbc_variable_rec(seed, evidence_frac, gids ? gids[i] : i, variable[i]);
    });
    return NB_OK;
}

extern "C" int nb_synth_kbc(int64_t nvar, uint64_t seed, int64_t n_weights, double evidence_frac, int64_t window,
                            double far_frac, double hub_frac, double fixed_frac, const double *mix3,
                            nb_weight_rec *weight, nb_variable_rec *variable, nb_factor_rec *factor, int64_t n_factor,
                            nb_ftv_rec *fmap, int64_t n_fmap)
{
    const KbcShape S = kbc_shape(nvar, seed, n_weights, window, far_frac, hub_frac, mix3);
    if (n_factor != S.n_factor() || n_fmap != nvar + 3 * S.n_imp + 2 * S.n_and + 3 * S.n_or)
        NB_FAIL(NB_ERR_INVALID, "nb_synth_kbc: array sizes do not match the mix");
    nb_synth_kbc_weights(seed, n_weights, fixed_frac, weight);
    nb_synth_kbc_variables(seed, evidence_frac, nullptr, nvar, variable);
    host_threads(n_factor, [&](int64_t a, int64_t b) {
        for (int64_t f = a; f < b; f++) {
            int func;
            int64_t m[3], off;
            const int arity = kbc_factor(S, f, func, m);
            if (f < nvar) off = f;
            else if (f < nvar + S.n_imp) off = nvar + 3 * (f - nvar);
            else if (f < nvar + S.n_imp + S.n_and) off = nvar + 3 * S.n_imp + 2 * (f - nvar - S.n_imp);
            else off = nvar + 3 * S.n_imp + 2 * S.n_and + 3 * (f - nvar - S.n_imp - S.n_and);
            kbc_factor_rec(S, f, func, arity, off, factor[f]);
            for (int j = 0; j < arity; j++) { fmap[off + j].vid = m[j]; fmap[off + j].dense_equal_to = 0; }
        }
    });
    return NB_OK;
}

// The factors with at least one member in the owner block [lo, hi), in increasing global factor id,
// members as GLOBAL variable ids.  Call with factor == NULL to size the arrays (*n_factor, *n_fmap
// are outputs), then again to fill them (*n_factor, *n_fmap are the sizes returned before).
extern "C" int nb_synth_kbc_block(int64_t nvar, uint64_t seed, int64_t n_weights, int64_t window, double far_frac,
                                  double hub_frac, const double *mix3, int64_t lo, int64_t hi, nb_factor_rec *factor,
                                  int64_t *n_factor, nb_ftv_rec *fmap, int64_t *n_fmap)
{
    const KbcShape S = kbc_shape(nvar, seed, n_weights, window, far_frac, hub_frac, mix3);
    const int64_t F = S.n_factor();
    const int nt = (int)std::min(32u, std::max(1u, std::thread::hardware_concurrency()));
    const int64_t chunk = (F + nt - 1) / nt;
    std::vector<int64_t> cf((size_t)nt + 1, 0), ce((size_t)nt + 1, 0);
    auto touches = [&](const int64_t *m, int arity) {
        for (int j = 0; j < arity; j++) if (m[j] >= lo && m[j] < hi) return true;
        return false;
    };
    run_threads(nt, [&](int t) {
        int64_t nf = 0, ne = 0;
        for (int64_t f = t * chunk; f < std::min(F, (t + 1) * chunk); f++) {
            int func;
            int64_t m[3];
            const int arity = kbc_factor(S, f, func, m);
            if (touches(m, arity)) { nf++; ne += arity; }
        }
        cf[(size_t)t + 1] = nf;
        ce[(size_t)t + 1] = ne;
    });
    for (int t = 0; t < nt; t++) { cf[(size_t)t + 1] += cf[(size_t)t]; ce[(size_t)t + 1] += ce[(size_t)t]; }
    if (!factor) { *n_factor = cf[(size_t)nt]; *n_fmap = ce[(size_t)nt]; return NB_OK; }
    if (*n_factor != cf[(size_t)nt] || *n_fmap != ce[(size_t)nt]) NB_FAIL(NB_ERR_INVALID, "nb_synth_kbc_block: sizes changed between the calls");
    run_threads(nt, [&](int t) {
        int64_t nf = cf[(size_t)t], ne = ce[(size_t)t];
        for (int64_t f = t * chunk; f < std::min(F, (t + 1) * chunk); f++) {
            int func;
            int64_t m[3];
            const int arity = kbc_factor(S, f, func, m);
            if (!touches(m, arity)) continue;
            kbc_factor_rec(S, f, func, arity, ne, factor[nf]);
            for (int j = 0; j < arity; j++) { fmap[ne + j].vid = m[j]; fmap[ne + j].dense_equal_to = 0; }
            nf++;
            ne += arity;
        }
    });
    return NB_OK;
}

// Ghost set of an owner block [lo, hi) and the translation of a rank-local fmap to local ids
// (owned variable v -> v - lo, ghost -> n_owned + its rank among the ghosts, ascending global id):
// what partition.extract_local does with numpy's unique / searchsorted, which takes a minute and
// a half on the 600 M members of a 2-GPU cut of the 1 B-edge graph.  A bitmap over the global ids
// and per-word prefix counts instead of a sort.  Call with ghosts == NULL for the count, then with
// a buffer of that size; rewrite != 0 also rewrites fmap[].vid.
extern "C" int nb_block_ghosts(nb_ftv_rec *fmap, int64_t n_fmap, int64_t nvar, int64_t lo, int64_t hi, int64_t *ghosts,
                               int64_t *n_ghosts, int rewrite)
{
    if (!fmap && n_fmap) NB_FAIL(NB_ERR_INVALID, "nb_block_ghosts: fmap is NULL");
    if (lo < 0 || hi < lo || hi > nvar) NB_FAIL(NB_ERR_INVALID, "nb_block_ghosts: bad block [%lld, %lld) of %lld", (long long)lo, (long long)hi, (long long)nvar);
    const int64_t words = (nvar + 63) / 64;
    std::vector<std::atomic<uint64_t>> bits((size_t)words);
    const int nt = (int)std::min(32u, std::max(1u, std::thread::hardware_concurrency()));
    std::atomic<int> bad{0};
    run_threads(nt, [&](int t) {
        for (int64_t w = words * t / nt; w < words * (t + 1) / nt; w++) bits[(size_t)w].store(0, std::memory_order_relaxed);
    });
    run_threads(nt, [&](int t) {
        for (int64_t i = n_fmap * t / nt; i < n_fmap * (t + 1) / nt; i++) {
            const int64_t v = fmap[i].vid;
            if (v < 0 || v >= nvar) { bad.store(1); continue; }
            if (v >= lo && v < hi) continue;
            const uint64_t m = 1ull << (v & 63);
            if (!(bits[(size_t)(v >> 6)].load(std::memory_order_relaxed) & m)) bits[(size_t)(v >> 6)].fetch_or(m, std::memory_order_relaxed);
        }
    });
    if (bad.load()) NB_FAIL(NB_ERR_INVALID, "nb_block_ghosts: a member id is outside [0, %lld)", (long long)nvar);
    std::vector<int64_t> pre((size_t)words + 1, 0);
    std::vector<int64_t> part((size_t)nt + 1, 0);
    run_threads(nt, [&](int t) {
        int64_t c = 0;
        for (int64_t w = words * t / nt; w < words * (t + 1) / nt; w++) c += __builtin_popcountll(bits[(size_t)w].load(std::memory_order_relaxed));
        part[(size_t)t + 1] = c;
    });
    for (int t = 0; t < nt; t++) part[(size_t)t + 1] += part[(size_t)t];
    const int64_t total = part[(size_t)nt];
    if (!ghosts) { *n_ghosts = total; return NB_OK; }
    if (*n_ghosts != total) NB_FAIL(NB_ERR_INVALID, "nb_block_ghosts: the ghost count changed between the calls");
    run_threads(nt, [&](int t) {
        int64_t c = part[(size_t)t];
        for (int64_t w = words * t / nt; w < words * (t + 1) / nt; w++) {
            pre[(size_t)w] = c;
            uint64_t x = bits[(size_t)w].load(std::memory_order_relaxed);
            while (x) { ghosts[c++] = w * 64 + __builtin_ctzll(x); x &= x - 1; }
        }
    });
    if (rewrite) {
        const int64_t n_owned = hi - lo;
        run_threads(nt, [&](int t) {
            for (int64_t i = n_fmap * t / nt; i < n_fmap * (t + 1) / nt; i++) {
                const int64_t v = fmap[i].vid;
                if (v >= lo && v < hi) { fmap[i].vid = v - lo; continue; }
                const uint64_t x = bits[(size_t)(v >> 6)].load(std::memory_order_relaxed) & ((1ull << (v & 63)) - 1);
                fmap[i].vid = n_owned + pre[(size_t)(v >> 6)] + __builtin_popcountll(x);
            }
        });
    }
    return NB_OK;
}

// partition.extract_local_by_owner in host threads: the share of rank `rank` under the placement
// owner[v] -- every factor with an owned member (factor order kept, ftv_offset renumbered), its
// members as local ids (owned variables first in ascending global id, then the ghosts in ascending
// global id), and the global id of every local variable.  Two calls: loc_factor == NULL returns the
// four counts.  Bitmaps + prefix popcounts, no sort (the numpy version needs ~1 us per variable and
// several 8-byte temporaries per fmap entry).
extern "C" int nb_extract_local(const nb_factor_rec *factor, int64_t n_factor, const nb_ftv_rec *fmap, int64_t n_fmap,
                                const int32_t *owner, int64_t nvar, int32_t rank, int64_t *n_loc_factor, int64_t *n_loc_fmap,
                                int64_t *n_owned, int64_t *n_ghost, nb_factor_rec *loc_factor, nb_ftv_rec *loc_fmap,
                                int64_t *global_vid)
{
    if ((!factor && n_factor) || (!fmap && n_fmap) || (!owner && nvar)) NB_FAIL(NB_ERR_INVALID, "nb_extract_local: NULL input");
    const int nt = (int)std::min(32u, std::max(1u, std::thread::hardware_concurrency()));
    const int64_t words = (nvar + 63) / 64;
    std::vector<std::atomic<uint64_t>> ghost((size_t)words);
    std::vector<uint64_t> mine((size_t)words, 0);
    std::vector<uint8_t> keep((size_t)n_factor, 0);
    std::vector<int64_t> cf((size_t)nt + 1, 0), ce((size_t)nt + 1, 0);
    std::atomic<int> bad{0};
    run_threads(nt, [&](int t) {
        for (int64_t w = words * t / nt; w < words * (t + 1) / nt; w++) {
            ghost[(size_t)w].store(0, std::memory_order_relaxed);
            uint64_t m = 0;
            for (int64_t v = w * 64; v < std::min(nvar, w * 64 + 64); v++)
                if (owner[v] == rank) m |= 1ull << (v & 63);
            mine[(size_t)w] = m;
        }
    });
    // kept factors and their ghost members
    run_threads(nt, [&](int t) {
        int64_t nf = 0, ne = 0;
        for (int64_t f = n_factor * t / nt; f < n_factor * (t + 1) / nt; f++) {
            const int64_t a = factor[f].arity, o = factor[f].ftv_offset;
            if (a < 0 || o < 0 || o + a > n_fmap) { bad.store(1); continue; }
            bool k = false;
            for (int64_t j = 0; j < a; j++) {
                const int64_t v = fmap[o + j].vid;
                if (v < 0 || v >= nvar) { bad.store(1); k = false; break; }
                if (owner[v] == rank) k = true;
            }
            if (!k) continue;
            keep[(size_t)f] = 1;
            nf++;
            ne += a;
            for (int64_t j = 0; j < a; j++) {
                const int64_t v = fmap[o + j].vid;
                if (owner[v] != rank) {
                    const uint64_t m = 1ull << (v & 63);
                    if (!(ghost[(size_t)(v >> 6)].load(std::memory_order_relaxed) & m)) ghost[(size_t)(v >> 6)].fetch_or(m, std::memory_order_relaxed);
                }
            }
        }
        cf[(size_t)t + 1] = nf;
        ce[(size_t)t + 1] = ne;
    });
    if (bad.load()) NB_FAIL(NB_ERR_INVALID, "nb_extract_local: a factor's members lie outside fmap or a member id outside [0, %lld)", (long long)nvar);
    for (int t = 0; t < nt; t++) { cf[(size_t)t + 1] += cf[(size_t)t]; ce[(size_t)t + 1] += ce[(size_t)t]; }
    // prefix popcounts of both bitmaps
    std::vector<int64_t> pm((size_t)words + 1, 0), pg((size_t)words + 1, 0), tm((size_t)nt + 1, 0), tg((size_t)nt + 1, 0);
    run_threads(nt, [&](int t) {
        int64_t a = 0, b = 0;
        for (int64_t w = words * t / nt; w < words * (t + 1) / nt; w++) {
            a += __builtin_popcountll(mine[(size_t)w]);
            b += __builtin_popcountll(ghost[(size_t)w].load(std::memory_order_relaxed));
        }
        tm[(size_t)t + 1] = a;
        tg[(size_t)t + 1] = b;
    });
    for (int t = 0; t < nt; t++) { tm[(size_t)t + 1] += tm[(size_t)t]; tg[(size_t)t + 1] += tg[(size_t)t]; }
    const int64_t no = tm[(size_t)nt], ng = tg[(size_t)nt];
    if (!loc_factor) {
        *n_loc_factor = cf[(size_t)nt]; *n_loc_fmap = ce[(size_t)nt]; *n_owned = no; *n_ghost = ng;
        return NB_OK;
    }
    if (*n_loc_factor != cf[(size_t)nt] || *n_loc_fmap != ce[(size_t)nt] || *n_owned != no || *n_ghost != ng)
        NB_FAIL(NB_ERR_INVALID, "nb_extract_local: the counts changed between the calls");
    run_threads(nt, [&](int t) {
        int64_t a = tm[(size_t)t], b = tg[(size_t)t];
        for (int64_t w = words * t / nt; w < words * (t + 1) / nt; w++) {
            pm[(size_t)w] = a;
            pg[(size_t)w] = b;
            uint64_t x = mine[(size_t)w];
            while (x) { global_vid[a++] = w * 64 + __builtin_ctzll(x); x &= x - 1; }
            x = ghost[(size_t)w].load(std::memory_order_relaxed);
            while (x) { global_vid[no + b++] = w * 64 + __builtin_ctzll(x); x &= x - 1; }
        }
    });
    run_threads(nt, [&](int t) {
        int64_t nf = cf[(size_t)t], ne = ce[(size_t)t];
        for (int64_t f = n_factor * t / nt; f < n_factor * (t + 1) / nt; f++) {
            if (!keep[(size_t)f]) continue;
            const int64_t a = factor[f].arity, o = factor[f].ftv_offset;
            loc_factor[nf] = factor[f];
            loc_factor[nf].ftv_offset = ne;
            for (int64_t j = 0; j < a; j++) {
                const int64_t v = fmap[o + j].vid;
                const uint64_t below = (1ull << (v & 63)) - 1;
                loc_fmap[ne + j].vid = owner[v] == rank
                    ? pm[(size_t)(v >> 6)] + __builtin_popcountll(mine[(size_t)(v >> 6)] & below)
                    : no + pg[(size_t)(v >> 6)] + __builtin_popcountll(ghost[(size_t)(v >> 6)].load(std::memory_order_relaxed) & below);
                loc_fmap[ne + j].dense_equal_to = fmap[o + j].dense_equal_to;
            }
            nf++;
            ne += a;
        }
    });
    return NB_OK;
}
