// Chromatic Gibbs sweep (inference.py:10-71 gibbsthread / draw_sample /
// potential) and the potential() parity hook.
//
// One launch per (colour, row class).  Thread path: one variable per thread,
// rows read from the SELL-32 stream so that the 32 lanes of a warp load 32
// consecutive words at every step.  Warp path: one long row per warp, lanes
// stride over its incidences and the per-value energies are reduced with
// shuffles (shared memory for categorical rows).
#include "nb_eval.cuh"

// T = element type of the value arrays (nb_val_t or nb_val16_t, see nb_graph::value_bytes)
template <class T>
struct SweepArgs : NbCardOf<T> {   // (cardinalities: a.card(meta, nid))
    const uint32_t *vmeta;
    const int64_t *slice_ptr;
    const uint32_t *twords;
    const int64_t *wrow_ptr;
    const uint32_t *wwords;
    const int64_t *inc_ptr;
    const uint2 *inc;
    const uint32_t *rng_id;
    const uint32_t *cstart;
    int32_t *count;
    int32_t *count_b;
    T *val;
    uint32_t *valbits;       // bit-packed mirror of val (nullptr: not in use), see nb_graph::d_valbits
    const double *weight;
    int64_t n_trows;
    uint64_t seed, epoch;
    int burnin, sample_evidence;
    // partitioned graphs with non-blocking halo pushes: neighbours' flags to wait for
    const volatile uint32_t *w_flags;
    const int32_t *w_neigh;
    int w_n;
    uint32_t w_phase;
    int *w_error;
};

// Prologue of every sweep kernel: ghost values may only be read once each neighbour rank has
// signalled the latest halo phase (its peer stores are fenced before the signal).
template <class T>
__device__ __forceinline__ void nb_wait_halo(const SweepArgs<T> &a)
{
    if (a.w_n == 0) return;
    if ((int)threadIdx.x < a.w_n) {
        const int r = a.w_neigh[threadIdx.x];
        const long long t0 = clock64();
        while ((int32_t)(a.w_flags[r] - a.w_phase) < 0) {
            if (clock64() - t0 > 20000000000ll) { *a.w_error = 1; break; }
        }
    }
    // the peer fenced its stores before the flag store; the acquire side is a system-scope fence in
    // the waiting threads before anybody reads a ghost slot
    __threadfence_system();
    __syncthreads();
}

template <class T>
static SweepArgs<T> sweep_args(nb_graph *g, int chain, int burnin, int sample_evidence, uint64_t seed, uint64_t epoch)
{
    SweepArgs<T> a;
    a.vmeta = g->d_vmeta; a.slice_ptr = g->d_slice_ptr; a.twords = g->d_twords;
    a.wrow_ptr = g->d_wrow_ptr; a.wwords = g->d_wwords; a.inc_ptr = g->d_inc_ptr; a.inc = g->d_inc;
    a.rng_id = g->d_rng_id; a.cstart = g->d_cstart; a.count = g->d_count; a.count_b = g->d_count_b; a.val = nb_vals<T>(g, chain);
    if constexpr (sizeof(T) > 1) a.vcard = g->d_vcard;
    a.valbits = (g->use_bits && chain == 0) ? g->d_valbits : nullptr;
    a.weight = g->d_weight; a.n_trows = g->n_trows; a.seed = seed; a.epoch = epoch;
    a.burnin = burnin; a.sample_evidence = sample_evidence;
    nb_p2p_wait_args(g, &a.w_flags, &a.w_neigh, &a.w_n, &a.w_phase, &a.w_error);
    return a;
}

// cardinality of new id nid
template <class T>
__device__ __forceinline__ int nb_card(const SweepArgs<T> &a, uint32_t meta, int64_t nid)
{
    return a.card(meta, (uint32_t)nid);
}

template <class T>
__device__ __forceinline__ void nb_tally(const SweepArgs<T> &a, int64_t nid, int card, int k)
{
    if (a.burnin) return;
    uint32_t cs = a.cstart[nid];
    if (card == 2) a.count[cs] += k;       // inference.py:30-31
    else a.count[cs + k] += 1;             // :32-33
}

template <bool WIDE, class T>
__global__ void __launch_bounds__(256) k_gibbs_thread(SweepArgs<T> a, int beg, int end)
{
    nb_wait_halo(a);
    int64_t nid = (int64_t)beg + blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (nid >= end) return;
    const uint32_t meta = a.vmeta[nid];
    const int evid = NB_META_EVID(meta);
    if (!NB_META_VALID(meta) || evid == 4) return;          // inference.py:21-23
    if (!(evid == 0 || a.sample_evidence)) return;          // :24
    NbRow r = nb_thread_row(a.twords, a.slice_ptr, nid);
    NbUniforms rng(a.rng_id[nid], a.epoch, NB_TAG_FREE, a.seed);
    int k = nb_sample_row<WIDE>(r, NB_META_ROWLEN(meta), (uint32_t)nid, meta, a.val, a, a.weight, rng);
    a.val[nid] = (T)k;
    nb_tally(a, nid, nb_card(a, meta, nid), k);
}

// FAST rows: truth-table stream, one 16-byte quad per incidence (weight value inlined), uniform
// trip count per warp.  The energy difference comes from nb_tt_delta (nb_eval.cuh), the same
// function the parity hook nb_potentials_records evaluates.
#ifndef NB_TT_MINB
#define NB_TT_MINB 6      /* minimum CTAs per SM of k_gibbs_tt: 40 registers, 75 % occupancy (C4 50 M: 1.45 -> 1.35 ms per sweep) */
#endif
#ifndef NB_TT_UNROLL_SWEEP
#define NB_TT_UNROLL_SWEEP 4
#endif
// Publishes the draws of one warp (32 consecutive ids = one word) in the bit mirror.
__device__ __forceinline__ void nb_publish_bits(uint32_t *valbits, int64_t nid, bool sampled, int k)
{
    const unsigned m = __ballot_sync(0xFFFFFFFFu, sampled), b = __ballot_sync(0xFFFFFFFFu, sampled && k);
    if ((threadIdx.x & 31) == 0 && m) valbits[nid >> 5] = (valbits[nid >> 5] & ~m) | b;
}

template <int UNROLL, int MINB, bool BITS, class T>
__global__ void __launch_bounds__(256, MINB) k_gibbs_tt(SweepArgs<T> a, const int64_t *__restrict__ tt_ptr,
                                                        const uint4 *__restrict__ tt, int beg, int end, uint32_t key)
{
    nb_wait_halo(a);
    const int64_t nid0 = (int64_t)beg + blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (!BITS && nid0 >= end) return;
    const bool in = nid0 < end;
    const int64_t nid = in ? nid0 : (int64_t)end - 1;         // (BITS: whole warps stay for the ballot)
    // independent loads first: they overlap with the stream
    const uint32_t meta = nb_lds(a.vmeta + nid);
    const uint32_t rid = nb_lds(a.rng_id + nid);
    const int64_t q0 = nb_lds(tt_ptr + (nid >> 5)), q1 = nb_lds(tt_ptr + (nid >> 5) + 1);
    const int n = (int)((q1 - q0) >> 5);                      // incidences of the longest row of this slice
    const double d = BITS ? nb_tt_delta_v<UNROLL>(tt + q0 + (nid & 31), n, (uint32_t)nid, NbValsBits{a.valbits})
                          : nb_tt_delta_v<UNROLL>(tt + q0 + (nid & 31), n, (uint32_t)nid, NbValsBytes<T>{a.val});   // e1 - e0
    const int evid = NB_META_EVID(meta);
    // inference.py:21-24
    const bool sampled = in && NB_META_VALID(meta) && evid != 4 && (evid == 0 || a.sample_evidence);
    if (!BITS && !sampled) return;
    const double u = nb_philox2x32_u53(rid, (uint32_t)a.epoch, key);
    // P(0) = 1 / (1 + exp(e1 - e0)): draw_sample (inference.py:36-52) for cardinality 2
    const float p0 = 1.0f / (1.0f + __expf((float)d));
    const int k = u <= (double)p0 ? 0 : 1;
    if (sampled) {
        a.val[nid] = (T)k;
        if (!a.burnin && k) __stcs(a.count_b + nid, nb_lds(a.count_b + nid) + 1);   // inference.py:30-31
    }
    if (BITS) nb_publish_bits(a.valbits, nid0, sampled, k);
}

// PAIR rows: 8-byte records, two per quad -- or, in uniform slices, bare member ids, four per quad.
#ifndef NB_TT2_BLOCK
#define NB_TT2_BLOCK 128  /* threads per CTA of k_gibbs_tt2 (C2 4096^2, one B200: 128 threads 0.1574, 256 0.1638, 512 0.1800 ms per sweep) */
#endif
template <bool BITS, class T>
__global__ void __launch_bounds__(NB_TT2_BLOCK) k_gibbs_tt2(SweepArgs<T> a, const int64_t *__restrict__ tt2_ptr,
                                                   const uint32_t *__restrict__ tt2_common,
                                                   const uint4 *__restrict__ tt2, int beg, int end, uint32_t key)
{
    nb_wait_halo(a);
    const int64_t nid0 = (int64_t)beg + blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (!BITS && nid0 >= end) return;
    const bool in = nid0 < end;
    const int64_t nid = in ? nid0 : (int64_t)end - 1;
    const uint32_t meta = nb_lds(a.vmeta + nid);
    const uint32_t rid = nb_lds(a.rng_id + nid);
    const int64_t q0 = nb_lds(tt2_ptr + (nid >> 5)), q1 = nb_lds(tt2_ptr + (nid >> 5) + 1);
    const uint32_t common = nb_lds(tt2_common + (nid >> 5));
    const int n = (int)((q1 - q0) >> 5);                      // quads of the longest row of this slice
    const double d = BITS ? nb_tt2_delta_v(tt2 + q0 + (nid & 31), n, common, (uint32_t)nid, NbValsBits{a.valbits}, a.weight)
                          : nb_tt2_delta_v(tt2 + q0 + (nid & 31), n, common, (uint32_t)nid, NbValsBytes<T>{a.val}, a.weight);   // e1 - e0
    const int evid = NB_META_EVID(meta);
    const bool sampled = in && NB_META_VALID(meta) && evid != 4 && (evid == 0 || a.sample_evidence);   // inference.py:21-24
    if (!BITS && !sampled) return;
    const double u = nb_philox2x32_u53(rid, (uint32_t)a.epoch, key);
    const float p0 = 1.0f / (1.0f + __expf((float)d));
    const int k = u <= (double)p0 ? 0 : 1;
    if (sampled) {
        a.val[nid] = (T)k;
        // inference.py:30-31.  One writer per tally and colour, so the atomic adds what a load and a store
        // would, as a reduction the thread does not wait for (C2: 1.9 % less time per sweep)
        if (!a.burnin && k) atomicAdd(a.count_b + nid, 1);
    }
    if (BITS) nb_publish_bits(a.valbits, nid0, sampled, k);
}

// val -> bit mirror (all-Boolean graphs): one word per warp
__global__ void k_pack_bits(const nb_val_t *__restrict__ val, uint32_t *__restrict__ bits, int64_t n)
{
    const int64_t n32 = (n + 31) & ~31ll;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n32; i += (int64_t)gridDim.x * blockDim.x) {
        const unsigned b = __ballot_sync(0xFFFFFFFFu, i < n && val[i] != 0);
        if ((threadIdx.x & 31) == 0) bits[i >> 5] = b;
    }
}

int nb_pack_value_bits(nb_graph *g)
{
    const int64_t n = g->n_trows + g->n_wrows;
    k_pack_bits<<<(unsigned)std::min<int64_t>((n + 255) / 256, 148 * 16), 256, 0, g->stream>>>(nb_vals<nb_val_t>(g, 0), g->d_valbits, n);
    NB_CUDA(cudaGetLastError());
    return NB_OK;
}

// CAT rows: categorical variable (cardinality <= 32) with AND_CAT / EQUAL_CAT_CONST factors.  One
// quad per incidence, uniform trip count per warp; the per-value energies live in a column of
// shared memory private to the thread (no parsing, no divergence), then one inverse-CDF draw.
struct NbCatSmemAcc {
    float (*e)[256];
    int tid;
    __device__ __forceinline__ void add(int k, float w) { e[k][tid] += w; }
};

template <class T>
__global__ void __launch_bounds__(256) k_gibbs_cat(SweepArgs<T> a, const int64_t *__restrict__ cat_ptr,
                                                   const uint4 *__restrict__ cat, int64_t first_id, int beg, int end)
{
    __shared__ float s_e[NB_CAT_MAX_CARD][256];
    nb_wait_halo(a);
    const int64_t nid = (int64_t)beg + blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (nid >= end) return;
    const uint32_t meta = nb_lds(a.vmeta + nid);
    const uint32_t rid = nb_lds(a.rng_id + nid);
    const uint32_t cs = nb_lds(a.cstart + nid);
    const int card = NB_META_CARD(meta);       // CAT rows: card <= NB_CAT_MAX_CARD
    const int64_t s = (nid - first_id) >> 5;
    const int64_t q0 = nb_lds(cat_ptr + s), q1 = nb_lds(cat_ptr + s + 1);
    const int n = (int)((q1 - q0) >> 5);
    const int tid = threadIdx.x;
#pragma unroll 4
    for (int k = 0; k < card; k++) s_e[k][tid] = 0.0f;
    NbCatSmemAcc acc{s_e, tid};
    nb_cat_energies(cat + q0 + (nid & 31), n, (uint32_t)nid, a.val, acc);
    const int evid = NB_META_EVID(meta);
    if (!NB_META_VALID(meta) || evid == 4) return;          // inference.py:21-23
    if (!(evid == 0 || a.sample_evidence)) return;          // :24
    // draw_sample (inference.py:36-52) with the maximum subtracted
    float mx = s_e[0][tid];
    for (int k = 1; k < card; k++) mx = fmaxf(mx, s_e[k][tid]);
    float tot = 0.0f;
    for (int k = 0; k < card; k++) { float z = __expf(s_e[k][tid] - mx); s_e[k][tid] = z; tot += z; }
    const float t = (float)nb_philox2x32_u53(rid, (uint32_t)a.epoch, nb_fold_key(a.seed, a.epoch, NB_TAG_FREE)) * tot;
    float acc_z = 0.0f;
    int pick = card - 1;
    for (int k = 0; k < card; k++) {
        acc_z += s_e[k][tid];
        if (acc_z >= t) { pick = k; break; }
    }
    a.val[nid] = (T)pick;
    if (!a.burnin) {
        if (card == 2) a.count[cs] += pick;                  // inference.py:30-31
        else a.count[cs + pick] += 1;                        // :32-33
    }
}

// ---------------------------------------------------------------------------
// warp path
// ---------------------------------------------------------------------------
#define NB_WARPS_PER_BLOCK 8

// Energies of every value over incidences [i0, i1) of the warp row `wr`, lanes striding over
// them.  dataType 0, card <= 4: returned in e[] on all lanes.  Otherwise the per-value
// energies land in the warp's shared array se[0..card).
// (card <= NB_MAX_CARD: wider rows take nb_warp_sample_wide)
template <bool WIDE, class T>
__device__ inline void nb_warp_row_energies(const uint32_t *__restrict__ wwords, const int64_t *__restrict__ wrow_ptr,
                                            const uint2 *__restrict__ inc, int64_t i0, int64_t i1,
                                            int64_t wr, uint32_t self, uint32_t meta,
                                            const T *__restrict__ vals, const double *__restrict__ weight,
                                            double e[4], double *se)
{
    const int lane = threadIdx.x & 31;
    const int card = NB_META_CARD(meta);
    const bool small = NB_META_DTYPE(meta) == 0 && card <= 4;
    NbRow r = nb_warp_row(wwords, wrow_ptr, wr);
    if (!small) {
        for (int k = lane; k < card; k += 32) se[k] = 0.0;
        __syncwarp();
    }
    for (int64_t i = i0 + lane; i < i1; i += 32) {
        uint2 ent = inc[i];
        int pos = (int)ent.x;
        NbHdr h = nb_read_hdr<WIDE>(r, pos);
        int mpos = nb_member_pos<WIDE>(h, pos);
        double w = __ldg(weight + h.wid);
        if (small) {
#pragma unroll
            for (int k = 0; k < 4; k++)
                if (k < card) e[k] += w * nb_eval_incidence(r, h, mpos, self, k, vals);
        } else if (NB_META_DTYPE(meta) == 0) {
            for (int k = 0; k < card; k++) atomicAdd(&se[k], w * nb_eval_incidence(r, h, mpos, self, k, vals));
        } else {
            int k = (int)ent.y;
            atomicAdd(&se[k], w * nb_eval_incidence(r, h, mpos, self, k, vals));
        }
    }
    if (small) {
#pragma unroll
        for (int k = 0; k < 4; k++) e[k] = nb_warp_sum(e[k]);
    } else {
        __syncwarp();
    }
}

// draw from the shared per-value energies (uniform on all lanes; lane 0's result is used)
__device__ inline int nb_draw_shared(const double *se, int card, NbUniforms &rng)
{
    NbReservoir res;
    for (int k = 0; k < card; k++)
        if (res.add(se[k], 1.0, rng.next32())) res.pick = k;
    return res.pick;
}

struct WarpTasks {
    const int32_t *task_row;
    const int32_t *task_beg;
    const int64_t *task_ptr;
    double *part;
    int stride;
};

// Phase 1: one warp per task (a slice of one long row) -> partial energies.
template <bool WIDE, class T>
__global__ void __launch_bounds__(32 * NB_WARPS_PER_BLOCK) k_gibbs_warp_partial(SweepArgs<T> a, WarpTasks t, int kbeg, int kend)
{
    __shared__ double s_e[NB_WARPS_PER_BLOCK][NB_MAX_CARD + 1];
    nb_wait_halo(a);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t task = (int64_t)kbeg + blockIdx.x * (int64_t)NB_WARPS_PER_BLOCK + warp;
    if (task >= kend) return;
    const int64_t wr = t.task_row[task];
    const int64_t nid = a.n_trows + wr;
    const uint32_t meta = a.vmeta[nid];
    const int evid = NB_META_EVID(meta), card = NB_META_CARD(meta);
    if (!NB_META_VALID(meta) || evid == 4) return;
    if (!(evid == 0 || a.sample_evidence)) return;
    if (sizeof(T) > 1 && card == 0) return;     // cardinality above 255: sampled whole by k_gibbs_warp_finish
    const int64_t i0 = a.inc_ptr[wr] + t.task_beg[task];
    const int64_t i1 = min(i0 + (int64_t)NB_WARP_TASK, a.inc_ptr[wr + 1]);
    double e[4] = {0.0, 0.0, 0.0, 0.0};
    nb_warp_row_energies<WIDE>(a.wwords, a.wrow_ptr, a.inc, i0, i1, wr, (uint32_t)nid, meta, a.val, a.weight, e, s_e[warp]);
    double *out = t.part + (size_t)task * t.stride;
    if (NB_META_DTYPE(meta) == 0 && card <= 4) {
        if (lane < 4) out[lane] = lane == 0 ? e[0] : (lane == 1 ? e[1] : (lane == 2 ? e[2] : e[3]));
    } else {
        for (int k = lane; k < card; k += 32) out[k] = s_e[warp][k];
    }
}

// Phase 2: one warp per row sums its tasks' partials, samples, stores, tallies.
template <bool WIDE, class T>
__global__ void __launch_bounds__(32 * NB_WARPS_PER_BLOCK) k_gibbs_warp_finish(SweepArgs<T> a, WarpTasks t, int wbeg, int wend)
{
    __shared__ double s_e[NB_WARPS_PER_BLOCK][NB_MAX_CARD + 1];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t wr = (int64_t)wbeg + blockIdx.x * (int64_t)NB_WARPS_PER_BLOCK + warp;
    if (wr >= wend) return;
    const int64_t nid = a.n_trows + wr;
    const uint32_t meta = a.vmeta[nid];
    const int evid = NB_META_EVID(meta), card = NB_META_CARD(meta);
    if (!NB_META_VALID(meta) || evid == 4) return;
    if (!(evid == 0 || a.sample_evidence)) return;
    if (sizeof(T) > 1 && card == 0) {           // cardinality above 255 (2-byte graphs)
        NbUniforms rng(a.rng_id[nid], a.epoch, NB_TAG_FREE, a.seed);
        const NbRow r = nb_warp_row(a.wwords, a.wrow_ptr, wr);
        const int k = nb_warp_sample_wide<WIDE>(r, (int)(a.wrow_ptr[wr + 1] - a.wrow_ptr[wr]), a.inc + a.inc_ptr[wr],
                                                (int)(a.inc_ptr[wr + 1] - a.inc_ptr[wr]), (uint32_t)nid, meta,
                                                nb_card(a, meta, nid), NbValsGlobal<T>(a.val), NbWtsGlobal{a.weight}, rng);
        if (lane == 0) {
            a.val[nid] = (T)k;
            nb_tally(a, nid, nb_card(a, meta, nid), k);
        }
        return;
    }
    // fixed summation tree (lane l takes tasks l, l + 32, ..., then the warp butterfly): the result
    // depends on the row's task list only, not on the launch or the partition
    const int64_t t0 = t.task_ptr[wr], t1 = t.task_ptr[wr + 1];
    for (int k = 0; k < card; k++) {
        double s = 0.0;
        for (int64_t q = t0 + lane; q < t1; q += 32) s += t.part[(size_t)q * t.stride + k];
        s = nb_warp_sum(s);
        if (lane == 0) s_e[warp][k] = s;
    }
    __syncwarp();
    NbUniforms rng(a.rng_id[nid], a.epoch, NB_TAG_FREE, a.seed);
    int k;
    if (NB_META_DTYPE(meta) == 0 && card <= 4) {
        double e[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
        for (int j = 0; j < 4; j++) if (j < card) e[j] = s_e[warp][j];
        k = nb_draw_small(e, card, rng.next());
    } else {
        k = nb_draw_shared(s_e[warp], card, rng);
    }
    if (lane == 0) {
        if (a.valbits && (int)a.val[nid] != k) atomicXor(a.valbits + (nid >> 5), 1u << (nid & 31));   // (all-Boolean graph)
        a.val[nid] = (T)k;
        nb_tally(a, nid, card, k);
    }
}

// The row classes of one colour are independent of each other (same colour: no shared factor), so
// with g->fan_out their kernels run CONCURRENTLY: the class with the most rows stays on the graph's
// stream, the others go to auxiliary streams forked and joined with events.  On the KBC shape a
// colour is one big FAST launch plus a small PAIR launch and two tiny hub (warp-path) launches, which
// used to run one after the other (launch gaps + under-filled tails: a few % of the sweep).
static int fan_streams(nb_graph *g)
{
    if (g->aux[0]) return NB_OK;
    for (int i = 0; i < NB_AUX_STREAMS; i++) {
        NB_CUDA(cudaStreamCreateWithFlags(&g->aux[i], cudaStreamNonBlocking));
        NB_CUDA(cudaEventCreateWithFlags(&g->ev_join[i], cudaEventDisableTiming));
    }
    NB_CUDA(cudaEventCreateWithFlags(&g->ev_fork, cudaEventDisableTiming));
    return NB_OK;
}

template <class T>
static int launch_gibbs_color_t(nb_graph *g, int color, int burnin, int sample_evidence, uint64_t seed, uint64_t epoch)
{
    const NbColorRange &c = g->colors[(size_t)color];
    SweepArgs<T> a = sweep_args<T>(g, 0, burnin, sample_evidence, seed, epoch);
    if (c.f_end > c.f_beg || c.c_end > c.c_beg) NB_TRY(nb_refresh_inlined_weights(g));
    // streams of the five row classes (PAIR, FAST, CAT, GEN, WARP)
    const int64_t rows[5] = {c.p_end - c.p_beg, c.f_end - c.f_beg, c.c_end - c.c_beg, c.t_end - c.t_beg, c.w_end - c.w_beg};
    cudaStream_t st[5] = {g->stream, g->stream, g->stream, g->stream, g->stream};
    int n_aux = 0, aux_of[5] = {-1, -1, -1, -1, -1};
    if (g->fan_out) {
        int big = 0, n_live = 0;
        for (int k = 0; k < 5; k++) { if (rows[k] > rows[big]) big = k; n_live += rows[k] > 0; }
        if (n_live > 1) {
            NB_TRY(fan_streams(g));
            NB_CUDA(cudaEventRecord(g->ev_fork, g->stream));
            for (int k = 0; k < 5; k++)
                if (k != big && rows[k] > 0 && n_aux < NB_AUX_STREAMS) {
                    aux_of[k] = n_aux;
                    st[k] = g->aux[n_aux];
                    NB_CUDA(cudaStreamWaitEvent(st[k], g->ev_fork, 0));
                    n_aux++;
                }
        }
    }
    if (c.p_end > c.p_beg) {
        unsigned grid = (unsigned)((c.p_end - c.p_beg + NB_TT2_BLOCK - 1) / NB_TT2_BLOCK);
        uint32_t key = nb_fold_key(seed, epoch, NB_TAG_FREE);
        bool bits = false;
        if constexpr (sizeof(T) == 1) {     // (the bit mirror exists on all-Boolean graphs only)
            bits = a.valbits != nullptr;
            if (bits) k_gibbs_tt2<true, T><<<grid, NB_TT2_BLOCK, 0, st[0]>>>(a, g->d_tt2_ptr, g->d_tt2_common, g->d_tt2, c.p_beg, c.p_end, key);
        }
        if (!bits) k_gibbs_tt2<false, T><<<grid, NB_TT2_BLOCK, 0, st[0]>>>(a, g->d_tt2_ptr, g->d_tt2_common, g->d_tt2, c.p_beg, c.p_end, key);
        g->launches++;
    }
    if (c.f_end > c.f_beg) {
        unsigned grid = (unsigned)((c.f_end - c.f_beg + 255) / 256);
        uint32_t key = nb_fold_key(seed, epoch, NB_TAG_FREE);
        bool bits = false;
        if constexpr (sizeof(T) == 1) {
            bits = a.valbits != nullptr;
            if (bits) k_gibbs_tt<NB_TT_UNROLL_SWEEP, NB_TT_MINB, true, T><<<grid, 256, 0, st[1]>>>(a, g->d_tt_ptr, g->d_tt, c.f_beg, c.f_end, key);
        }
        if (!bits) k_gibbs_tt<NB_TT_UNROLL_SWEEP, NB_TT_MINB, false, T><<<grid, 256, 0, st[1]>>>(a, g->d_tt_ptr, g->d_tt, c.f_beg, c.f_end, key);
        g->launches++;
    }
    if (c.c_end > c.c_beg) {
        unsigned grid = (unsigned)((c.c_end - c.c_beg + 255) / 256);
        k_gibbs_cat<T><<<grid, 256, 0, st[2]>>>(a, g->d_cat_ptr, g->d_cat, g->n_frows, c.c_beg, c.c_end);
        g->launches++;
    }
    if (c.t_end > c.t_beg) {
        unsigned grid = (unsigned)((c.t_end - c.t_beg + 255) / 256);
        if (g->wide) k_gibbs_thread<true, T><<<grid, 256, 0, st[3]>>>(a, c.t_beg, c.t_end);
        else k_gibbs_thread<false, T><<<grid, 256, 0, st[3]>>>(a, c.t_beg, c.t_end);
        g->launches++;
    }
    if (c.w_end > c.w_beg) {
        WarpTasks t{g->d_wtask_row, g->d_wtask_beg, g->d_wtask_ptr, g->d_wpart, g->wpart_stride};
        unsigned grid1 = (unsigned)((c.k_end - c.k_beg + NB_WARPS_PER_BLOCK - 1) / NB_WARPS_PER_BLOCK);
        unsigned grid2 = (unsigned)((c.w_end - c.w_beg + NB_WARPS_PER_BLOCK - 1) / NB_WARPS_PER_BLOCK);
        if (g->wide) {
            k_gibbs_warp_partial<true, T><<<grid1, 32 * NB_WARPS_PER_BLOCK, 0, st[4]>>>(a, t, c.k_beg, c.k_end);
            k_gibbs_warp_finish<true, T><<<grid2, 32 * NB_WARPS_PER_BLOCK, 0, st[4]>>>(a, t, c.w_beg, c.w_end);
        } else {
            k_gibbs_warp_partial<false, T><<<grid1, 32 * NB_WARPS_PER_BLOCK, 0, st[4]>>>(a, t, c.k_beg, c.k_end);
            k_gibbs_warp_finish<false, T><<<grid2, 32 * NB_WARPS_PER_BLOCK, 0, st[4]>>>(a, t, c.w_beg, c.w_end);
        }
        g->launches += 2;
    }
    for (int k = 0; k < 5; k++)
        if (aux_of[k] >= 0) {                       // join: the next colour reads what these kernels wrote
            NB_CUDA(cudaEventRecord(g->ev_join[aux_of[k]], st[k]));
            NB_CUDA(cudaStreamWaitEvent(g->stream, g->ev_join[aux_of[k]], 0));
        }
    NB_CUDA(cudaGetLastError());
    return NB_OK;
}

int nb_check_tally_room(const nb_graph *g, int burnin, int64_t n_sweeps)
{
    if (!burnin && n_sweeps > 0 && g->tally_bound > (int64_t)INT32_MAX - n_sweeps)
        NB_FAIL(NB_ERR_UNSUPPORTED, "%lld tallying sweeps could take a tally from %lld past 2^31 - 1 (the device tallies "
                "are int32): read the counts and reset them first", (long long)n_sweeps, (long long)g->tally_bound);
    return NB_OK;
}

int nb_launch_gibbs_color(nb_graph *g, int color, int burnin, int sample_evidence, uint64_t seed, uint64_t epoch)
{
    if (color < 0) NB_FAIL(NB_ERR_INVALID, "negative colour %d", color);
    if (color >= g->n_colors) return NB_OK;   // partitioned graphs: a colour this rank does not own
    if (!burnin) {
        if (g->tally_launches.size() != (size_t)g->n_colors) g->tally_launches.assign((size_t)g->n_colors, 0);
        int64_t &n = g->tally_launches[(size_t)color];
        if (g->tally_base + n + 1 > INT32_MAX)
            NB_FAIL(NB_ERR_UNSUPPORTED, "a tally of colour %d could pass 2^31 - 1 (the device tallies are int32): "
                    "read the counts and reset them first", color);
        n++;
        g->tally_bound = std::max(g->tally_bound, g->tally_base + n);
    }
    return g->value_bytes == 1 ? launch_gibbs_color_t<nb_val_t>(g, color, burnin, sample_evidence, seed, epoch)
                               : launch_gibbs_color_t<nb_val16_t>(g, color, burnin, sample_evidence, seed, epoch);
}

// ---------------------------------------------------------------------------
// potential() parity hook (inference.py:55-71): one thread per requested
// variable walks its row once per value, summing in bucket order.
// ---------------------------------------------------------------------------
template <bool WIDE, class T>
__global__ void k_potentials(SweepArgs<T> a, const int32_t *old2new, const int64_t *var_ids, int64_t n,
                             const int64_t *out_offsets, double *out)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t nid = old2new[var_ids[i]];
    const uint32_t meta = a.vmeta[nid];
    const int card = nb_card(a, meta, nid);
    NbRow r = nid < a.n_trows ? nb_thread_row(a.twords, a.slice_ptr, nid) : nb_warp_row(a.wwords, a.wrow_ptr, nid - a.n_trows);
    const int len = nid < a.n_trows ? NB_META_ROWLEN(meta)
                                    : (int)(a.wrow_ptr[nid - a.n_trows + 1] - a.wrow_ptr[nid - a.n_trows]);
    double *o = out + out_offsets[i];
    for (int k = 0; k < card; k++) {
        double e = 0.0;
        if (NB_META_DTYPE(meta) == 0) {
            e = nb_row_energy_k<WIDE>(r, len, (uint32_t)nid, k, a.val, a.weight);
        } else {
            int pos = 0, cur = -1;
            while (pos < len) {
                NbHdr h = nb_read_hdr<WIDE>(r, pos);
                if (h.code == C_MARK) cur = (int)h.wid;
                else if (cur == k)
                    e = nb_acc(e, a.weight[h.wid], nb_eval_incidence(r, h, nb_member_pos<WIDE>(h, pos), (uint32_t)nid, k, a.val));
                pos += nb_inc_words<WIDE>(h);
            }
        }
        o[k] = e;
    }
}

int nb_run_potentials(nb_graph *g, int chain, const int64_t *var_ids, int64_t n, const int64_t *out_offsets,
                      double *out, int64_t n_out)
{
    if (chain < 0 || chain > 1) NB_FAIL(NB_ERR_INVALID, "chain must be 0 or 1");
    if (n == 0) return NB_OK;
    for (int64_t i = 0; i < n; i++)
        if (var_ids[i] < 0 || var_ids[i] >= g->V) NB_FAIL(NB_ERR_INVALID, "variable id %lld out of range", (long long)var_ids[i]);
    int64_t *d_ids, *d_off;
    double *d_out;
    NB_CUDA(cudaMalloc(&d_ids, (size_t)n * 8));
    NB_CUDA(cudaMalloc(&d_off, (size_t)n * 8));
    NB_CUDA(cudaMalloc(&d_out, (size_t)std::max<int64_t>(n_out, 1) * 8));
    cudaMemcpyAsync(d_ids, var_ids, (size_t)n * 8, cudaMemcpyHostToDevice, g->stream);
    cudaMemcpyAsync(d_off, out_offsets, (size_t)n * 8, cudaMemcpyHostToDevice, g->stream);
    cudaMemsetAsync(d_out, 0, (size_t)n_out * 8, g->stream);
    unsigned grid = (unsigned)((n + 127) / 128);
    if (g->value_bytes == 1) {
        SweepArgs<nb_val_t> a = sweep_args<nb_val_t>(g, chain, 1, 1, 0, 0);
        if (g->wide) k_potentials<true><<<grid, 128, 0, g->stream>>>(a, g->d_old2new, d_ids, n, d_off, d_out);
        else k_potentials<false><<<grid, 128, 0, g->stream>>>(a, g->d_old2new, d_ids, n, d_off, d_out);
    } else {
        SweepArgs<nb_val16_t> a = sweep_args<nb_val16_t>(g, chain, 1, 1, 0, 0);
        if (g->wide) k_potentials<true><<<grid, 128, 0, g->stream>>>(a, g->d_old2new, d_ids, n, d_off, d_out);
        else k_potentials<false><<<grid, 128, 0, g->stream>>>(a, g->d_old2new, d_ids, n, d_off, d_out);
    }
    cudaMemcpyAsync(out, d_out, (size_t)n_out * 8, cudaMemcpyDeviceToHost, g->stream);
    cudaError_t e = cudaStreamSynchronize(g->stream);
    cudaFree(d_ids); cudaFree(d_off); cudaFree(d_out);
    NB_CUDA(e);
    NB_CUDA(cudaGetLastError());
    return NB_OK;
}

// ---------------------------------------------------------------------------
// Parity hook for the RECORD streams: the same device functions the sweep kernels call
// (nb_tt2_delta / nb_tt_delta / nb_cat_energies) evaluated for the listed variables, so that the
// energies the hot kernels sample from can be compared with the reference's potential()
// (inference.py:55-71) deterministically.  PAIR / FAST rows write {0, e1 - e0}; CAT rows write the
// fp32 per-value energies; rows of the generic classes write nothing (row_class tells).
// ---------------------------------------------------------------------------
struct NbCatLocalAcc {
    float *e;
    __device__ __forceinline__ void add(int k, float w) { e[k] += w; }
};

struct RecordStreams {
    const int64_t *tt2_ptr; const uint32_t *tt2_common; const uint4 *tt2;
    const int64_t *tt_ptr; const uint4 *tt;
    const int64_t *cat_ptr; const uint4 *cat;
    int64_t n_prows, n_frows, n_crows;
};

template <class T>
__global__ void k_potentials_records(SweepArgs<T> a, RecordStreams R, const int32_t *old2new, const int64_t *var_ids, int64_t n,
                                     const int64_t *out_offsets, double *out, int32_t *row_class)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t nid = old2new[var_ids[i]];
    const uint32_t meta = a.vmeta[nid];
    double *o = out + out_offsets[i];
    const int64_t s = nid >> 5;
    if (nid < R.n_prows) {
        const int64_t q0 = R.tt2_ptr[s];
        o[0] = 0.0;
        o[1] = nb_tt2_delta(R.tt2 + q0 + (nid & 31), (int)((R.tt2_ptr[s + 1] - q0) >> 5), R.tt2_common[s], (uint32_t)nid, a.val, a.weight);
        row_class[i] = NB_CLASS_PAIR;
    } else if (nid < R.n_frows) {
        const int64_t q0 = R.tt_ptr[s];
        o[0] = 0.0;
        o[1] = nb_tt_delta(R.tt + q0 + (nid & 31), (int)((R.tt_ptr[s + 1] - q0) >> 5), (uint32_t)nid, a.val);
        row_class[i] = NB_CLASS_FAST;
    } else if (nid < R.n_crows) {
        const int64_t sc = (nid - R.n_frows) >> 5;
        const int64_t q0 = R.cat_ptr[sc];
        float e[NB_CAT_MAX_CARD];
        for (int k = 0; k < NB_CAT_MAX_CARD; k++) e[k] = 0.0f;
        NbCatLocalAcc acc{e};
        nb_cat_energies(R.cat + q0 + (nid & 31), (int)((R.cat_ptr[sc + 1] - q0) >> 5), (uint32_t)nid, a.val, acc);
        const int card = NB_META_CARD(meta);   // CAT rows: card <= NB_CAT_MAX_CARD
        for (int k = 0; k < card; k++) o[k] = (double)e[k];
        row_class[i] = NB_CLASS_CAT;
    } else {
        row_class[i] = nid < a.n_trows ? NB_CLASS_GEN : NB_CLASS_WARP;
    }
}

int nb_run_potentials_records(nb_graph *g, int chain, const int64_t *var_ids, int64_t n, const int64_t *out_offsets,
                              double *out, int64_t n_out, int32_t *row_class)
{
    if (chain < 0 || chain > 1) NB_FAIL(NB_ERR_INVALID, "chain must be 0 or 1");
    if (n == 0) return NB_OK;
    for (int64_t i = 0; i < n; i++)
        if (var_ids[i] < 0 || var_ids[i] >= g->V) NB_FAIL(NB_ERR_INVALID, "variable id %lld out of range", (long long)var_ids[i]);
    NB_TRY(nb_refresh_inlined_weights(g));
    int64_t *d_ids, *d_off;
    double *d_out;
    int32_t *d_cls;
    NB_CUDA(cudaMalloc(&d_ids, (size_t)n * 8));
    NB_CUDA(cudaMalloc(&d_off, (size_t)n * 8));
    NB_CUDA(cudaMalloc(&d_cls, (size_t)n * 4));
    NB_CUDA(cudaMalloc(&d_out, (size_t)std::max<int64_t>(n_out, 1) * 8));
    cudaMemcpyAsync(d_ids, var_ids, (size_t)n * 8, cudaMemcpyHostToDevice, g->stream);
    cudaMemcpyAsync(d_off, out_offsets, (size_t)n * 8, cudaMemcpyHostToDevice, g->stream);
    cudaMemsetAsync(d_out, 0, (size_t)n_out * 8, g->stream);
    RecordStreams R{g->d_tt2_ptr, g->d_tt2_common, g->d_tt2, g->d_tt_ptr, g->d_tt, g->d_cat_ptr, g->d_cat,
                    g->n_prows, g->n_frows, g->n_crows};
    if (g->value_bytes == 1) {
        SweepArgs<nb_val_t> a = sweep_args<nb_val_t>(g, chain, 1, 1, 0, 0);
        a.w_n = 0;
        k_potentials_records<<<(unsigned)((n + 127) / 128), 128, 0, g->stream>>>(a, R, g->d_old2new, d_ids, n, d_off, d_out, d_cls);
    } else {
        SweepArgs<nb_val16_t> a = sweep_args<nb_val16_t>(g, chain, 1, 1, 0, 0);
        a.w_n = 0;
        k_potentials_records<<<(unsigned)((n + 127) / 128), 128, 0, g->stream>>>(a, R, g->d_old2new, d_ids, n, d_off, d_out, d_cls);
    }
    cudaMemcpyAsync(out, d_out, (size_t)n_out * 8, cudaMemcpyDeviceToHost, g->stream);
    cudaMemcpyAsync(row_class, d_cls, (size_t)n * 4, cudaMemcpyDeviceToHost, g->stream);
    cudaError_t e = cudaStreamSynchronize(g->stream);
    cudaFree(d_ids); cudaFree(d_off); cudaFree(d_out); cudaFree(d_cls);
    NB_CUDA(e);
    NB_CUDA(cudaGetLastError());
    return NB_OK;
}
