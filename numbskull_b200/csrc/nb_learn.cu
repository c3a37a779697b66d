// Weight learning sweep (learning.py:12-125 learnthread / sample_and_sgd).
//
// An epoch walks the graph in mini-batch CELLS: blocks of consecutive variable ids (outer) and,
// inside a block, the colours (inner) -- see DESIGN.md "learning".  In a cell every owned variable
// samples the evidence chain and the free chain in the same pass over its row, then walks the row
// again for the per-factor gradient (f(proposal | free) - f(evidence | evid)) * featureValue.
// Gradients and visit counts are REDUCED BY WEIGHT ID in integers (order-independent, hence
// deterministic), and the SGD / L2-shrink / L1-truncated-gradient update is applied once per cell.
//
// The whole epoch is ONE persistent cooperative kernel (k_learn_cells): the CTAs stay resident,
// walk the cells together and meet at a grid barrier after each one -- a cell of the
// labelling-function model holds ~1000 rows, far too little for a launch of its own (round 1:
// 3216 launches and 113 ms per epoch on 1 M x 100).  Weight tables of up to NB_LEARN_SMEM_W entries
// are staged in shared memory: every CTA keeps its own copy of the weights, reduces its gradients in
// shared-memory tables, adds them to a global integer table (one atomic per touched weight and
// CTA), and after the barrier applies the closed-form update to its own copy -- identical inputs,
// identical result in every CTA, one barrier per cell.  Larger tables accumulate straight into the
// global integer table and are applied by the grid (two barriers per cell).
#include <algorithm>
#include <cmath>
#include <cooperative_groups.h>

#include "nb_eval.cuh"

namespace cg = cooperative_groups;

#define NB_LEARN_SMEM_W 2048
#define NB_LEARN_THREADS 256
#define NB_LWARPS (NB_LEARN_THREADS / 32)

// Gradients accumulate in 64-bit fixed point (2^-20 units; truth-table rows contribute integers):
// integer addition is associative, so per-weight sums do not depend on the order in which threads,
// CTAs or atomics land.
#define NB_GRAD_UNIT 1048576.0
#define NB_GRAD_SHIFT 20
typedef long long nb_fix_t;

// T = element type of the value arrays (nb_val_t or nb_val16_t, see nb_graph::value_bytes)
template <class T>
struct LearnArgs : NbCardOf<T> {   // (cardinalities: a.card(meta, nid))
    const uint32_t *vmeta;
    const int64_t *slice_ptr;
    const uint32_t *twords;
    const int64_t *wrow_ptr;
    const uint32_t *wwords;
    const int64_t *inc_ptr;
    const uint2 *inc;
    const uint32_t *rng_id;
    const T *vinit;
    T *val_free;
    T *val_evid;
    double *weight;
    const uint8_t *wfixed;
    int64_t n_trows;
    int W;
    uint64_t seed, epoch;
    double step, reg_param, truncation;
    int regularization, learn_non_evidence;
    // truth-table rows
    const int64_t *tt_ptr;
    const uint4 *tt;
    const uint32_t *tt_base;
    const uint32_t *tt_wid;   // weight id per quad (the quads themselves inline the weight VALUE for the Gibbs sweep)
    // categorical record rows (new ids [cat_first, ...)): records + weight ids, see nb_cat_energies
    const int64_t *cat_ptr;
    const uint4 *cat;
    const uint32_t *cat_wid;
    int64_t cat_first;
    // reduction by weight id: three rotating global tables [3][W] (cell c uses c % 3)
    nb_fix_t *g_grad;
    uint32_t *g_cnt;
    // NUMBSKULL_B200_LEARN_TRACE=1: per-phase nanoseconds summed over CTAs and cells
    // [0] range lookup + zeroing  [1] truth-table rows  [2] thread rows  [3] warp rows  [4] flush
    // [5] grid barrier  [6] apply  [7] cells processed  [8] sum over cells of the slowest CTA's work time
    unsigned *bar;            // grid barrier state {arrivals, generation}
    unsigned long long *trace;
    unsigned long long *trace_cell;   // [n cells] scratch: max work time of the cell over the CTAs
    unsigned long long *trace_cta;    // [grid][3] per-CTA sums: truth-table rows, thread rows, whole work phase
};

__device__ __forceinline__ unsigned long long nb_now()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// Where the cells' rows are: block b of n_blocks covers the units [T b / nb, T (b + 1) / nb) of
// T = n_win * k_sub units; unit u is sub-range (u % k_sub) of k_sub of id window u / k_sub.  Inside a
// (row class, colour) group the rows are sorted by window, so a block is one contiguous id range per
// group; windows are cut further (k_sub > 1) when even one window holds more visits of a weight than
// the mini-batch bound allows (tied weights on large graphs).
struct CellPlan {
    const int32_t *win_start;   // [NB_N_CLASSES * (n_colors + 1)][n_win + 1] first new id of each window per group
    const uint8_t *long_rows;   // [n_colors] truth-table rows of the colour average >= 16 incidences: one warp per row
    int64_t n_win;
    int n_colors;               // colours of THIS graph
    int n_blocks, k_sub;
    int64_t n_trows;
};

__host__ __device__ __forceinline__ int nb_plan_pos(const CellPlan &p, int group, int64_t unit)
{
    const int32_t *ws = p.win_start + (size_t)group * (size_t)(p.n_win + 1);
    const int64_t w = unit / p.k_sub, j = unit % p.k_sub;
    if (w >= p.n_win) return ws[p.n_win];
    const int64_t s = ws[w], e = ws[w + 1];
    return (int)(s + (e - s) * j / p.k_sub);
}

__host__ __device__ __forceinline__ void nb_plan_range(const CellPlan &p, int cls, int color, int block, int &beg, int &end)
{
    const int64_t T = p.n_win * (int64_t)p.k_sub;
    const int group = cls * (p.n_colors + 1) + color;
    beg = nb_plan_pos(p, group, T * block / p.n_blocks);
    end = nb_plan_pos(p, group, T * (block + 1) / p.n_blocks);
}

// ---------------------------------------------------------------------------
// closed-form application of n per-visit updates (learning.py:110-125):
//   L2: each visit does w = w * s - step * g_i, s = 1 / (1 + reg_param * step),
//       so n visits give w * s^n - step * sum_i g_i s^(n-i); the g_i are spread
//       evenly over the batch, i.e. sum_i g_i s^(n-i) ~= G * (1 - s^n) / (n (1 - s)).
//   L1: w -= step * G, then the m truncating visits' soft-threshold, merged.
// ---------------------------------------------------------------------------
__device__ __forceinline__ double nb_apply_update(double w, double G, uint32_t cnt, int regularization, double step,
                                                  double reg_param, double truncation)
{
    if (regularization == 2) {
        if (cnt == 0) return w - step * G;
        double s = 1.0 / (1.0 + reg_param * step);
        double sn = pow(s, (double)cnt);
        double geo = (s < 1.0) ? (1.0 - sn) / ((double)cnt * (1.0 - s)) : 1.0;
        return w * sn - step * G * geo;
    }
    w -= step * G;
    if (regularization == 1 && cnt > 0) {
        double l1 = reg_param * step * truncation * (double)cnt;
        w = w > 0.0 ? fmax(0.0, w - l1) : fmin(0.0, w + l1);
    }
    return w;
}

// Per-CTA view of the reduction targets and the weights during one cell.
template <bool SMEM>
struct LearnCtx {
    const double *w;        // weights: this CTA's shared copy (SMEM) or the global table
    int32_t *gi;            // SMEM: shared integer gradient table (truth-table rows)
    nb_fix_t *gf;           // shared (SMEM) or global fixed-point gradient table
    uint32_t *cnt;          // shared or global visit counts
    // (global table: cached in L1 like the values -- updated only between two grid barriers)
    __device__ __forceinline__ double weight(uint32_t i) const { return SMEM ? w[i] : __ldca(w + i); }
    __device__ __forceinline__ void add_int(uint32_t wid, int g, uint32_t c) const
    {
        if (SMEM) { if (g) atomicAdd(gi + wid, g); }
        else if (g) atomicAdd((unsigned long long *)(gf + wid), (unsigned long long)((long long)g << NB_GRAD_SHIFT));
        if (c) atomicAdd(cnt + wid, c);
    }
    __device__ __forceinline__ void add_real(uint32_t wid, double g, uint32_t c) const
    {
        if (g != 0.0) atomicAdd((unsigned long long *)(gf + wid), (unsigned long long)__double2ll_rn(g * NB_GRAD_UNIT));
        if (c) atomicAdd(cnt + wid, c);
    }
};

template <bool SMEM>
struct CtxWts {
    LearnCtx<SMEM> c;
    __device__ __forceinline__ double operator()(uint32_t i) const { return c.weight(i); }
};

// visit counter increment of one variable (learning.py:90: one truncation draw per variable)
template <class T>
__device__ __forceinline__ uint32_t nb_cnt_inc(const LearnArgs<T> &a, uint32_t id)
{
    if (a.regularization == 1) {
        NbUniforms tr(id, a.epoch, NB_TAG_TRUNC, a.seed);
        return tr.next() < 1.0 / a.truncation ? 1u : 0u;
    }
    return a.regularization == 2 ? 1u : 0u;
}

// second pass over a row: gradient of every visited incidence with a learnable weight
template <bool WIDE, bool SMEM, class T>
__device__ NB_EVAL_FN void nb_row_gradient(const NbRow &r, int len, uint32_t self, uint32_t meta, int ev, int prop,
                                       const LearnArgs<T> &a, uint32_t cnt_inc, const LearnCtx<SMEM> &ctx,
                                       int first_inc, int inc_stride, const uint2 *inc_list, int n_inc)
{
    const bool cat = NB_META_DTYPE(meta) == 1;
    const NbValsCG<T> vF(a.val_free), vE(a.val_evid);
    if (inc_list == nullptr) {
        int pos = 0, cur = -1;
        while (pos < len) {
            NbHdr h = nb_read_hdr<WIDE>(r, pos);
            if (h.code == C_MARK) cur = (int)h.wid;
            else if (!h.fixed && (!cat || cur == ev || cur == prop)) {
                int mpos = nb_member_pos<WIDE>(h, pos);
                double f1 = nb_eval_incidence_v(r, h, mpos, self, prop, vF);
                double f0 = nb_eval_incidence_v(r, h, mpos, self, ev, vE);
                double feat = h.feat ? nb_read_feature<WIDE>(r, h, pos) : 1.0;
                ctx.add_real(h.wid, (f1 - f0) * feat, cnt_inc);
            }
            pos += nb_inc_words<WIDE>(h);
        }
    } else {
        for (int i = first_inc; i < n_inc; i += inc_stride) {
            uint2 ent = inc_list[i];
            int pos = (int)ent.x, cur = (int)ent.y;
            NbHdr h = nb_read_hdr<WIDE>(r, pos);
            if (h.fixed || (cat && cur != ev && cur != prop)) continue;
            int mpos = nb_member_pos<WIDE>(h, pos);
            double f1 = nb_eval_incidence_v(r, h, mpos, self, prop, vF);
            double f0 = nb_eval_incidence_v(r, h, mpos, self, ev, vE);
            double feat = h.feat ? nb_read_feature<WIDE>(r, h, pos) : 1.0;
            ctx.add_real(h.wid, (f1 - f0) * feat, cnt_inc);
        }
    }
}

// ---------------------------------------------------------------------------
// thread path: generic rows (GEN class) and categorical record rows (CAT class), one row per thread
// ---------------------------------------------------------------------------
template <bool WIDE, bool SMEM, class T>
__device__ __noinline__ void learn_thread_rows(const LearnArgs<T> &a, const LearnCtx<SMEM> &ctx, int beg0, int end0, int beg1, int end1)
{
    const int64_t n0 = end0 - beg0, ntot = n0 + (end1 - beg1);
    const CtxWts<SMEM> wts{ctx};
    for (int64_t it = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; it < ntot; it += (int64_t)gridDim.x * blockDim.x) {
        const int64_t nid = it < n0 ? beg0 + it : beg1 + (it - n0);
        const uint32_t meta = a.vmeta[nid];
        const int evid = NB_META_EVID(meta);
        if (!NB_META_VALID(meta) || evid == 4) continue;                   // learning.py:24-26
        NbRow r = nb_thread_row(a.twords, a.slice_ptr, nid);
        const int len = NB_META_ROWLEN(meta);
        const uint32_t self = (uint32_t)nid, id = a.rng_id[nid];
        int ev;
        if (evid != 1) {                                                    // :53-57
            NbUniforms rng(id, a.epoch, NB_TAG_EVID, a.seed);
            ev = nb_sample_row_v<WIDE>(r, len, self, meta, NbValsCG<T>(a.val_evid, a), wts, rng);
        } else {
            ev = (int)a.vinit[nid];                                         // :60-61
        }
        a.val_evid[nid] = (T)ev;                                            // :63
        NbUniforms rng(id, a.epoch, NB_TAG_FREE, a.seed);
        int prop = nb_sample_row_v<WIDE>(r, len, self, meta, NbValsCG<T>(a.val_free, a), wts, rng);   // :65-67
        a.val_free[nid] = (T)prop;                                          // :69
        if (!a.learn_non_evidence && evid != 1) continue;                   // :70-71
        nb_row_gradient<WIDE, SMEM>(r, len, self, meta, ev, prop, a, nb_cnt_inc(a, id), ctx, 0, 1, nullptr, 0);
    }
}

template <class T>
__device__ __forceinline__ int nb_ldv(const T *v, uint32_t i) { return (int)__ldca(v + i); }   // see NbValsCG
// ---------------------------------------------------------------------------
// categorical record rows (CAT class), one row per thread.  Same records as the Gibbs sweep
// (nb_cat_energies: one 16-byte quad per incidence of an AND_CAT / EQUAL_CAT_CONST factor in its
// value bucket), but the weights are read live through cat_wid -- they move every cell -- and both
// chains are drawn.  Walking the generic words instead costs ~1000 instructions per card-16 row.
// ---------------------------------------------------------------------------
__device__ __forceinline__ bool nb_cat_sat(uint32_t m, int xa, int xb)
{
    const int no = (int)((m >> 24) & 3u);
    return no < 3 && (no < 1 || xa == (int)((m >> 8) & 0xFFu)) && (no < 2 || xb == (int)((m >> 16) & 0xFFu));
}

// draw_sample (inference.py:36-52) from the per-value energies e[0..card), one uniform
__device__ __forceinline__ int nb_cat_draw(float *e, int card, double u)
{
    float mx = e[0];
    for (int k = 1; k < card; k++) mx = fmaxf(mx, e[k]);
    float tot = 0.0f;
    for (int k = 0; k < card; k++) { const float z = __expf(e[k] - mx); e[k] = z; tot += z; }
    const float t = (float)u * tot;
    float acc = 0.0f;
    for (int k = 0; k < card; k++) {
        acc += e[k];
        if (acc >= t) return k;
    }
    return card - 1;
}

template <bool SMEM, class T>
__device__ __forceinline__ int nb_cat_sample_l(const uint4 *qp, const uint32_t *wp, int n, int card, const T *vals,
                                               const LearnCtx<SMEM> &ctx, float *e, double u)
{
    for (int k = 0; k < card; k++) e[k] = 0.0f;
    for (int j = 0; j < n; j += 2) {
        uint4 q[2];
        uint32_t wid[2];
        int xa[2], xb[2];
        const bool in1 = j + 1 < n;
        q[0] = __ldg(qp + (size_t)j * 32);
        wid[0] = __ldg(wp + (size_t)j * 32);
        q[1] = in1 ? __ldg(qp + (size_t)(j + 1) * 32) : make_uint4(q[0].x, q[0].y, nb_pack_cat(0, 0, 0, 3, 1), 0u);
        wid[1] = in1 ? __ldg(wp + (size_t)(j + 1) * 32) : wid[0];
#pragma unroll
        for (int t = 0; t < 2; t++) { xa[t] = nb_ldv(vals, q[t].x); xb[t] = nb_ldv(vals, q[t].y); }
#pragma unroll
        for (int t = 0; t < 2; t++)
            if (nb_cat_sat(q[t].z, xa[t], xb[t])) e[q[t].z & 0xFFu] += (float)ctx.weight(wid[t]);
    }
    return nb_cat_draw(e, card, u);
}

template <bool SMEM, class T>
__device__ __noinline__ void learn_cat_rows(const LearnArgs<T> &a, const LearnCtx<SMEM> &ctx, int beg, int end, uint32_t kf, uint32_t ke)
{
    float e[NB_CAT_MAX_CARD];
    const T *vF = a.val_free, *vE = a.val_evid;
    for (int64_t nid = (int64_t)beg + blockIdx.x * (int64_t)blockDim.x + threadIdx.x; nid < end; nid += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t meta = __ldg(a.vmeta + nid);
        const int evid = NB_META_EVID(meta);
        if (!NB_META_VALID(meta) || evid == 4) continue;                   // learning.py:24-26
        const int card = NB_META_CARD(meta);                               // CAT rows: card <= NB_CAT_MAX_CARD
        const uint32_t id = __ldg(a.rng_id + nid);
        const int64_t s = (nid - a.cat_first) >> 5;
        const int64_t q0 = __ldg(a.cat_ptr + s), q1 = __ldg(a.cat_ptr + s + 1);
        const int n = (int)((q1 - q0) >> 5);
        const uint4 *qp = a.cat + q0 + (nid & 31);
        const uint32_t *wp = a.cat_wid + q0 + (nid & 31);
        int ev;
        if (evid != 1) ev = nb_cat_sample_l<SMEM>(qp, wp, n, card, vE, ctx, e, nb_philox2x32_u53(id, (uint32_t)a.epoch, ke));   // :53-57
        else ev = (int)a.vinit[nid];                                        // :60-61
        a.val_evid[nid] = (T)ev;                                            // :63
        const int prop = nb_cat_sample_l<SMEM>(qp, wp, n, card, vF, ctx, e, nb_philox2x32_u53(id, (uint32_t)a.epoch, kf));   // :65-67
        a.val_free[nid] = (T)prop;                                          // :69
        if (!a.learn_non_evidence && evid != 1) continue;                   // :70-71
        // gradient (learning.py:73-108): the incidences of the buckets of the two chains' values
        const uint32_t cinc = nb_cnt_inc(a, id);
        for (int j = 0; j < n; j++) {
            const uint4 q = __ldg(qp + (size_t)j * 32);
            const uint32_t m = q.z;
            const int k = (int)(m & 0xFFu);
            if (((m >> 26) & 1u) || (k != ev && k != prop)) continue;
            const int f1 = (k == prop && nb_cat_sat(m, nb_ldv(vF, q.x), nb_ldv(vF, q.y))) ? 1 : 0;
            const int f0 = (k == ev && nb_cat_sat(m, nb_ldv(vE, q.x), nb_ldv(vE, q.y))) ? 1 : 0;
            ctx.add_int(__ldg(wp + (size_t)j * 32), f1 - f0, cinc);
        }
    }
}

// ---------------------------------------------------------------------------
// warp path: one long row per warp
// ---------------------------------------------------------------------------
// per-value energies of a warp row into e[4] (dataType 0, card <= 4) or the shared array se
template <bool WIDE, bool SMEM, class T>
__device__ inline void nb_warp_energies_l(const NbRow &r, const uint2 *inc, int n_inc, uint32_t self, uint32_t meta,
                                          const T *vals, const LearnCtx<SMEM> &ctx, double e[4], double *se)
{
    const int lane = threadIdx.x & 31, card = NB_META_CARD(meta);   // <= NB_MAX_CARD: wider rows take nb_warp_sample_wide
    const bool small = NB_META_DTYPE(meta) == 0 && card <= 4;
    const NbValsCG<T> v(vals);
    if (!small) {
        for (int k = lane; k < card; k += 32) se[k] = 0.0;
        __syncwarp();
    }
    for (int i = lane; i < n_inc; i += 32) {
        uint2 ent = inc[i];
        int pos = (int)ent.x;
        NbHdr h = nb_read_hdr<WIDE>(r, pos);
        int mpos = nb_member_pos<WIDE>(h, pos);
        double w = ctx.weight(h.wid);
        if (small) {
#pragma unroll
            for (int k = 0; k < 4; k++)
                if (k < card) e[k] += w * nb_eval_incidence_v(r, h, mpos, self, k, v);
        } else if (NB_META_DTYPE(meta) == 0) {
            for (int k = 0; k < card; k++) atomicAdd(&se[k], w * nb_eval_incidence_v(r, h, mpos, self, k, v));
        } else {
            atomicAdd(&se[(int)ent.y], w * nb_eval_incidence_v(r, h, mpos, self, (int)ent.y, v));
        }
    }
    if (small) {
#pragma unroll
        for (int k = 0; k < 4; k++) e[k] = nb_warp_sum(e[k]);
    } else {
        __syncwarp();
    }
}

template <bool WIDE, bool SMEM, class T>
__device__ NB_EVAL_FN int nb_warp_sample_l(const NbRow &r, const uint2 *inc, int n_inc, uint32_t self, uint32_t meta,
                                       const T *vals, const LearnCtx<SMEM> &ctx, double *se, NbUniforms &rng)
{
    const int card = NB_META_CARD(meta);
    double e[4] = {0.0, 0.0, 0.0, 0.0};
    nb_warp_energies_l<WIDE, SMEM>(r, inc, n_inc, self, meta, vals, ctx, e, se);
    int k;
    if (NB_META_DTYPE(meta) == 0 && card <= 4) k = nb_draw_small(e, card, rng.next());
    else {
        NbReservoir res;
        for (int j = 0; j < card; j++)
            if (res.add(se[j], 1.0, rng.next32())) res.pick = j;
        k = res.pick;
    }
    __syncwarp();
    return k;
}

// the sampler of one chain for a warp row: the shared-memory one, or nb_warp_sample_wide for a
// cardinality above 255 (2-byte graphs)
template <bool WIDE, bool SMEM, class T>
__device__ __forceinline__ int nb_warp_sample_any(const LearnArgs<T> &a, const NbRow &r, int64_t wr, const uint2 *inc, int n_inc,
                                                  uint32_t self, uint32_t meta, const T *vals, const LearnCtx<SMEM> &ctx,
                                                  double *se, NbUniforms &rng)
{
    if (sizeof(T) > 1 && NB_META_CARD(meta) == 0)
        return nb_warp_sample_wide<WIDE>(r, (int)(a.wrow_ptr[wr + 1] - a.wrow_ptr[wr]), inc, n_inc, self, meta,
                                         a.card(meta, self), NbValsCG<T>(vals), CtxWts<SMEM>{ctx}, rng);
    return nb_warp_sample_l<WIDE, SMEM>(r, inc, n_inc, self, meta, vals, ctx, se, rng);
}

template <bool WIDE, bool SMEM, class T>
__device__ __noinline__ void learn_warp_rows(const LearnArgs<T> &a, const LearnCtx<SMEM> &ctx, double *s_e, int wbeg, int wend)
{
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int64_t wr = (int64_t)wbeg + blockIdx.x * (int64_t)NB_LWARPS + warp; wr < wend;
         wr += (int64_t)gridDim.x * NB_LWARPS) {
        const int64_t nid = a.n_trows + wr;
        const uint32_t meta = a.vmeta[nid];
        const int evid = NB_META_EVID(meta);
        if (!NB_META_VALID(meta) || evid == 4) continue;
        NbRow r = nb_warp_row(a.wwords, a.wrow_ptr, wr);
        const uint2 *inc = a.inc + a.inc_ptr[wr];
        const int n_inc = (int)(a.inc_ptr[wr + 1] - a.inc_ptr[wr]);
        const uint32_t self = (uint32_t)nid, id = a.rng_id[nid];
        int ev;
        if (evid != 1) {
            NbUniforms rng(id, a.epoch, NB_TAG_EVID, a.seed);
            ev = nb_warp_sample_any<WIDE, SMEM>(a, r, wr, inc, n_inc, self, meta, a.val_evid, ctx, s_e, rng);
        } else {
            ev = (int)a.vinit[nid];
        }
        NbUniforms rng(id, a.epoch, NB_TAG_FREE, a.seed);
        int prop = nb_warp_sample_any<WIDE, SMEM>(a, r, wr, inc, n_inc, self, meta, a.val_free, ctx, s_e, rng);
        if (lane == 0) { a.val_evid[nid] = (T)ev; a.val_free[nid] = (T)prop; }
        if (!a.learn_non_evidence && evid != 1) continue;
        nb_row_gradient<WIDE, SMEM>(r, 0, self, meta, ev, prop, a, nb_cnt_inc(a, id), ctx, lane, 32, inc, n_inc);
    }
}

// ---------------------------------------------------------------------------
// truth-table rows (Boolean variable, arity <= 3, unit featureValue): one warp per
// SELL slice with a uniform trip count.  f(k) = f(0) + k (f(1) - f(0)) comes from
// the two tables, so the gradient is an INTEGER.
// ---------------------------------------------------------------------------

// (two id ranges per call: the cell's PAIR rows and its FAST rows -- one copy of the code)
template <bool SMEM, class T>
__device__ __noinline__ void learn_tt_slices(const LearnArgs<T> &a, const LearnCtx<SMEM> &ctx, int beg0, int end0, int beg1, int end1,
                                             uint32_t kfree, uint32_t kevid, uint32_t ktrunc, int rot)
{
    const unsigned FULL = 0xFFFFFFFFu;
    const int lane = threadIdx.x & 31;
    const int64_t warp_global = blockIdx.x * (int64_t)NB_LWARPS + (threadIdx.x >> 5);
    const int64_t n_warps = (int64_t)gridDim.x * NB_LWARPS;
    const T *vF = a.val_free, *vE = a.val_evid;
    const int64_t s0b = beg0 >> 5, s0e = end0 > beg0 ? (((int64_t)end0 + 31) >> 5) : s0b;
    const int64_t s1b = beg1 >> 5, s1e = end1 > beg1 ? (((int64_t)end1 + 31) >> 5) : s1b;
    const int64_t ns0 = s0e - s0b, ns = ns0 + (s1e - s1b);

    int64_t it_first = warp_global + rot;
    if (it_first >= n_warps) it_first -= n_warps;
    for (int64_t it = it_first; it < ns; it += n_warps) {
        const bool first = it < ns0;
        const int64_t s = first ? s0b + it : s1b + (it - ns0);
        const int beg = first ? beg0 : beg1, end = first ? end0 : end1;
        const int64_t nid = (s << 5) + lane;
        const uint32_t meta = a.vmeta[nid];
        const uint32_t rid = a.rng_id[nid];
        const int evid = NB_META_EVID(meta);
        const bool valid = nid >= beg && nid < end && NB_META_VALID(meta) && evid != 4;   // learning.py:24-26
        const int64_t q0 = a.tt_ptr[s];
        const int n = (int)((a.tt_ptr[s + 1] - q0) >> 5);
        const uint4 *qp = a.tt + q0 + lane;
        const uint32_t *bp = a.tt_base + q0 + lane;
        const uint32_t *wp = a.tt_wid + q0 + lane;

        // ---- pass 1: e1 - e0 under both chains (current weights by id: the values inlined in the
        //      quads are only refreshed for the Gibbs sweep) ----
        double dF = 0.0, dE = 0.0;
        for (int j = 0; j < n; j += 2) {
            uint4 q[2];
            uint32_t wid[2];
#pragma unroll
            for (int t = 0; t < 2; t++) {
                q[t] = (j + t < n) ? __ldg(qp + (size_t)(j + t) * 32)
                                   : make_uint4((uint32_t)nid, (uint32_t)nid, NB_TT_NEUTRAL | NB_TT_FIXED_BIT, 0u);
                wid[t] = (j + t < n) ? __ldg(wp + (size_t)(j + t) * 32) : 0u;
            }
            int xf[2][2], xe[2][2];
            double w[2];
#pragma unroll
            for (int t = 0; t < 2; t++) {
                xf[t][0] = nb_ldv(vF, q[t].x); xf[t][1] = nb_ldv(vF, q[t].y);
                xe[t][0] = nb_ldv(vE, q[t].x); xe[t][1] = nb_ldv(vE, q[t].y);
                w[t] = ctx.weight(wid[t]);
            }
#pragma unroll
            for (int t = 0; t < 2; t++) {
                dF = fma(w[t], (double)nb_tt_diff(q[t].z, nb_tt_index(xf[t][0], xf[t][1])), dF);
                dE = fma(w[t], (double)nb_tt_diff(q[t].z, nb_tt_index(xe[t][0], xe[t][1])), dE);
            }
        }
        // ---- both samples (learning.py:53-69) ----
        int ev;
        if (evid != 1) {
            const double u = nb_philox2x32_u53(rid, (uint32_t)a.epoch, kevid);
            ev = u <= (double)(1.0f / (1.0f + __expf((float)dE))) ? 0 : 1;
        } else {
            ev = (int)a.vinit[nid];
        }
        const double uf = nb_philox2x32_u53(rid, (uint32_t)a.epoch, kfree);
        const int prop = uf <= (double)(1.0f / (1.0f + __expf((float)dF))) ? 0 : 1;
        if (valid) { a.val_evid[nid] = (T)ev; a.val_free[nid] = (T)prop; }
        const bool active = valid && (a.learn_non_evidence || evid == 1);        // :70-71
        uint32_t cinc = 1;
        if (a.regularization == 1)                                                // :90
            cinc = nb_philox2x32_u53(rid, (uint32_t)a.epoch, ktrunc) < 1.0 / a.truncation ? 1u : 0u;
        else if (a.regularization != 2) cinc = 0;

        // ---- pass 2: integer gradient of every learnable incidence (:97-125) ----
        if (__ballot_sync(FULL, active) == 0u) continue;
        for (int j = 0; j < n; j++) {
            const uint4 q = __ldg(qp + (size_t)j * 32);
            const uint32_t b = __ldg(bp + (size_t)j * 32);
            const uint32_t wid = __ldg(wp + (size_t)j * 32);
            // this variable's own slots are ignored by the tables (they may read its fresh values)
            const int iF = nb_tt_index(nb_ldv(vF, q.x), nb_ldv(vF, q.y)), iE = nb_tt_index(nb_ldv(vE, q.x), nb_ldv(vE, q.y));
            const int fF = ((int)((b >> (2 * iF)) & 3u) - 1) + prop * nb_tt_diff(q.z, iF);
            const int fE = ((int)((b >> (2 * iE)) & 3u) - 1) + ev * nb_tt_diff(q.z, iE);
            const bool contrib = active && !(q.z & NB_TT_FIXED_BIT);
            const unsigned who = __ballot_sync(FULL, contrib);
            if (who == 0u) continue;
            const int leader = __ffs(who) - 1;
            const uint32_t w0 = __shfl_sync(FULL, wid, leader);
            if (__all_sync(FULL, !contrib || wid == w0)) {
                const int G = __reduce_add_sync(FULL, contrib ? fF - fE : 0);
                const unsigned Cn = __reduce_add_sync(FULL, contrib ? cinc : 0u);
                if (lane == leader) ctx.add_int(w0, G, Cn);
            } else if (contrib) {
                ctx.add_int(wid, fF - fE, cinc);
            }
        }
    }
}

// Same algorithm, one WARP per row with the lanes striding over the row's quads: used when the
// rows are long (data-programming models: a label variable with ~100 labelling functions) or when
// a cell has fewer rows than the grid has warps.  A cell is a chain of dependent memory round trips
// (the work per cell is tiny), so the row is read ONCE: every lane issues all its loads up front
// (four incidences per lane and group: quad, weight id, f(0) table, then the member values of both
// chains), and keeps what the gradient needs -- f(0) and f(1) - f(0) under each chain, 10 bits --
// in registers until both samples are drawn.  Rows of more than NB_ROW_STASH * 32 incidences re-read
// their tail from memory.
#define NB_ROW_GROUP 4                       /* incidences per lane whose loads are in flight together */
#define NB_ROW_STASH (2 * NB_ROW_GROUP)      /* incidences per lane kept in registers */

__device__ __forceinline__ uint32_t nb_pack_grad(uint32_t table, uint32_t base, int iF, int iE, bool live)
{
    // [1:0] f(0)+1 free  [4:2] f(1)-f(0)+2 free  [6:5] f(0)+1 evid  [9:7] diff evid  [10] contributes
    return ((base >> (2 * iF)) & 3u) | (((table >> (3 * iF)) & 7u) << 2) | (((base >> (2 * iE)) & 3u) << 5) |
           (((table >> (3 * iE)) & 7u) << 7) | ((live ? 1u : 0u) << 10);
}
__device__ __forceinline__ int nb_grad_of(uint32_t p, int prop, int ev)
{
    const int fF = ((int)(p & 3u) - 1) + prop * ((int)((p >> 2) & 7u) - 2);
    const int fE = ((int)((p >> 5) & 3u) - 1) + ev * ((int)((p >> 7) & 7u) - 2);
    return fF - fE;
}

template <bool SMEM, class T>
__device__ __noinline__ void learn_tt_rows(const LearnArgs<T> &a, const LearnCtx<SMEM> &ctx, int beg0, int end0, int beg1, int end1,
                                           uint32_t kfree, uint32_t kevid, uint32_t ktrunc, int rot)
{
    const int lane = threadIdx.x & 31;
    const int64_t warp_global = blockIdx.x * (int64_t)NB_LWARPS + (threadIdx.x >> 5);
    const int64_t n_warps = (int64_t)gridDim.x * NB_LWARPS;
    const T *vF = a.val_free, *vE = a.val_evid;
    const int64_t n0 = max(end0 - beg0, 0), ntot = n0 + max(end1 - beg1, 0);

    int64_t it_first = warp_global + rot;
    if (it_first >= n_warps) it_first -= n_warps;          // rot < n_warps
    for (int64_t it = it_first; it < ntot; it += n_warps) {
        const int64_t nid = it < n0 ? beg0 + it : beg1 + (it - n0);
        const uint32_t meta = a.vmeta[nid];
        const uint32_t rid = a.rng_id[nid];
        const int vin = (int)a.vinit[nid];
        const int64_t s = nid >> 5;
        const int64_t q0 = a.tt_ptr[s];
        const int n = (int)((a.tt_ptr[s + 1] - q0) >> 5);
        const int evid = NB_META_EVID(meta);
        if (!NB_META_VALID(meta) || evid == 4) continue;                         // learning.py:24-26
        const uint4 *qp = a.tt + q0 + (nid & 31);
        const uint32_t *bp = a.tt_base + q0 + (nid & 31);
        const uint32_t *wp = a.tt_wid + q0 + (nid & 31);
        uint32_t st_g[NB_ROW_STASH], st_w[NB_ROW_STASH];
#pragma unroll
        for (int u = 0; u < NB_ROW_STASH; u++) { st_g[u] = 0u; st_w[u] = 0u; }
        double dF = 0.0, dE = 0.0;
        // ---- the row, NB_ROW_GROUP * 32 incidences at a time: all loads first ----
#pragma unroll
        for (int grp = 0; grp < NB_ROW_STASH / NB_ROW_GROUP; grp++) {
            if (grp * NB_ROW_GROUP * 32 < n) {
                uint4 q[NB_ROW_GROUP];
                uint32_t wid[NB_ROW_GROUP], b[NB_ROW_GROUP];
#pragma unroll
                for (int u = 0; u < NB_ROW_GROUP; u++) {
                    const int j = lane + 32 * (grp * NB_ROW_GROUP + u);
                    const bool in = j < n;
                    q[u] = in ? __ldg(qp + (size_t)j * 32) : make_uint4((uint32_t)nid, (uint32_t)nid, NB_TT_NEUTRAL | NB_TT_FIXED_BIT, 0u);
                    wid[u] = in ? __ldg(wp + (size_t)j * 32) : 0u;
                    b[u] = in ? __ldg(bp + (size_t)j * 32) : NB_TT_BASE_NEUTRAL;
                }
                int xf[NB_ROW_GROUP][2], xe[NB_ROW_GROUP][2];
#pragma unroll
                for (int u = 0; u < NB_ROW_GROUP; u++) {
                    xf[u][0] = nb_ldv(vF, q[u].x); xf[u][1] = nb_ldv(vF, q[u].y);
                    xe[u][0] = nb_ldv(vE, q[u].x); xe[u][1] = nb_ldv(vE, q[u].y);
                }
#pragma unroll
                for (int u = 0; u < NB_ROW_GROUP; u++) {
                    const int iF = nb_tt_index(xf[u][0], xf[u][1]), iE = nb_tt_index(xe[u][0], xe[u][1]);
                    const double w = ctx.weight(wid[u]);
                    dF = fma(w, (double)nb_tt_diff(q[u].z, iF), dF);
                    dE = fma(w, (double)nb_tt_diff(q[u].z, iE), dE);
                    st_g[grp * NB_ROW_GROUP + u] = nb_pack_grad(q[u].z, b[u], iF, iE, !(q[u].z & NB_TT_FIXED_BIT));
                    st_w[grp * NB_ROW_GROUP + u] = wid[u];
                }
            }
        }
        for (int j = lane + 32 * NB_ROW_STASH; j < n; j += 32) {                 // tail of a very long row
            const uint4 q = __ldg(qp + (size_t)j * 32);
            const double w = ctx.weight(__ldg(wp + (size_t)j * 32));
            dF = fma(w, (double)nb_tt_diff(q.z, nb_tt_index(nb_ldv(vF, q.x), nb_ldv(vF, q.y))), dF);
            dE = fma(w, (double)nb_tt_diff(q.z, nb_tt_index(nb_ldv(vE, q.x), nb_ldv(vE, q.y))), dE);
        }
        dF = nb_warp_sum(dF);
        dE = nb_warp_sum(dE);
        int ev;
        if (evid != 1) {
            const double u = nb_philox2x32_u53(rid, (uint32_t)a.epoch, kevid);
            ev = u <= (double)(1.0f / (1.0f + __expf((float)dE))) ? 0 : 1;
        } else {
            ev = vin;
        }
        const double uf = nb_philox2x32_u53(rid, (uint32_t)a.epoch, kfree);
        const int prop = uf <= (double)(1.0f / (1.0f + __expf((float)dF))) ? 0 : 1;
        __syncwarp();
        if (lane == 0) { a.val_evid[nid] = (T)ev; a.val_free[nid] = (T)prop; }
        if (!a.learn_non_evidence && evid != 1) continue;                        // :70-71
        uint32_t cinc = 1;
        if (a.regularization == 1)
            cinc = nb_philox2x32_u53(rid, (uint32_t)a.epoch, ktrunc) < 1.0 / a.truncation ? 1u : 0u;
        else if (a.regularization != 2) cinc = 0;
        // ---- integer gradients from the registers (:97-125) ----
#pragma unroll
        for (int u = 0; u < NB_ROW_STASH; u++)
            if (st_g[u] & (1u << 10)) ctx.add_int(st_w[u], nb_grad_of(st_g[u], prop, ev), cinc);
        for (int j = lane + 32 * NB_ROW_STASH; j < n; j += 32) {
            const uint4 q = __ldg(qp + (size_t)j * 32);
            if (q.z & NB_TT_FIXED_BIT) continue;
            const uint32_t b = __ldg(bp + (size_t)j * 32);
            // slots that point at the variable itself are ignored by the tables
            const int iF = nb_tt_index(nb_ldv(vF, q.x), nb_ldv(vF, q.y)), iE = nb_tt_index(nb_ldv(vE, q.x), nb_ldv(vE, q.y));
            ctx.add_int(__ldg(wp + (size_t)j * 32), nb_grad_of(nb_pack_grad(q.z, b, iF, iE, true), prop, ev), cinc);
        }
    }
}

// ---------------------------------------------------------------------------
// the persistent epoch kernel
// ---------------------------------------------------------------------------
// Grid barrier (the kernel is launched cooperatively: all CTAs are resident).  CTAs that wait back
// off with nanosleep instead of polling flat out: in a cell with fewer rows than warps most CTAs
// arrive at once and 100+ pollers hammering one L2 line slowed the CTAs still working.
__device__ __forceinline__ void nb_grid_sync(unsigned *bar)
{
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        const unsigned gen = *(volatile unsigned *)(bar + 1);      // generation BEFORE arriving
        if (atomicAdd(bar, 1u) == gridDim.x - 1) {
            *(volatile unsigned *)bar = 0u;
            __threadfence();
            atomicAdd(bar + 1, 1u);
        } else {
            unsigned ns = 20;
            while (*(volatile unsigned *)(bar + 1) == gen) { __nanosleep(ns); if (ns < 320) ns *= 2; }
        }
        __threadfence();
    }
    __syncthreads();
}

// (1-byte graphs only: 2-byte graphs learn in throughput mode)
template <bool WIDE, bool SMEM>
__global__ void __launch_bounds__(NB_LEARN_THREADS) k_learn_cells(LearnArgs<nb_val_t> a, CellPlan plan, int cell_beg, int cell_end,
                                                                  int only_color)
{
    extern __shared__ unsigned char s_raw[];
    __shared__ double s_e[NB_LWARPS][NB_MAX_CARD + 1];
    __shared__ int s_rng[2][2 * NB_N_CLASSES];
    const int W = a.W;
    // shared layout (SMEM): weights f64 [W] | fixed-point sums i64 [W] | integer sums i32 [W] | counts u32 [W]
    double *s_w = (double *)s_raw;
    nb_fix_t *s_gf = (nb_fix_t *)(s_raw + (size_t)8 * (SMEM ? W : 0));
    int32_t *s_gi = (int32_t *)(s_raw + (size_t)16 * (SMEM ? W : 0));
    uint32_t *s_cnt = (uint32_t *)(s_raw + (size_t)20 * (SMEM ? W : 0));
    if (SMEM) {
        for (int w = threadIdx.x; w < W; w += blockDim.x) { s_w[w] = __ldcg(a.weight + w); s_gf[w] = 0; s_gi[w] = 0; s_cnt[w] = 0u; }
        __syncthreads();
    }
    const uint32_t kf = nb_fold_key(a.seed, a.epoch, NB_TAG_FREE), ke = nb_fold_key(a.seed, a.epoch, NB_TAG_EVID),
                   kt = nb_fold_key(a.seed, a.epoch, NB_TAG_TRUNC);

    int k = 0;   // cells processed so far in this launch (uniform across the grid): picks the rotating table
    for (int cell = cell_beg; cell < cell_end; cell++) {
        // cells enumerate (block, colour) with the colour running fastest; only_color >= 0: the
        // caller drives the colours itself (partitioned graphs) and `cell` is the block
        const int block = only_color >= 0 ? cell : cell / plan.n_colors;
        const int color = only_color >= 0 ? only_color : cell % plan.n_colors;
        const bool tr = a.trace != nullptr && threadIdx.x == 0;
        unsigned long long t0 = tr ? nb_now() : 0ull, t1;
        // The cell's id ranges (64-bit divisions and dependent loads) come from shared memory: five
        // threads of the LAST warp looked them up while the previous cell was being processed.
        __syncthreads();
        if (cell == cell_beg) {
            if (threadIdx.x < NB_N_CLASSES) nb_plan_range(plan, (int)threadIdx.x, color, block, s_rng[cell & 1][2 * threadIdx.x], s_rng[cell & 1][2 * threadIdx.x + 1]);
            __syncthreads();
        }
        {
            const int t = (int)threadIdx.x - (NB_LEARN_THREADS - 32);
            if (t >= 0 && t < NB_N_CLASSES && cell + 1 < cell_end) {
                const int nblock = only_color >= 0 ? cell + 1 : (cell + 1) / plan.n_colors;
                const int ncolor = only_color >= 0 ? only_color : (cell + 1) % plan.n_colors;
                nb_plan_range(plan, t, ncolor, nblock, s_rng[(cell + 1) & 1][2 * t], s_rng[(cell + 1) & 1][2 * t + 1]);
            }
        }
        const int *rng = s_rng[cell & 1];
        const int pb = rng[2 * NB_CLASS_PAIR], pe = rng[2 * NB_CLASS_PAIR + 1], fb = rng[2 * NB_CLASS_FAST],
                  fe = rng[2 * NB_CLASS_FAST + 1], cb = rng[2 * NB_CLASS_CAT], ce = rng[2 * NB_CLASS_CAT + 1],
                  tb = rng[2 * NB_CLASS_GEN], te = rng[2 * NB_CLASS_GEN + 1];
        int wb = rng[2 * NB_CLASS_WARP], we = rng[2 * NB_CLASS_WARP + 1];
        wb -= (int)plan.n_trows;          // warp rows are addressed by their index
        we -= (int)plan.n_trows;
        if (pe <= pb && fe <= fb && ce <= cb && te <= tb && we <= wb) continue;   // uniform across the grid
        const int slot = k % 3;
        nb_fix_t *g_gf = a.g_grad + (size_t)slot * W;
        uint32_t *g_cn = a.g_cnt + (size_t)slot * W;
        LearnCtx<SMEM> ctx;
        ctx.w = SMEM ? s_w : a.weight;
        ctx.gi = s_gi;
        ctx.gf = SMEM ? s_gf : g_gf;
        ctx.cnt = SMEM ? s_cnt : g_cn;

        // the table of the NEXT cell is cleared now: its last readers (cell k - 2) passed the previous
        // barrier, its next writers (cell k + 1) start after this cell's barrier.  Table 0 is cleared
        // by the host before the launch.
        {
            nb_fix_t *z_gf = a.g_grad + (size_t)((k + 1) % 3) * W;
            uint32_t *z_cn = a.g_cnt + (size_t)((k + 1) % 3) * W;
            for (int64_t w = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; w < W; w += (int64_t)gridDim.x * blockDim.x) {
                z_gf[w] = 0;
                z_cn[w] = 0u;
            }
        }
        const unsigned long long t_begin = t0;
#define NB_TRACE(i) if (a.trace != nullptr) { __syncthreads(); if (tr) { t1 = nb_now(); atomicAdd(a.trace + (i), t1 - t0); \
            if ((i) == 1 || (i) == 2) a.trace_cta[3 * blockIdx.x + (i) - 1] += t1 - t0; t0 = t1; } }
        NB_TRACE(0)
        if (pe > pb || fe > fb) {
            // One warp per row when the rows are long -- or when the cell holds fewer truth-table rows
            // than the grid has warps, whatever their length: a thread walking a 100-incidence row on
            // its own is a chain of 100 dependent loads (the 1 % of label variables that the
            // colouring puts with the labelling functions kept one warp busy for 150 us per cell
            // while 2367 others waited at the barrier).
            const int64_t n_warps = (int64_t)gridDim.x * NB_LWARPS;
            const bool by_row = plan.long_rows[color] != 0 || (int64_t)(pe - pb) + (fe - fb) <= 2 * n_warps;
            // the first row of the cell goes to a different warp every cell: the idle CTAs rotate
            const int rot = (int)(((int64_t)k * 37 * NB_LWARPS) % n_warps);
            if (by_row) learn_tt_rows<SMEM>(a, ctx, pb, pe, fb, fe, kf, ke, kt, rot);
            else learn_tt_slices<SMEM>(a, ctx, pb, pe, fb, fe, kf, ke, kt, rot);
        }
        NB_TRACE(1)
        if (ce > cb) learn_cat_rows<SMEM>(a, ctx, cb, ce, kf, ke);
        if (te > tb) learn_thread_rows<WIDE, SMEM>(a, ctx, 0, 0, tb, te);
        NB_TRACE(2)
        if (we > wb) learn_warp_rows<WIDE, SMEM>(a, ctx, s_e[threadIdx.x >> 5], wb, we);
        NB_TRACE(3)

        if (SMEM) {
            // flush this CTA's tables: one integer atomic per touched weight
            __syncthreads();
            for (int w = threadIdx.x; w < W; w += blockDim.x) {
                const nb_fix_t gsum = s_gf[w] + ((nb_fix_t)s_gi[w] << NB_GRAD_SHIFT);
                const uint32_t c = s_cnt[w];
                if (gsum) atomicAdd((unsigned long long *)(g_gf + w), (unsigned long long)gsum);
                if (c) atomicAdd(g_cn + w, c);
                s_gf[w] = 0; s_gi[w] = 0; s_cnt[w] = 0u;
            }
        }
        NB_TRACE(4)
        if (tr) { atomicMax(a.trace_cell + (cell - cell_beg), t0 - t_begin); a.trace_cta[3 * blockIdx.x + 2] += t0 - t_begin; }
        nb_grid_sync(a.bar);     // (fences the CTAs' writes: values, tables)
        NB_TRACE(5)
        if (SMEM) {
            // every CTA applies the same sums to its own copy of the weights; CTA 0 publishes them
            for (int w = threadIdx.x; w < W; w += blockDim.x) {
                const nb_fix_t Gi = __ldcg(g_gf + w);
                const uint32_t n = __ldcg(g_cn + w);
                if ((Gi != 0 || n != 0u) && !a.wfixed[w]) {
                    const double nw = nb_apply_update(s_w[w], (double)Gi * (1.0 / NB_GRAD_UNIT), n, a.regularization, a.step,
                                                      a.reg_param, a.truncation);
                    s_w[w] = nw;
                    if (blockIdx.x == 0) a.weight[w] = nw;
                }
            }
            __syncthreads();
        } else {
            for (int64_t w = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; w < W; w += (int64_t)gridDim.x * blockDim.x) {
                const nb_fix_t Gi = __ldcg(g_gf + w);
                const uint32_t n = __ldcg(g_cn + w);
                if ((Gi != 0 || n != 0u) && !a.wfixed[w])
                    __stcg(a.weight + w, nb_apply_update(__ldcg(a.weight + w), (double)Gi * (1.0 / NB_GRAD_UNIT), n,
                                                        a.regularization, a.step, a.reg_param, a.truncation));
            }
            nb_grid_sync(a.bar);
        }
        NB_TRACE(6)
        if (tr && blockIdx.x == 0) { atomicAdd(a.trace + 7, 1ull); atomicAdd(a.trace + 8, a.trace_cell[cell - cell_beg]); }
#undef NB_TRACE
        k++;
    }
}

// ---------------------------------------------------------------------------
// Throughput mode.  When a cell holds far more rows than the persistent grid has threads (big graphs
// with moderate tying: the KBC and categorical shapes), latency per cell does not matter and
// occupancy does: the persistent kernel carries every row class and needs 128 registers (two CTAs
// per SM).  Such cells are run as ordinary launches of one lean kernel per row class -- the same
// device functions, 64-register budgets, full grids -- plus one apply kernel; a handful of launches
// per cell is nothing against cells of hundreds of microseconds.
// ---------------------------------------------------------------------------
template <bool SMEM, class T>
__device__ __forceinline__ LearnCtx<SMEM> nb_lean_ctx(const LearnArgs<T> &a, unsigned char *s_raw, int slot)
{
    const int W = a.W;
    double *s_w = (double *)s_raw;
    nb_fix_t *s_gf = (nb_fix_t *)(s_raw + (size_t)8 * (SMEM ? W : 0));
    int32_t *s_gi = (int32_t *)(s_raw + (size_t)16 * (SMEM ? W : 0));
    uint32_t *s_cnt = (uint32_t *)(s_raw + (size_t)20 * (SMEM ? W : 0));
    if (SMEM) {
        for (int w = threadIdx.x; w < W; w += blockDim.x) { s_w[w] = a.weight[w]; s_gf[w] = 0; s_gi[w] = 0; s_cnt[w] = 0u; }
        __syncthreads();
    }
    LearnCtx<SMEM> ctx;
    ctx.w = SMEM ? s_w : a.weight;
    ctx.gi = s_gi;
    ctx.gf = SMEM ? s_gf : a.g_grad + (size_t)slot * W;
    ctx.cnt = SMEM ? s_cnt : a.g_cnt + (size_t)slot * W;
    return ctx;
}

template <bool SMEM, class T>
__device__ __forceinline__ void nb_lean_flush(const LearnArgs<T> &a, const LearnCtx<SMEM> &ctx, int slot)
{
    if (!SMEM) return;
    __syncthreads();
    nb_fix_t *g_gf = a.g_grad + (size_t)slot * a.W;
    uint32_t *g_cn = a.g_cnt + (size_t)slot * a.W;
    for (int w = threadIdx.x; w < a.W; w += blockDim.x) {
        const nb_fix_t gsum = ctx.gf[w] + ((nb_fix_t)ctx.gi[w] << NB_GRAD_SHIFT);
        const uint32_t c = ctx.cnt[w];
        if (gsum) atomicAdd((unsigned long long *)(g_gf + w), (unsigned long long)gsum);
        if (c) atomicAdd(g_cn + w, c);
    }
}

template <bool SMEM, class T>
__global__ void __launch_bounds__(NB_LEARN_THREADS, 3) k_cell_tt(LearnArgs<T> a, int pb, int pe, int fb, int fe, int by_row, int slot,
                                                                 uint32_t kf, uint32_t ke, uint32_t kt)
{
    extern __shared__ unsigned char s_raw[];
    const LearnCtx<SMEM> ctx = nb_lean_ctx<SMEM, T>(a, s_raw, slot);
    if (by_row) learn_tt_rows<SMEM>(a, ctx, pb, pe, fb, fe, kf, ke, kt, 0);
    else learn_tt_slices<SMEM>(a, ctx, pb, pe, fb, fe, kf, ke, kt, 0);
    nb_lean_flush<SMEM, T>(a, ctx, slot);
}

template <bool WIDE, bool SMEM, class T>
__global__ void __launch_bounds__(NB_LEARN_THREADS, 4) k_cell_thread(LearnArgs<T> a, int tb, int te, int slot)
{
    extern __shared__ unsigned char s_raw[];
    const LearnCtx<SMEM> ctx = nb_lean_ctx<SMEM, T>(a, s_raw, slot);
    learn_thread_rows<WIDE, SMEM>(a, ctx, 0, 0, tb, te);
    nb_lean_flush<SMEM, T>(a, ctx, slot);
}

template <bool SMEM, class T>
__global__ void __launch_bounds__(NB_LEARN_THREADS, 4) k_cell_cat(LearnArgs<T> a, int cb, int ce, int slot, uint32_t kf, uint32_t ke)
{
    extern __shared__ unsigned char s_raw[];
    const LearnCtx<SMEM> ctx = nb_lean_ctx<SMEM, T>(a, s_raw, slot);
    learn_cat_rows<SMEM>(a, ctx, cb, ce, kf, ke);
    nb_lean_flush<SMEM, T>(a, ctx, slot);
}

template <bool WIDE, bool SMEM, class T>
__global__ void __launch_bounds__(NB_LEARN_THREADS, 2) k_cell_warp(LearnArgs<T> a, int wb, int we, int slot)
{
    extern __shared__ unsigned char s_raw[];
    __shared__ double s_e[NB_LWARPS][NB_MAX_CARD + 1];
    const LearnCtx<SMEM> ctx = nb_lean_ctx<SMEM, T>(a, s_raw, slot);
    learn_warp_rows<WIDE, SMEM>(a, ctx, s_e[threadIdx.x >> 5], wb, we);
    nb_lean_flush<SMEM, T>(a, ctx, slot);
}

// apply the cell's sums to the global weights and clear the table for its next use
template <class T>
__global__ void k_cell_apply(LearnArgs<T> a, int slot)
{
    nb_fix_t *g_gf = a.g_grad + (size_t)slot * a.W;
    uint32_t *g_cn = a.g_cnt + (size_t)slot * a.W;
    for (int64_t w = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; w < a.W; w += (int64_t)gridDim.x * blockDim.x) {
        const nb_fix_t Gi = g_gf[w];
        const uint32_t n = g_cn[w];
        if (Gi == 0 && n == 0u) continue;
        g_gf[w] = 0;
        g_cn[w] = 0u;
        if (!a.wfixed[w])
            a.weight[w] = nb_apply_update(a.weight[w], (double)Gi * (1.0 / NB_GRAD_UNIT), n, a.regularization, a.step,
                                          a.reg_param, a.truncation);
    }
}

// visits per weight of one colour (upper bound: every incidence of a learnable row)
struct RowRanges {
    int beg[4], end[4];    // thread-row id ranges (PAIR, FAST, CAT, GEN)
    int wbeg, wend;        // warp rows
};

template <bool WIDE, class T>
__global__ void k_visit_histogram(LearnArgs<T> a, RowRanges rr, uint32_t *hist)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    int64_t nid = -1;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int64_t n = rr.end[k] - rr.beg[k];
        if (nid < 0 && i >= 0 && i < n) nid = rr.beg[k] + i;
        if (nid < 0) i -= n;
    }
    if (nid < 0) {
        if (i >= rr.wend - rr.wbeg) return;
        nid = a.n_trows + rr.wbeg + i;
    }
    const uint32_t meta = a.vmeta[nid];
    const int evid = NB_META_EVID(meta);
    if (!NB_META_VALID(meta) || evid == 4) return;
    if (!a.learn_non_evidence && evid != 1) return;
    NbRow r = nid < a.n_trows ? nb_thread_row(a.twords, a.slice_ptr, nid) : nb_warp_row(a.wwords, a.wrow_ptr, nid - a.n_trows);
    int len = nid < a.n_trows ? NB_META_ROWLEN(meta)
                              : (int)(a.wrow_ptr[nid - a.n_trows + 1] - a.wrow_ptr[nid - a.n_trows]);
    int pos = 0;
    while (pos < len) {
        NbHdr h = nb_read_hdr<WIDE>(r, pos);
        if (h.code != C_MARK && !h.fixed) atomicAdd(hist + h.wid, 1u);
        pos += nb_inc_words<WIDE>(h);
    }
}

__global__ void k_max_u32(const uint32_t *x, int n, uint32_t *out)
{
    uint32_t m = 0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) m = max(m, x[i]);
    atomicMax(out, m);
}

// ---------------------------------------------------------------------------
// host driver
// ---------------------------------------------------------------------------
template <class T>
static LearnArgs<T> learn_args(nb_graph *g)
{
    LearnArgs<T> a{};
    a.vmeta = g->d_vmeta; a.slice_ptr = g->d_slice_ptr; a.twords = g->d_twords;
    a.wrow_ptr = g->d_wrow_ptr; a.wwords = g->d_wwords; a.inc_ptr = g->d_inc_ptr; a.inc = g->d_inc;
    a.rng_id = g->d_rng_id; a.vinit = (const T *)g->d_vinit; a.val_free = nb_vals<T>(g, 0); a.val_evid = nb_vals<T>(g, 1);
    if constexpr (sizeof(T) > 1) a.vcard = g->d_vcard;
    a.weight = g->d_weight; a.wfixed = g->d_wfixed; a.n_trows = g->n_trows; a.W = (int)g->W;
    a.g_grad = g->d_grad; a.g_cnt = g->d_nvis; a.bar = g->d_learn_bar;
    a.tt_ptr = g->d_tt_ptr; a.tt = g->d_tt; a.tt_base = g->d_tt_base; a.tt_wid = g->d_tt_wid;
    a.cat_ptr = g->d_cat_ptr; a.cat = g->d_cat; a.cat_wid = g->d_cat_wid; a.cat_first = g->n_frows;
    return a;
}

static int ensure_learn_buffers(nb_graph *g)
{
    if (!g->d_grad) {
        NB_TRY(nb_alloc(g, &g->d_grad, 3 * (size_t)std::max<int64_t>(g->W, 1)));     // three rotating tables, zeroed
        NB_TRY(nb_alloc(g, &g->d_nvis, 3 * (size_t)std::max<int64_t>(g->W, 1)));
        NB_TRY(nb_alloc(g, &g->d_learn_bar, 64));
    }
    return NB_OK;
}

// max over weights of the gradient visits one sweep of colour c can make
template <class T>
static int color_visit_bounds(nb_graph *g, LearnArgs<T> a, std::vector<int64_t> &out)
{
    out.assign((size_t)g->n_colors, 0);
    uint32_t *d_max, *d_hist;
    NB_TRY(nb_alloc(g, &d_max, 1));
    NB_CUDA(cudaMalloc(&d_hist, (size_t)std::max<int64_t>(g->W, 1) * 4));
    int rc = NB_OK;
    for (int c = 0; c < g->n_colors && rc == NB_OK; c++) {
        const NbColorRange &cr = g->colors[(size_t)c];
        RowRanges rr;
        rr.beg[0] = cr.p_beg; rr.end[0] = cr.p_end; rr.beg[1] = cr.f_beg; rr.end[1] = cr.f_end;
        rr.beg[2] = cr.c_beg; rr.end[2] = cr.c_end; rr.beg[3] = cr.t_beg; rr.end[3] = cr.t_end;
        rr.wbeg = cr.w_beg; rr.wend = cr.w_end;
        int64_t n = (cr.p_end - cr.p_beg) + (cr.f_end - cr.f_beg) + (cr.c_end - cr.c_beg) + (cr.t_end - cr.t_beg) +
                    (cr.w_end - cr.w_beg);
        if (n == 0) continue;
        cudaMemsetAsync(d_hist, 0, (size_t)g->W * 4, g->stream);
        cudaMemsetAsync(d_max, 0, 4, g->stream);
        unsigned grid = (unsigned)((n + 255) / 256);
        if (g->wide) k_visit_histogram<true, T><<<grid, 256, 0, g->stream>>>(a, rr, d_hist);
        else k_visit_histogram<false, T><<<grid, 256, 0, g->stream>>>(a, rr, d_hist);
        k_max_u32<<<64, 256, 0, g->stream>>>(d_hist, (int)g->W, d_max);
        uint32_t m = 0;
        cudaMemcpyAsync(&m, d_max, 4, cudaMemcpyDeviceToHost, g->stream);
        if (cudaStreamSynchronize(g->stream) != cudaSuccess) rc = NB_ERR_CUDA;
        out[(size_t)c] = m;
    }
    cudaFree(d_hist);
    if (rc != NB_OK) NB_FAIL(NB_ERR_CUDA, "visit histogram failed: %s", cudaGetErrorString(cudaGetLastError()));
    return NB_OK;
}

// per-graph cache of the visit bounds (depends on learn_non_evidence) and the device-side plan data
template <class T>
static int learn_prepare(nb_graph *g, LearnArgs<T> &a, std::vector<int64_t> &vmax, int learn_non_evidence)
{
    NB_TRY(ensure_learn_buffers(g));
    a = learn_args<T>(g);
    a.learn_non_evidence = learn_non_evidence;
    if (g->learn_vmax_flag != learn_non_evidence || (int)g->learn_vmax.size() != g->n_colors) {
        NB_TRY(color_visit_bounds(g, a, g->learn_vmax));
        g->learn_vmax_flag = learn_non_evidence;
    }
    vmax = g->learn_vmax;
    if (!g->d_long_rows) {
        std::vector<uint8_t> lr((size_t)std::max(g->n_colors, 1), 0);
        for (int c = 0; c < g->n_colors; c++) {
            const NbColorRange &cr = g->colors[(size_t)c];
            const int64_t rows = (cr.p_end - cr.p_beg) + (cr.f_end - cr.f_beg) + (cr.c_end - cr.c_beg) + (cr.t_end - cr.t_beg) +
                                 (cr.w_end - cr.w_beg);
            // truth-table rows of this colour average >= 16 incidences: spread each row over a warp
            lr[(size_t)c] = ((cr.p_end - cr.p_beg) + (cr.f_end - cr.f_beg)) > 0 && cr.edges >= 16 * rows;
        }
        g->learn_long_rows = lr;
        NB_TRY(nb_alloc(g, &g->d_long_rows, lr.size(), false));
        NB_CUDA(cudaMemcpyAsync(g->d_long_rows, lr.data(), lr.size(), cudaMemcpyHostToDevice, g->stream));
        NB_CUDA(cudaStreamSynchronize(g->stream));
    }
    return NB_OK;
}

// Mini-batch size: at most this many visits of any one weight between two applications.  The
// reference applies every visit immediately (learning.py:110-125); a batch of n visits with a
// stale weight moves it by about step * n * E[g], which must stay small against the scale on
// which the gradient itself changes or strongly driven transients overshoot (and L1 then traps
// the weights at 0).  step * n <= 0.25 keeps the batched trajectory on the per-visit one
// (measured against the CPU reference port on the labelling-function model, tools/lf_check.py).
static int64_t default_batch_visits(double step, int64_t batch_visits)
{
    return batch_visits > 0 ? batch_visits : (int64_t)std::max(1.0, std::floor(0.25 / std::max(std::fabs(step), 1e-12)));
}

// Number of id blocks per epoch: enough that no weight collects more than the batch bound in a block.
// NOT capped at the number of id windows: when one window already exceeds the bound (a weight tied
// across a large graph) the plan cuts the windows further (CellPlan::k_sub).
static int block_count(const nb_graph *g, const std::vector<int64_t> &vmax, int64_t bv)
{
    int64_t total = 0;
    for (int64_t v : vmax) total += v;       // a weight can be visited from every colour inside a block
    int64_t nb = std::max<int64_t>(1, (total + bv - 1) / bv);
    const int64_t cap = std::max<int64_t>(1, std::min<int64_t>(g->V, 1ll << 30));   // one variable per cell at the very least
    return (int)std::min<int64_t>(nb, cap);
}

static CellPlan make_plan(const nb_graph *g, int n_blocks)
{
    CellPlan p;
    p.win_start = g->d_win_start;
    p.long_rows = g->d_long_rows;
    p.n_win = g->n_win;
    p.n_colors = g->n_colors;
    p.n_blocks = std::max(1, n_blocks);
    p.k_sub = (int)std::max<int64_t>(1, ((int64_t)p.n_blocks + g->n_win - 1) / std::max<int64_t>(g->n_win, 1));
    p.n_trows = g->n_trows;
    return p;
}

int nb_learn_block_count(nb_graph *g, double step, int learn_non_evidence, int64_t batch_visits, int *n_blocks)
{
    std::vector<int64_t> vmax;
    if (g->value_bytes == 1) {
        LearnArgs<nb_val_t> a;
        NB_TRY(learn_prepare(g, a, vmax, learn_non_evidence));
    } else {
        LearnArgs<nb_val16_t> a;
        NB_TRY(learn_prepare(g, a, vmax, learn_non_evidence));
    }
    *n_blocks = block_count(g, vmax, default_batch_visits(step, batch_visits));
    return NB_OK;
}

template <bool WIDE, bool SMEM>
static int launch_cells_t(nb_graph *g, LearnArgs<nb_val_t> a, CellPlan plan, int cell_beg, int cell_end, int only_color)
{
    const size_t smem = SMEM ? (size_t)g->W * 24 : 0;
    auto kern = k_learn_cells<WIDE, SMEM>;
    if (smem > 32 * 1024) NB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0, sms = 0;
    NB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, NB_LEARN_THREADS, smem));
    NB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, g->device));
    if (per_sm < 1) NB_FAIL(NB_ERR_CUDA, "the learning kernel does not fit on an SM");
    // all CTAs must be co-resident (grid barrier); two per SM hide each other's latencies
    const int grid = sms * std::min(per_sm, 2);
    static const bool trace_on = [] { const char *e = getenv("NUMBSKULL_B200_LEARN_TRACE"); return e && atoi(e) != 0; }();
    unsigned long long *d_trace = nullptr;
    if (trace_on) {
        const size_t n = 64 + 3 * 4096 + (size_t)(cell_end - cell_beg);
        NB_CUDA(cudaMalloc(&d_trace, n * 8));
        NB_CUDA(cudaMemsetAsync(d_trace, 0, n * 8, g->stream));
        a.trace = d_trace;
        a.trace_cta = d_trace + 64;
        a.trace_cell = d_trace + 64 + 3 * 4096;
    }
    NB_CUDA(cudaMemsetAsync(a.g_grad, 0, (size_t)g->W * sizeof(nb_fix_t), g->stream));   // rotating table 0
    NB_CUDA(cudaMemsetAsync(a.g_cnt, 0, (size_t)g->W * sizeof(uint32_t), g->stream));
    void *args[] = {&a, &plan, &cell_beg, &cell_end, &only_color};
    NB_CUDA(cudaLaunchCooperativeKernel((void *)kern, dim3((unsigned)grid), dim3(NB_LEARN_THREADS), args, smem, g->stream));
    g->launches++;
    if (d_trace) {
        std::vector<unsigned long long> hv(64 + 3 * 4096 + (size_t)std::min(cell_end - cell_beg, 4096));
        if (false) {}
        unsigned long long *h = hv.data();
        NB_CUDA(cudaMemcpyAsync(h, d_trace, hv.size() * 8, cudaMemcpyDeviceToHost, g->stream));
        NB_CUDA(cudaStreamSynchronize(g->stream));
        cudaFree(d_trace);
        {
            std::vector<std::pair<unsigned long long, int>> tot;
            for (int b = 0; b < grid && b < 4096; b++) tot.push_back({h[64 + 3 * b + 2], b});
            std::sort(tot.begin(), tot.end());
            fprintf(stderr, "[learn trace] per-CTA work (ms): min %.3f (cta %d) median %.3f max %.3f (cta %d); slowest CTAs:",
                    1e-6 * tot.front().first, tot.front().second, 1e-6 * tot[tot.size() / 2].first, 1e-6 * tot.back().first,
                    tot.back().second);
            for (size_t i = tot.size() > 6 ? tot.size() - 6 : 0; i < tot.size(); i++)
                fprintf(stderr, " %d: tt %.3f thr %.3f all %.3f;", tot[i].second, 1e-6 * h[64 + 3 * tot[i].second],
                        1e-6 * h[64 + 3 * tot[i].second + 1], 1e-6 * tot[i].first);
            fprintf(stderr, "\n");
            {
                const int nc = std::min(cell_end - cell_beg, 4096), ncol = std::max(plan.n_colors, 1);
                std::vector<double> sum((size_t)ncol, 0.0), cnt((size_t)ncol, 0.0);
                for (int c = 0; c < nc; c++) { sum[(size_t)(c % ncol)] += 1e-3 * h[64 + 3 * 4096 + c]; cnt[(size_t)(c % ncol)] += 1; }
                fprintf(stderr, "[learn trace] slowest CTA's work per cell by colour (us):");
                for (int c = 0; c < ncol && c < 12; c++) fprintf(stderr, " %.1f", sum[(size_t)c] / std::max(cnt[(size_t)c], 1.0));
                fprintf(stderr, "\n");
            }
        }
        const double cells = (double)std::max<unsigned long long>(h[7], 1), per = 1e-3 / (cells * grid);
        fprintf(stderr, "[learn trace] %d CTAs, %.0f cells; us per cell and CTA: lookup %.2f, tt rows %.2f, thread rows %.2f, "
                        "warp rows %.2f, flush %.2f, barrier wait %.2f, apply %.2f; slowest CTA's work per cell %.2f us\n",
                grid, cells, h[0] * per, h[1] * per, h[2] * per, h[3] * per, h[4] * per, h[5] * per, h[6] * per,
                1e-3 * (double)h[8] / cells);
    }
    return NB_OK;
}

static int launch_cells(nb_graph *g, const LearnArgs<nb_val_t> &a, const CellPlan &plan, int cell_beg, int cell_end, int only_color)
{
    const bool smem = g->W <= NB_LEARN_SMEM_W;
    if (g->wide) return smem ? launch_cells_t<true, true>(g, a, plan, cell_beg, cell_end, only_color)
                             : launch_cells_t<true, false>(g, a, plan, cell_beg, cell_end, only_color);
    return smem ? launch_cells_t<false, true>(g, a, plan, cell_beg, cell_end, only_color)
                : launch_cells_t<false, false>(g, a, plan, cell_beg, cell_end, only_color);
}

// one cell as ordinary launches (throughput mode)
template <bool WIDE, bool SMEM, class T>
static int launch_cell_lean_t(nb_graph *g, const LearnArgs<T> &a, const CellPlan &plan, int block, int color)
{
    CellPlan hp = plan;
    hp.win_start = g->win_start.data();            // host copy of the window table
    int rng[2 * NB_N_CLASSES];
    for (int cls = 0; cls < NB_N_CLASSES; cls++) nb_plan_range(hp, cls, color, block, rng[2 * cls], rng[2 * cls + 1]);
    const int pb = rng[2 * NB_CLASS_PAIR], pe = rng[2 * NB_CLASS_PAIR + 1], fb = rng[2 * NB_CLASS_FAST], fe = rng[2 * NB_CLASS_FAST + 1],
              cb = rng[2 * NB_CLASS_CAT], ce = rng[2 * NB_CLASS_CAT + 1], tb = rng[2 * NB_CLASS_GEN], te = rng[2 * NB_CLASS_GEN + 1];
    const int wb = rng[2 * NB_CLASS_WARP] - (int)g->n_trows, we = rng[2 * NB_CLASS_WARP + 1] - (int)g->n_trows;
    if (pe <= pb && fe <= fb && ce <= cb && te <= tb && we <= wb) return NB_OK;
    const size_t smem = SMEM ? (size_t)g->W * 24 : 0;
    int sms = 0;
    NB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, g->device));
    // shared-memory tables are flushed once per CTA: fewer, longer-lived CTAs (the loops are grid-stride)
    const int64_t cap = (int64_t)sms * (SMEM ? 8 : 32);
    const uint32_t kf = nb_fold_key(a.seed, a.epoch, NB_TAG_FREE), ke = nb_fold_key(a.seed, a.epoch, NB_TAG_EVID),
                   kt = nb_fold_key(a.seed, a.epoch, NB_TAG_TRUNC);
    if (smem > 32 * 1024) {
        NB_CUDA(cudaFuncSetAttribute(k_cell_tt<SMEM, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        NB_CUDA(cudaFuncSetAttribute(k_cell_thread<WIDE, SMEM, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        NB_CUDA(cudaFuncSetAttribute(k_cell_cat<SMEM, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        NB_CUDA(cudaFuncSetAttribute(k_cell_warp<WIDE, SMEM, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    if (pe > pb || fe > fb) {
        const int64_t rows = (int64_t)(pe - pb) + (fe - fb);
        const int by_row = (g->learn_long_rows[(size_t)color] || rows <= 2 * cap * NB_LWARPS) ? 1 : 0;
        const int64_t need = by_row ? (rows + NB_LWARPS - 1) / NB_LWARPS : (rows / 32 + 2 + NB_LWARPS - 1) / NB_LWARPS;
        k_cell_tt<SMEM, T><<<(unsigned)std::max<int64_t>(1, std::min(need, cap)), NB_LEARN_THREADS, smem, g->stream>>>(
            a, pb, pe, fb, fe, by_row, 0, kf, ke, kt);
        g->launches++;
    }
    if (ce > cb) {
        const int64_t need = ((int64_t)(ce - cb) + NB_LEARN_THREADS - 1) / NB_LEARN_THREADS;
        k_cell_cat<SMEM, T><<<(unsigned)std::max<int64_t>(1, std::min(need, cap)), NB_LEARN_THREADS, smem, g->stream>>>(a, cb, ce, 0, kf, ke);
        g->launches++;
    }
    if (te > tb) {
        const int64_t need = ((int64_t)(te - tb) + NB_LEARN_THREADS - 1) / NB_LEARN_THREADS;
        k_cell_thread<WIDE, SMEM, T><<<(unsigned)std::max<int64_t>(1, std::min(need, cap)), NB_LEARN_THREADS, smem, g->stream>>>(a, tb, te, 0);
        g->launches++;
    }
    if (we > wb) {
        const int64_t need = ((int64_t)(we - wb) + NB_LWARPS - 1) / NB_LWARPS;
        k_cell_warp<WIDE, SMEM, T><<<(unsigned)std::max<int64_t>(1, std::min(need, cap)), NB_LEARN_THREADS, smem, g->stream>>>(a, wb, we, 0);
        g->launches++;
    }
    k_cell_apply<T><<<(unsigned)std::max<int64_t>(1, std::min<int64_t>((g->W + 255) / 256, cap)), 256, 0, g->stream>>>(a, 0);
    g->launches++;
    return NB_OK;
}

template <class T>
static int launch_cell_lean(nb_graph *g, const LearnArgs<T> &a, const CellPlan &plan, int block, int color)
{
    const bool smem = g->W <= NB_LEARN_SMEM_W;
    if (g->wide) return smem ? launch_cell_lean_t<true, true>(g, a, plan, block, color) : launch_cell_lean_t<true, false>(g, a, plan, block, color);
    return smem ? launch_cell_lean_t<false, true>(g, a, plan, block, color) : launch_cell_lean_t<false, false>(g, a, plan, block, color);
}

// Latency mode (persistent kernel) or throughput mode (lean launches per cell)?  The persistent
// grid has 2 x 256 threads per SM; beyond ~16 rows per thread and cell the cells are long enough
// (hundreds of microseconds) for launch overhead not to matter and for occupancy to decide.
// 2-byte graphs always learn in throughput mode: the persistent kernel is instantiated for 1-byte
// values only (it is the 128-register kernel whose instruction footprint DESIGN.md section 4 keeps small).
static int lean_mode(const nb_graph *g, int64_t cells, bool *lean)
{
    const char *e = getenv("NUMBSKULL_B200_LEARN_MODE");   // 1 persistent, 2 lean (tests compare the two)
    const int force = e ? atoi(e) : 0;
    if (g->value_bytes != 1) {
        if (force == 1)
            NB_FAIL(NB_ERR_UNSUPPORTED, "NUMBSKULL_B200_LEARN_MODE=1 (latency mode) is not available on graphs with "
                                        "cardinalities above 255: they learn in throughput mode only");
        *lean = true;
        return NB_OK;
    }
    if (force == 1 || force == 2) { *lean = force == 2; return NB_OK; }
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, g->device);
    *lean = g->V / std::max<int64_t>(cells, 1) > (int64_t)sms * 2 * NB_LEARN_THREADS * 2;
    return NB_OK;
}

// one (block, colour) cell: the partitioned runner exchanges halo values between the cells itself
template <class T>
static int learn_color_t(nb_graph *g, int color, int block, int n_blocks, double step, int regularization, double reg_param,
                         double truncation, int learn_non_evidence, uint64_t seed, uint64_t epoch)
{
    LearnArgs<T> a;
    std::vector<int64_t> vmax;
    NB_TRY(learn_prepare(g, a, vmax, learn_non_evidence));
    a.seed = seed; a.reg_param = reg_param; a.truncation = truncation; a.regularization = regularization;
    a.step = step; a.epoch = epoch;
    bool lean = true;
    NB_TRY(lean_mode(g, (int64_t)n_blocks * g->n_colors, &lean));
    if (lean) {
        NB_CUDA(cudaMemsetAsync(a.g_grad, 0, (size_t)g->W * sizeof(nb_fix_t), g->stream));
        NB_CUDA(cudaMemsetAsync(a.g_cnt, 0, (size_t)g->W * sizeof(uint32_t), g->stream));
        NB_TRY(launch_cell_lean(g, a, make_plan(g, n_blocks), block, color));
    } else if constexpr (sizeof(T) == 1) {
        NB_TRY(launch_cells(g, a, make_plan(g, n_blocks), block, block + 1, color));
    }
    g->weights_version++;
    NB_CUDA(cudaGetLastError());
    return NB_OK;
}

int nb_learn_color(nb_graph *g, int color, int block, int n_blocks, double step, int regularization, double reg_param,
                   double truncation, int learn_non_evidence, uint64_t seed, uint64_t epoch)
{
    if (color < 0 || color >= g->n_colors) return NB_OK;   // a colour this rank does not own
    if (n_blocks < 1 || block < 0 || block >= n_blocks) NB_FAIL(NB_ERR_INVALID, "block %d of %d", block, n_blocks);
    if (g->value_bytes == 1)
        return learn_color_t<nb_val_t>(g, color, block, n_blocks, step, regularization, reg_param, truncation,
                                       learn_non_evidence, seed, epoch);
    return learn_color_t<nb_val16_t>(g, color, block, n_blocks, step, regularization, reg_param, truncation,
                                     learn_non_evidence, seed, epoch);
}

// Parity hook: the ORIGINAL ids of the variables that cell (block, colour) of an epoch cut into
// n_blocks blocks holds, class by class in new-id order (the plan nb_learn_color walks).
int nb_learn_cell_id_list(nb_graph *g, int color, int block, int n_blocks, int64_t *ids, int64_t *n)
{
    if (n_blocks < 1 || block < 0 || block >= n_blocks) NB_FAIL(NB_ERR_INVALID, "block %d of %d", block, n_blocks);
    *n = 0;
    if (color < 0 || color >= g->n_colors) return NB_OK;
    CellPlan hp = make_plan(g, n_blocks);
    hp.win_start = g->win_start.data();            // host copy of the window table
    std::vector<int32_t> n2o;
    for (int cls = 0; cls < NB_N_CLASSES; cls++) {
        int beg = 0, end = 0;
        nb_plan_range(hp, cls, color, block, beg, end);
        if (end <= beg) continue;
        n2o.resize((size_t)(end - beg));
        NB_CUDA(cudaMemcpy(n2o.data(), g->d_new2old + beg, n2o.size() * 4, cudaMemcpyDeviceToHost));
        for (int32_t v : n2o)
            if (v >= 0) ids[(*n)++] = v;
    }
    return NB_OK;
}

template <class T>
static int run_learn_t(nb_graph *g, int64_t n_epochs, double *stepsize, double decay, int regularization, double reg_param,
                       double truncation, int learn_non_evidence, uint64_t seed, int64_t batch_visits)
{
    LearnArgs<T> a;
    std::vector<int64_t> vmax;
    NB_TRY(learn_prepare(g, a, vmax, learn_non_evidence));
    a.seed = seed; a.reg_param = reg_param; a.truncation = truncation; a.regularization = regularization;
    double step = *stepsize;
    for (int64_t ep = 0; ep < n_epochs; ep++) {
        a.step = step;
        a.epoch = g->epoch_counter++;
        const int nb = block_count(g, vmax, default_batch_visits(step, batch_visits));
        const int64_t cells = (int64_t)nb * g->n_colors;
        bool lean = true;
        NB_TRY(lean_mode(g, cells, &lean));
        if (lean) {
            // throughput mode: a few lean launches per cell (table 0 starts clear, k_cell_apply clears it again)
            NB_CUDA(cudaMemsetAsync(a.g_grad, 0, (size_t)g->W * sizeof(nb_fix_t), g->stream));
            NB_CUDA(cudaMemsetAsync(a.g_cnt, 0, (size_t)g->W * sizeof(uint32_t), g->stream));
            const CellPlan plan = make_plan(g, nb);
            for (int b = 0; b < nb; b++)
                for (int c = 0; c < g->n_colors; c++) NB_TRY(launch_cell_lean(g, a, plan, b, c));
        } else if constexpr (sizeof(T) == 1) {
            // latency mode: one persistent launch per epoch (cell indices are 32-bit: split absurdly long epochs)
            for (int64_t c0 = 0; c0 < cells; c0 += (1 << 30)) {
                const int64_t c1 = std::min<int64_t>(cells, c0 + (1 << 30));
                NB_TRY(launch_cells(g, a, make_plan(g, nb), (int)c0, (int)c1, -1));
            }
        }
        g->weights_version++;
        NB_CUDA(cudaGetLastError());
        step *= decay;   // factorgraph.py:206
    }
    *stepsize = step;
    return NB_OK;
}

int nb_run_learn(nb_graph *g, int64_t n_epochs, double *stepsize, double decay, int regularization, double reg_param,
                 double truncation, int learn_non_evidence, uint64_t seed, int64_t batch_visits)
{
    if (n_epochs <= 0) return NB_OK;
    if (g->value_bytes == 1)
        return run_learn_t<nb_val_t>(g, n_epochs, stepsize, decay, regularization, reg_param, truncation, learn_non_evidence,
                                     seed, batch_visits);
    return run_learn_t<nb_val16_t>(g, n_epochs, stepsize, decay, regularization, reg_param, truncation, learn_non_evidence,
                                   seed, batch_visits);
}
