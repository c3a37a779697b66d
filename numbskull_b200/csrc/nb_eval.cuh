// Device-side incidence-stream reader, factor evaluation and sampling helpers.
#pragma once
#include "nb_common.cuh"

// ---------------------------------------------------------------------------
// Philox4x32-10 (Salmon, Moraes, Dror, Shaw: "Parallel random numbers: as easy
// as 1, 2, 3", SC'11).  Counter = (variable global id, epoch, stream tag, 0),
// key = 64-bit seed: every (variable, sweep, purpose) has its own stream, so
// results do not depend on the launch geometry, the colouring or the partition.
// ---------------------------------------------------------------------------
__host__ __device__ inline void nb_philox_round(uint32_t *c, const uint32_t *k)
{
    const uint64_t p0 = (uint64_t)0xD2511F53u * c[0];
    const uint64_t p1 = (uint64_t)0xCD9E8D57u * c[2];
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k[0];
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k[1];
    c[1] = (uint32_t)p1;
    c[3] = (uint32_t)p0;
    c[0] = n0;
    c[2] = n2;
}

__host__ __device__ inline void nb_philox4x32(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                              uint64_t seed, uint32_t out[4])
{
    uint32_t c[4] = {c0, c1, c2, c3};
    uint32_t k[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
#pragma unroll
    for (int r = 0; r < 10; r++) {
        nb_philox_round(c, k);
        k[0] += 0x9E3779B9u;
        k[1] += 0xBB67AE85u;
    }
    out[0] = c[0]; out[1] = c[1]; out[2] = c[2]; out[3] = c[3];
}

// 53-bit uniform in [0, 1) from two 32-bit words
__host__ __device__ inline double nb_u53(uint32_t hi, uint32_t lo)
{
    return (double)((((uint64_t)hi << 32) | lo) >> 11) * (1.0 / 9007199254740992.0);
}

// stream tags (third counter word): purpose << 24 | block
#define NB_TAG_FREE 0u
#define NB_TAG_EVID 1u
#define NB_TAG_TRUNC 2u

// Uniform stream of one (variable, epoch, purpose): two doubles per Philox call.
struct NbUniforms {
    uint32_t id, epoch_lo, epoch_hi_tag;
    uint64_t seed;
    uint32_t block;
    uint32_t r[4];
    int left;   // unread 32-bit words of the current Philox block
    __device__ NbUniforms(uint32_t id_, uint64_t epoch, uint32_t tag, uint64_t seed_)
        : id(id_), epoch_lo((uint32_t)epoch), epoch_hi_tag((uint32_t)((epoch >> 32) & 0xFFFFu) | (tag << 24)),
          seed(seed_), block(0), left(0) {}
    __device__ __forceinline__ uint32_t word()
    {
        if (left == 0) { nb_philox4x32(id, epoch_lo, epoch_hi_tag, block++, seed, r); left = 4; }
        left--;
        return left == 3 ? r[0] : (left == 2 ? r[1] : (left == 1 ? r[2] : r[3]));
    }
    // 53-bit uniform (two words): the single draw of small-cardinality variables
    __device__ double next() { uint32_t hi = word(); return nb_u53(hi, word()); }
    // 32-bit uniform (one word): the per-value decisions of the streaming categorical sampler
    __device__ double next32() { return ((double)word() + 0.5) * (1.0 / 4294967296.0); }
};

// ---------------------------------------------------------------------------
// Row cursor: word i of a row lives at p[i * stride] (stride 32 for the SELL-32
// thread-path stream, 1 for contiguous warp-path rows).
// ---------------------------------------------------------------------------
struct NbRow {
    const uint32_t *p;
    int quad;  // 1: SELL-32 quad layout (word i at p[(i / 4) * 128 + i % 4]); 0: contiguous row
    __device__ __forceinline__ uint32_t w(int i) const
    {
        return quad ? __ldg(p + (((size_t)(i >> 2)) << 7) + (i & 3)) : __ldg(p + i);
    }
};

// row of thread-path variable nid (new id) / of warp row wr
__device__ __forceinline__ NbRow nb_thread_row(const uint32_t *twords, const int64_t *slice_ptr, int64_t nid)
{
    return NbRow{twords + ((slice_ptr[nid >> 5] + (nid & 31)) << 2), 1};
}
// address of word i of thread-path row nid (the SELL-32 layout NbRow::w reads), for in-place patches
__device__ __forceinline__ uint32_t *nb_thread_row_word(uint32_t *twords, const int64_t *slice_ptr, int64_t nid, int i)
{
    return twords + ((slice_ptr[nid >> 5] + (nid & 31)) << 2) + (((size_t)(i >> 2)) << 7) + (i & 3);
}
__device__ __forceinline__ NbRow nb_warp_row(const uint32_t *wwords, const int64_t *wrow_ptr, int64_t wr)
{
    return NbRow{wwords + wrow_ptr[wr], 0};
}

template <bool WIDE>
__device__ __forceinline__ NbHdr nb_read_hdr(const NbRow &r, int pos)
{
    NbHdr h;
    if (WIDE) {
        uint32_t a = r.w(pos), b = r.w(pos + 1);
        h.wid = a;
        h.code = (int)(b >> 27);
        h.feat = (int)((b >> 26) & 1u);
        h.fixed = (int)((b >> 25) & 1u);
        h.arity = (int)(b & 0xFFFFFFu);
    } else {
        uint32_t a = r.w(pos);
        h.code = (int)(a >> 27);
        if (h.code == C_MARK) {
            h.wid = a & 0x7FFFFFFu;
            h.feat = h.fixed = h.arity = 0;
        } else {
            h.feat = (int)((a >> 26) & 1u);
            h.fixed = (int)((a >> 25) & 1u);
            h.arity = (int)((a >> 20) & 31u);
            h.wid = a & 0xFFFFFu;
        }
    }
    return h;
}

template <bool WIDE>
__device__ __forceinline__ int nb_hdr_words() { return WIDE ? 2 : 1; }

// words of the incidence that starts with header h (header included); MARK = header only
template <bool WIDE>
__device__ __forceinline__ int nb_inc_words(const NbHdr &h)
{
    if (h.code == C_MARK) return nb_hdr_words<WIDE>();
    return nb_incidence_words(WIDE, h.code, h.arity, h.feat);
}

// featureValue of the incidence whose header is at `pos` (stored after members and extra)
template <bool WIDE>
__device__ __forceinline__ double nb_read_feature(const NbRow &r, const NbHdr &h, int pos)
{
    int fpos = pos + (WIDE ? 2 : 1) + h.arity * (nb_code_has_eq(h.code) ? 2 : 1) + (nb_code_has_extra(h.code) ? 1 : 0);
    uint32_t lo = r.w(fpos), hi = r.w(fpos + 1);
    return __hiloint2double((int)hi, (int)lo);
}

// ---------------------------------------------------------------------------
// eval_factor (inference.py:149-413) on one incidence.  `mpos` is the position
// of the first member word, `self` the new id of the sampled variable, `k` the
// value it is forced to; everything else is read from `vals`.  Loops run to the
// end instead of returning early so the member gathers are independent loads.
// ---------------------------------------------------------------------------
// Where member values come from.  The sweeps read the chain's value array; the table builders
// (nb_build.cu) force the values of the (at most two) other members of an incidence, so that the
// truth tables of the record streams are tabulated by THIS evaluator and nothing else.
//
// The accessors are templates on the element type of the value array (nb_val_t or nb_val16_t) and
// also answer the cardinality of a variable (NbCardOf): on 1-byte graphs that is the card field of
// its vmeta word and the accessor is a bare pointer, as before; on 2-byte graphs a card field of 0
// sends the lookup to nb_graph::d_vcard.  SweepArgs / LearnArgs derive from it too: on 1-byte
// graphs it is an empty base, so their layout (and the kernels' code) is what it was before.
template <class T>
struct NbCardOf {
    __host__ __device__ __forceinline__ NbCardOf(const uint16_t * = nullptr) {}
    __device__ __forceinline__ int card(uint32_t meta, uint32_t) const { return NB_META_CARD(meta); }
};
template <>
struct NbCardOf<nb_val16_t> {
    const uint16_t *vcard;
    __host__ __device__ __forceinline__ NbCardOf(const uint16_t *c = nullptr) : vcard(c) {}
    __device__ __forceinline__ int card(uint32_t meta, uint32_t id) const
    {
        const int c = NB_META_CARD(meta);
        return c ? c : (int)__ldg(vcard + id);
    }
};

template <class T>
struct NbValsGlobal : NbCardOf<T> {
    const T *__restrict__ v;
    __device__ __forceinline__ NbValsGlobal(const T *v_, const NbCardOf<T> &cards = NbCardOf<T>()) : NbCardOf<T>(cards), v(v_) {}
    __device__ __forceinline__ int operator()(uint32_t vid) const { return (int)v[vid]; }
};
// Same for the persistent learning kernel, which reads values other CTAs wrote earlier in the same
// launch: a plain cached load (ld.global.ca, never the non-coherent path).  Inside a cell nobody
// writes what another thread reads (colouring), and between cells every CTA passes the grid
// barrier, whose fence invalidates the SM's L1 (CCTL.IVALL) before anybody reads again.  Bypassing
// L1 altogether (ld.global.cg) cost the categorical rows a factor of four: their samplers re-read
// the same few neighbours for every candidate value.
template <class T>
struct NbValsCG : NbCardOf<T> {
    const T *v;
    __device__ __forceinline__ NbValsCG(const T *v_, const NbCardOf<T> &cards = NbCardOf<T>()) : NbCardOf<T>(cards), v(v_) {}
    __device__ __forceinline__ int operator()(uint32_t vid) const { return (int)__ldca(v + vid); }
};
// weight accessors: global (read-only for the launch), global through L2, or a shared-memory copy
struct NbWtsGlobal {
    const double *__restrict__ w;
    __device__ __forceinline__ double operator()(uint32_t i) const { return __ldg(w + i); }
};
struct NbWtsCG {
    const double *w;
    __device__ __forceinline__ double operator()(uint32_t i) const { return __ldca(w + i); }
};
struct NbWtsShared {
    const double *w;
    __device__ __forceinline__ double operator()(uint32_t i) const { return w[i]; }
};
struct NbValsForced {
    uint32_t ida, idb;
    int xa, xb;
    __device__ __forceinline__ int operator()(uint32_t vid) const { return vid == ida ? xa : (vid == idb ? xb : 0); }
};

template <class Vals>
__device__ __forceinline__ int nb_member(const NbRow &r, int mpos, int step, int j, uint32_t self,
                                         int k, const Vals &vals)
{
    uint32_t vid = r.w(mpos + j * step);
    return vid == self ? k : vals(vid);
}

// NOT inlined: the 26-way switch is called from a dozen places in the generic samplers and the
// learning kernel; inlined everywhere it blew the persistent learning kernel up to 855 KB of SASS
// (k_gibbs_thread: 195 KB), and every mini-batch cell then ran out of a cold instruction cache
// (ncu: 81 % i-cache hit rate, the slowest CTA 6x slower than the average one).
#ifndef NB_EVAL_INLINE
#define NB_EVAL_FN __noinline__
#else
#define NB_EVAL_FN inline
#endif
template <class Vals>
__device__ NB_EVAL_FN double nb_eval_incidence_v(const NbRow &r, const NbHdr &h, int mpos, uint32_t self,
                                                   int k, const Vals &vals)
{
    const int a = h.arity;
    const int step = nb_code_has_eq(h.code) ? 2 : 1;
    switch (h.code) {
    case C_NOOP:
        return 0.0;
    case C_IMPLY_NATURAL: {  // inference.py:162-176 (the -1 branch is unreachable)
        bool all = true;
        for (int j = 0; j < a; j++) all &= nb_member(r, mpos, 1, j, self, k, vals) != 0;
        return all ? 1.0 : 0.0;
    }
    case C_OR: {  // :177-183
        bool any = false;
        for (int j = 0; j < a; j++) any |= nb_member(r, mpos, 1, j, self, k, vals) == 1;
        return any ? 1.0 : -1.0;
    }
    case C_AND:
    case C_ISTRUE: {  // :193-200
        bool all = true;
        for (int j = 0; j < a; j++) all &= nb_member(r, mpos, 1, j, self, k, vals) != 0;
        return all ? 1.0 : -1.0;
    }
    case C_EQUAL: {  // :184-192
        if (a == 0) return 1.0;
        int first = nb_member(r, mpos, 1, 0, self, k, vals);
        bool eq = true;
        for (int j = 1; j < a; j++) eq &= nb_member(r, mpos, 1, j, self, k, vals) == first;
        return eq ? 1.0 : -1.0;
    }
    case C_LINEAR:
    case C_RATIO:
    case C_LOGICAL: {  // :201-231
        if (a == 0) return h.code == C_RATIO ? 0.0 : 0.0;
        int head = nb_member(r, mpos, 1, a - 1, self, k, vals);
        int cnt = 0;
        for (int j = 0; j < a - 1; j++) cnt += nb_member(r, mpos, 1, j, self, k, vals) == head;
        if (h.code == C_LINEAR) return (double)cnt;
        if (h.code == C_RATIO) return log((double)(1 + cnt));
        return cnt > 0 ? 1.0 : 0.0;
    }
    case C_IMPLY_MLN:
    case C_IMPLY_NATURAL_CAT:
    case C_IMPLY_MLN_CAT: {  // :232-246, :266-295 -- head read through the aliased slot, as coded
        if (a == 0) return 0.0;
        bool body = true;
        for (int j = 0; j < a - 1; j++) {
            int x = nb_member(r, mpos, step, j, self, k, vals);
            if (h.code == C_IMPLY_MLN) body &= x != 0;
            else body &= x == (int)r.w(mpos + j * step + 1);
        }
        uint32_t last = r.w(mpos + (a - 1) * step);
        uint32_t alias = r.w(mpos + a * step);
        int head = last == self ? k : (alias == 0xFFFFFFFFu ? 0 : vals(alias));
        if (h.code == C_IMPLY_MLN) return !body ? 1.0 : (head ? 1.0 : 0.0);
        bool hit = head == (int)r.w(mpos + (a - 1) * step + 1);
        if (h.code == C_IMPLY_NATURAL_CAT) return !body ? 0.0 : (hit ? 1.0 : -1.0);
        return !body ? 1.0 : (hit ? 1.0 : 0.0);
    }
    case C_AND_CAT:
    case C_EQUAL_CAT_CONST: {  // :251-258
        bool all = true;
        for (int j = 0; j < a; j++)
            all &= nb_member(r, mpos, 2, j, self, k, vals) == (int)r.w(mpos + 2 * j + 1);
        return all ? 1.0 : 0.0;
    }
    case C_OR_CAT: {  // :259-265
        bool any = false;
        for (int j = 0; j < a; j++)
            any |= nb_member(r, mpos, 2, j, self, k, vals) == (int)r.w(mpos + 2 * j + 1);
        return any ? 1.0 : -1.0;
    }
    case C_DP_CLASS_PRIOR:  // :301-305
        return nb_member(r, mpos, 1, 0, self, k, vals) == 1 ? 1.0 : -1.0;
    case C_DP_LF_PRIOR: {  // :306-315
        int l = nb_member(r, mpos, 1, 0, self, k, vals);
        return l == 2 ? -1.0 : (l == 0 ? 0.0 : 1.0);
    }
    case C_DP_LF_PROPENSITY: {  // :316-320
        int abstain = (int)r.w(mpos + a);
        return nb_member(r, mpos, 1, 0, self, k, vals) == abstain ? 0.0 : 1.0;
    }
    case C_DP_LF_ACCURACY:
    case C_DP_LF_CLASS_PROPENSITY: {  // :321-347
        int y = nb_member(r, mpos, 1, 0, self, k, vals);
        int l = nb_member(r, mpos, 1, 1, self, k, vals);
        int abstain = (int)r.w(mpos + a);
        if (l == abstain) return 0.0;
        if (h.code == C_DP_LF_ACCURACY) return y == l ? 1.0 : -1.0;
        return y == 1 ? 1.0 : -1.0;
    }
    case C_DP_DEP_FIXING:
    case C_DP_DEP_REINFORCING: {  // :348-381
        int y = nb_member(r, mpos, 1, 0, self, k, vals);
        int l1 = nb_member(r, mpos, 1, 1, self, k, vals);
        int l2 = nb_member(r, mpos, 1, 2, self, k, vals);
        int abstain = (int)r.w(mpos + a);
        if (l1 == abstain) return l2 != 1 ? -1.0 : 0.0;
        if (h.code == C_DP_DEP_FIXING)
            return ((l1 == 0 && l2 == 1 && y == 1) || (l1 == 1 && l2 == 0 && y == 0)) ? 1.0 : 0.0;
        return ((l1 == 0 && l2 == 0 && y == 0) || (l1 == 1 && l2 == 1 && y == 1)) ? 1.0 : 0.0;
    }
    case C_DP_DEP_EXCLUSIVE: {  // :382-388
        int l1 = nb_member(r, mpos, 1, 0, self, k, vals);
        int l2 = nb_member(r, mpos, 1, 1, self, k, vals);
        int abstain = (int)r.w(mpos + a);
        return (l1 == abstain || l2 == abstain) ? 0.0 : -1.0;
    }
    case C_DP_DEP_SIMILAR:  // :389-394
        return nb_member(r, mpos, 1, 0, self, k, vals) == nb_member(r, mpos, 1, 1, self, k, vals) ? 1.0 : 0.0;
    case C_UFO: {  // :399-405; a selector beyond the factor's own members yields 0
        int v0 = nb_member(r, mpos, 1, 0, self, k, vals);
        if (v0 == 0 || v0 - 1 >= a) return 0.0;
        return (double)nb_member(r, mpos, 1, v0 - 1, self, k, vals);
    }
    default:
        return 0.0;
    }
}

template <class T>
__device__ __forceinline__ double nb_eval_incidence(const NbRow &r, const NbHdr &h, int mpos, uint32_t self,
                                                    int k, const T *__restrict__ vals)
{
    return nb_eval_incidence_v(r, h, mpos, self, k, NbValsGlobal<T>(vals));
}

// position of the first member word of the incidence whose header is at `pos`
template <bool WIDE>
__device__ __forceinline__ int nb_member_pos(const NbHdr &h, int pos)
{
    return pos + nb_hdr_words<WIDE>();
}

// p += w * f without FMA contraction: bit-identical to the reference's
// double-precision `p += weight * eval_factor(...)` when summed in bucket order.
__device__ __forceinline__ double nb_acc(double p, double w, double f) { return __dadd_rn(p, __dmul_rn(w, f)); }

// ---------------------------------------------------------------------------
// Streaming categorical sampler: P(pick = k) = exp(e_k) / sum_j exp(e_j) in
// one pass (weighted reservoir with a running maximum for stability).
// ---------------------------------------------------------------------------
struct NbReservoir {
    double m, s;
    int pick;
    bool empty;
    __device__ NbReservoir() : m(0.0), s(0.0), pick(0), empty(true) {}
    // add `mult` items of energy e; returns true when the pick moved to this group.  The
    // rescaling factors only shape sampling probabilities: fp32 exp (1e-7 relative) is ample.
    __device__ bool add(double e, double mult, double u)
    {
        if (empty) { m = e; s = mult; empty = false; return true; }
        double t;
        if (e > m) { s = s * (double)__expf((float)(m - e)) + mult; m = e; t = mult; }
        else { t = mult * (double)__expf((float)(e - m)); s += t; }
        return u * s < t;
    }
};

// ---------------------------------------------------------------------------
// energies of a dataType-0 row for k < card <= 4, all candidate values in one
// pass over the row (sum order = bucket order = the reference's)
// ---------------------------------------------------------------------------
template <bool WIDE, class Vals, class Wts>
__device__ __forceinline__ void nb_row_energies4_v(const NbRow &r, int len, uint32_t self, int card,
                                                   const Vals &vals, const Wts &weight, double e[4])
{
    int pos = 0;
    while (pos < len) {
        NbHdr h = nb_read_hdr<WIDE>(r, pos);
        int mpos = nb_member_pos<WIDE>(h, pos);
        double w = weight(h.wid);
#pragma unroll
        for (int k = 0; k < 4; k++)
            if (k < card) e[k] = nb_acc(e[k], w, nb_eval_incidence_v(r, h, mpos, self, k, vals));
        pos += nb_inc_words<WIDE>(h);
    }
}

// energy of value k of a dataType-0 row (any cardinality)
template <bool WIDE, class Vals, class Wts>
__device__ __forceinline__ double nb_row_energy_k_v(const NbRow &r, int len, uint32_t self, int k,
                                                    const Vals &vals, const Wts &weight)
{
    double e = 0.0;
    int pos = 0;
    while (pos < len) {
        NbHdr h = nb_read_hdr<WIDE>(r, pos);
        e = nb_acc(e, weight(h.wid), nb_eval_incidence_v(r, h, nb_member_pos<WIDE>(h, pos), self, k, vals));
        pos += nb_inc_words<WIDE>(h);
    }
    return e;
}

template <bool WIDE, class T>
__device__ __forceinline__ double nb_row_energy_k(const NbRow &r, int len, uint32_t self, int k,
                                                  const T *__restrict__ vals,
                                                  const double *__restrict__ weight)
{
    return nb_row_energy_k_v<WIDE>(r, len, self, k, NbValsGlobal<T>(vals), NbWtsGlobal{weight});
}

// j-th value (ascending) of a categorical row that has no bucket marker
template <bool WIDE>
__device__ inline int nb_nth_empty_value(const NbRow &r, int len, int j)
{
    int cur = 0, pos = 0;
    while (pos < len) {
        NbHdr h = nb_read_hdr<WIDE>(r, pos);
        if (h.code == C_MARK) {
            int gap = (int)h.wid - cur;
            if (j < gap) return cur + j;
            j -= gap;
            cur = (int)h.wid + 1;
        }
        pos += nb_inc_words<WIDE>(h);
    }
    return cur + j;
}

// inverse-CDF draw over k < card <= 4 energies (draw_sample, inference.py:36-52,
// with the maximum subtracted before exp -- mathematically identical)
__device__ __forceinline__ int nb_draw_small(const double e[4], int card, double u)
{
    if (card == 2) {
        double p0 = (double)(1.0f / (1.0f + __expf((float)(e[1] - e[0]))));
        return u <= p0 ? 0 : 1;
    }
    double m = e[0];
#pragma unroll
    for (int k = 1; k < 4; k++) if (k < card) m = fmax(m, e[k]);
    double z[4], tot = 0.0;
#pragma unroll
    for (int k = 0; k < 4; k++) { z[k] = k < card ? (double)__expf((float)(e[k] - m)) : 0.0; tot += z[k]; z[k] = tot; }
    double t = u * tot;
    int pick = card - 1;
#pragma unroll
    for (int k = 3; k >= 0; k--) if (k < card && z[k] >= t) pick = k;
    return pick;
}

// Sample one variable whose row is `r` (thread path, or any row walked by one thread).
template <bool WIDE, class Vals, class Wts>
__device__ NB_EVAL_FN int nb_sample_row_v(const NbRow &r, int len, uint32_t self, uint32_t meta,
                                            const Vals &vals, const Wts &weight, NbUniforms &rng)
{
    const int card = vals.card(meta, self);
    if (NB_META_DTYPE(meta) == 0) {
        if (card <= 4) {
            double e[4] = {0.0, 0.0, 0.0, 0.0};
            nb_row_energies4_v<WIDE>(r, len, self, card, vals, weight, e);
            return nb_draw_small(e, card, rng.next());
        }
        NbReservoir res;
        for (int k = 0; k < card; k++)
            if (res.add(nb_row_energy_k_v<WIDE>(r, len, self, k, vals, weight), 1.0, rng.next32())) res.pick = k;
        return res.pick;
    }
    // categorical: buckets in ascending value order, each introduced by a MARK
    NbReservoir res;
    int pos = 0, cur = -1, nonempty = 0;
    double e = 0.0;
    while (pos < len) {
        NbHdr h = nb_read_hdr<WIDE>(r, pos);
        if (h.code == C_MARK) {
            if (cur >= 0 && res.add(e, 1.0, rng.next32())) res.pick = cur;
            cur = (int)h.wid;
            e = 0.0;
            nonempty++;
        } else {
            e = nb_acc(e, weight(h.wid), nb_eval_incidence_v(r, h, nb_member_pos<WIDE>(h, pos), self, cur, vals));
        }
        pos += nb_inc_words<WIDE>(h);
    }
    if (cur >= 0 && res.add(e, 1.0, rng.next32())) res.pick = cur;
    int n_empty = card - nonempty;
    if (n_empty > 0 && res.add(0.0, (double)n_empty, rng.next32())) {
        int j = min(n_empty - 1, (int)(rng.next32() * (double)n_empty));
        res.pick = nb_nth_empty_value<WIDE>(r, len, j);
    }
    return res.pick;
}

template <bool WIDE, class T>
__device__ inline int nb_sample_row(const NbRow &r, int len, uint32_t self, uint32_t meta,
                                    const T *__restrict__ vals, const NbCardOf<T> &cards, const double *__restrict__ weight,
                                    NbUniforms &rng)
{
    return nb_sample_row_v<WIDE>(r, len, self, meta, NbValsGlobal<T>(vals, cards), NbWtsGlobal{weight}, rng);
}


__device__ __forceinline__ double nb_warp_sum(double x)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xFFFFFFFFu, x, o);
    return x;
}

// Sample a warp row whose cardinality is above 255 (2-byte graphs), one warp, every lane returns
// the same value.  Such a row's per-value energies do not fit the warp's shared array (and a task
// partial of card doubles per task would scale with n_tasks x card), so the row is sampled from its
// incidences directly and needs no memory beyond the row itself:
//   dataType 1: the incidences are in bucket order, i.e. ascending value order.  The lanes evaluate
//     32 consecutive incidences at a time; the energies are then folded in incidence order into one
//     sum per value (shuffles, identical on every lane), and each finished value enters the
//     reservoir, followed by the single group of empty buckets -- nb_sample_row_v's semantics.
//   dataType 0: every incidence contributes to every value: one warp reduction per value.
template <bool WIDE, class Vals, class Wts>
__device__ NB_EVAL_FN int nb_warp_sample_wide(const NbRow &r, int len, const uint2 *__restrict__ inc, int n_inc,
                                                uint32_t self, uint32_t meta, int card, const Vals &vals,
                                                const Wts &weight, NbUniforms &rng)
{
    const int lane = threadIdx.x & 31;
    NbReservoir res;
    if (NB_META_DTYPE(meta) == 0) {
        for (int k = 0; k < card; k++) {
            double e = 0.0;
            for (int i = lane; i < n_inc; i += 32) {
                const int pos = (int)inc[i].x;
                const NbHdr h = nb_read_hdr<WIDE>(r, pos);
                e += weight(h.wid) * nb_eval_incidence_v(r, h, nb_member_pos<WIDE>(h, pos), self, k, vals);
            }
            if (res.add(nb_warp_sum(e), 1.0, rng.next32())) res.pick = k;
        }
        return res.pick;
    }
    int cur = -1, nonempty = 0;
    double e = 0.0;
    for (int base = 0; base < n_inc; base += 32) {
        int k = -1;
        double x = 0.0;
        if (base + lane < n_inc) {
            const uint2 ent = inc[base + lane];
            const NbHdr h = nb_read_hdr<WIDE>(r, (int)ent.x);
            k = (int)ent.y;
            x = weight(h.wid) * nb_eval_incidence_v(r, h, nb_member_pos<WIDE>(h, (int)ent.x), self, k, vals);
        }
        const int m = min(32, n_inc - base);
        for (int j = 0; j < m; j++) {
            const int kj = __shfl_sync(0xFFFFFFFFu, k, j);
            const double xj = __shfl_sync(0xFFFFFFFFu, x, j);
            if (kj != cur) {
                if (cur >= 0 && res.add(e, 1.0, rng.next32())) res.pick = cur;
                cur = kj;
                e = 0.0;
                nonempty++;
            }
            e += xj;
        }
    }
    if (cur >= 0 && res.add(e, 1.0, rng.next32())) res.pick = cur;
    const int n_empty = card - nonempty;
    if (n_empty > 0 && res.add(0.0, (double)n_empty, rng.next32())) {
        const int j = min(n_empty - 1, (int)(rng.next32() * (double)n_empty));
        res.pick = nb_nth_empty_value<WIDE>(r, len, j);
    }
    return res.pick;
}


// ---------------------------------------------------------------------------
// Philox2x32-10 (same family, 64-bit counter, 32-bit key): one 53-bit uniform
// per call, used where a variable needs a single draw per sweep.
// ---------------------------------------------------------------------------
__host__ __device__ inline double nb_philox2x32_u53(uint32_t c0, uint32_t c1, uint32_t key)
{
#pragma unroll
    for (int r = 0; r < 10; r++) {
        const uint64_t p = (uint64_t)0xD256D193u * c0;
        c0 = (uint32_t)(p >> 32) ^ key ^ c1;
        c1 = (uint32_t)p;
        key += 0x9E3779B9u;
    }
    return nb_u53(c0, c1);
}

__host__ __device__ inline uint32_t nb_fold_key(uint64_t seed, uint64_t epoch, uint32_t tag)
{
    uint64_t x = seed ^ ((epoch >> 32) * 0x9E3779B97F4A7C15ull) ^ ((uint64_t)tag << 56);
    x ^= x >> 33; x *= 0xFF51AFD7ED558CCDull; x ^= x >> 33;
    return (uint32_t)x ^ (uint32_t)(x >> 32);
}

// ---------------------------------------------------------------------------
// Truth-table (TT) stream of the FAST row class.  A FAST row belongs to a
// Boolean variable whose incidences all have arity <= 3 and an integer-valued
// function; each incidence is ONE 16-byte quad
//     { other member A (new id), other member B (new id), table, weight (fp32 bits) }
// where table holds, for the 3 x 3 combinations of (min(xA, 2), min(xB, 2)),
// the 3-bit code of f(self = 1) - f(self = 0) + 2 at bit 3 * (3 * a + b); bit 27
// = weight is fixed / padding.  Unused member slots point at the variable itself, padding
// quads carry the all-zero-difference table, so every lane of a warp runs the
// same trip count with no parsing at all.  The weight VALUE is inlined (a random
// gather of weight[wid] per incidence costs a full 32-sector request per warp
// and was half of the L1/L2 traffic of the sweep on the KBC shape); the weight
// ids live in a parallel word per quad (tt_wid) that only the learning sweep and
// the refresh kernel (nb_sweep.cu k_tt_refresh) read.
// ---------------------------------------------------------------------------
// Streaming loads.  The record streams, slice pointers and per-variable words are read once per
// sweep; the value array is gathered at random and re-used.  ncu on the KBC shape showed the
// streams washing the values out of L2 (28 % L2 hit rate, 2.2x the necessary DRAM bytes), so
// everything that streams is loaded evict-first (ld.global.cs) and the values keep the cache.
template <class T>
__device__ __forceinline__ T nb_lds(const T *p) { return __ldcs(p); }

#define NB_TT_NEUTRAL 0x2492492u   /* 9 x code 2 (difference 0) */
#define NB_TT_FIXED_BIT (1u << 27) /* weight is fixed (also set on padding quads): no gradient */
// A parallel word per quad (used by the learning sweep only) holds f(self = 0) + 1 in 2 bits per
// combination, so that f(k) = f(0) + k * (f(1) - f(0)) is available for both chains.
#define NB_TT_BASE_NEUTRAL 0x15555u /* 9 x code 1 (value 0) */

__host__ __device__ inline bool nb_code_tt_const_compare(int c)
{
    return c == C_NOOP || c == C_IMPLY_NATURAL || c == C_OR || c == C_AND || c == C_ISTRUE;
}
__host__ __device__ inline bool nb_code_tt_ok(int c)
{
    return nb_code_tt_const_compare(c) || c == C_EQUAL || c == C_LINEAR || c == C_LOGICAL ||
           (c >= C_DP_CLASS_PRIOR && c <= C_DP_DEP_SIMILAR);
}

__device__ __forceinline__ int nb_tt_index(int xa, int xb) { return min(xa, 2) * 3 + min(xb, 2); }
__device__ __forceinline__ int nb_tt_diff(uint32_t table, int idx) { return (int)((table >> (3 * idx)) & 7u) - 2; }

// Tabulate the incidence whose header sits at `pos` of the generic row `r` of variable `self`
// (dataType 0, cardinality 2, arity <= 3) with nb_eval_incidence_v -- the one evaluator.  The
// (at most two) members other than `self` are returned in other[] (unused slots = self).
template <bool WIDE>
__device__ inline NbHdr nb_tabulate(const NbRow &r, int pos, uint32_t self, uint32_t other[2], uint32_t &table,
                                    uint32_t &base)
{
    const NbHdr h = nb_read_hdr<WIDE>(r, pos);
    const int mpos = pos + nb_hdr_words<WIDE>();
    int n_other = 0;
    other[0] = other[1] = self;
    for (int j = 0; j < h.arity && j < 3; j++) {
        const uint32_t u = r.w(mpos + j);
        if (u != self && n_other < 2) other[n_other++] = u;
    }
    table = 0u;
    base = 0u;
    for (int xa = 0; xa < 3; xa++)
        for (int xb = 0; xb < 3; xb++) {
            const NbValsForced vals{other[0], other[1], xa, xb};
            const int f0 = (int)nb_eval_incidence_v(r, h, mpos, self, 0, vals);
            const int f1 = (int)nb_eval_incidence_v(r, h, mpos, self, 1, vals);
            table |= (uint32_t)(f1 - f0 + 2) << (3 * (3 * xa + xb));
            base |= (uint32_t)(f0 + 1) << (2 * (3 * xa + xb));
        }
    return h;
}

// e1 - e0 of a FAST row from its quads (lane-strided SELL layout: quad j at qp[j * 32]).
#define NB_TT_UNROLL_DEFAULT 4
// where the record kernels read member values from: the byte array, or (large all-Boolean graphs,
// see nb_graph::d_valbits) a bit-packed mirror of it that stays L2-resident
template <class T>
struct NbValsBytes {
    const T *__restrict__ v;
    __device__ __forceinline__ int operator()(uint32_t id) const { return (int)v[id]; }
};
struct NbValsBits {
    const uint32_t *__restrict__ b;
    __device__ __forceinline__ int operator()(uint32_t id) const { return (int)((b[id >> 5] >> (id & 31u)) & 1u); }
};

template <int NB_TT_UNROLL = NB_TT_UNROLL_DEFAULT, class Vals>
__device__ __forceinline__ double nb_tt_delta_v(const uint4 *__restrict__ qp, int n, uint32_t self, const Vals vals)
{
    double d = 0.0;
    for (int j = 0; j < n; j += NB_TT_UNROLL) {
        uint4 q[NB_TT_UNROLL];
#pragma unroll
        for (int t = 0; t < NB_TT_UNROLL; t++)
            q[t] = (j + t < n) ? nb_lds(qp + (size_t)(j + t) * 32) : make_uint4(self, self, NB_TT_NEUTRAL, 0u);
        int xa[NB_TT_UNROLL], xb[NB_TT_UNROLL];
#pragma unroll
        for (int t = 0; t < NB_TT_UNROLL; t++) {
            xa[t] = vals(q[t].x);
            xb[t] = vals(q[t].y);
        }
#pragma unroll
        for (int t = 0; t < NB_TT_UNROLL; t++)
            d = fma((double)__uint_as_float(q[t].w), (double)nb_tt_diff(q[t].z, nb_tt_index(xa[t], xb[t])), d);
    }
    return d;
}
template <int NB_TT_UNROLL = NB_TT_UNROLL_DEFAULT, class T>
__device__ __forceinline__ double nb_tt_delta(const uint4 *__restrict__ qp, int n, uint32_t self,
                                              const T *__restrict__ vals)
{
    return nb_tt_delta_v<NB_TT_UNROLL>(qp, n, self, NbValsBytes<T>{vals});
}

// Pair records (NB_CLASS_PAIR): incidences with at most ONE other member take 8 bytes,
//     { other member (new id, or the variable itself), table:9 | fixed:1 | wid:22 }
// table = 3-bit code of f(1) - f(0) + 2 for min(x_other, 2) in {0, 1, 2}; two records per quad.
// UNIFORM slices: when every record of the 32 rows of a slice carries the same second word
// (every tied-weight MRF: the Ising grid has ONE (table, weight) pair), the word is hoisted into
// tt2_common[slice] and the slice stores bare 4-byte member ids, four per quad
// (NB_PAIR_NONE = no record).
#define NB_PAIR_NEUTRAL 0x92u          /* 3 x code 2 */
#define NB_PAIR_FIXED_BIT (1u << 9)
#define NB_PAIR_NONE 0xFFFFFFFFu       /* tt2_common: slice is not uniform; member id: empty record */
#define NB_PAIR_ANY 0xFFFFFFFEu        /* build only: a row without records fits any common word */
__host__ __device__ inline uint32_t nb_pack_pair(uint32_t table9, int fixed, uint32_t wid)
{
    return table9 | ((uint32_t)fixed << 9) | (wid << 10);
}

#define NB_TT2_UNROLL 2
template <class Vals>
__device__ __forceinline__ double nb_tt2_delta_v(const uint4 *__restrict__ qp, int n, uint32_t common, uint32_t self,
                                                 const Vals vals, const double *__restrict__ weight)
{
    if (common != NB_PAIR_NONE) {
        const double w = __ldg(weight + (common >> 10));
        int acc = 0;
        for (int j = 0; j < n; j++) {
            const uint4 q = nb_lds(qp + (size_t)j * 32);
            const uint32_t o[4] = {q.x, q.y, q.z, q.w};
            int x[4];
#pragma unroll
            for (int t = 0; t < 4; t++) x[t] = vals(o[t] == NB_PAIR_NONE ? self : o[t]);
#pragma unroll
            for (int t = 0; t < 4; t++)
                acc += o[t] == NB_PAIR_NONE ? 0 : (int)((common >> (3 * min(x[t], 2))) & 7u) - 2;
        }
        return w * (double)acc;
    }
    const uint32_t neutral = nb_pack_pair(NB_PAIR_NEUTRAL, 1, 0u);
    double d = 0.0;
    for (int j = 0; j < n; j += NB_TT2_UNROLL) {
        uint4 q[NB_TT2_UNROLL];
#pragma unroll
        for (int t = 0; t < NB_TT2_UNROLL; t++)
            q[t] = (j + t < n) ? nb_lds(qp + (size_t)(j + t) * 32) : make_uint4(self, neutral, self, neutral);
        int x0[NB_TT2_UNROLL], x1[NB_TT2_UNROLL];
        double w0[NB_TT2_UNROLL], w1[NB_TT2_UNROLL];
#pragma unroll
        for (int t = 0; t < NB_TT2_UNROLL; t++) {
            x0[t] = vals(q[t].x);
            x1[t] = vals(q[t].z);
            w0[t] = __ldg(weight + (q[t].y >> 10));
            w1[t] = __ldg(weight + (q[t].w >> 10));
        }
#pragma unroll
        for (int t = 0; t < NB_TT2_UNROLL; t++) {
            d = fma(w0[t], (double)((int)((q[t].y >> (3 * min(x0[t], 2))) & 7u) - 2), d);
            d = fma(w1[t], (double)((int)((q[t].w >> (3 * min(x1[t], 2))) & 7u) - 2), d);
        }
    }
    return d;
}
template <class T>
__device__ __forceinline__ double nb_tt2_delta(const uint4 *__restrict__ qp, int n, uint32_t common, uint32_t self,
                                               const T *__restrict__ vals, const double *__restrict__ weight)
{
    return nb_tt2_delta_v(qp, n, common, self, NbValsBytes<T>{vals}, weight);
}

// Categorical records (NB_CLASS_CAT): one quad per incidence of an AND_CAT / EQUAL_CAT_CONST factor
// (inference.py:251-258) seen from a categorical variable in its bucket k:
//     { other A, other B, k:8 | eqA:8 | eqB:8 | n_others:2 | fixed:1, weight (fp32 bits) }
// (like the FAST quads the record inlines the weight VALUE; the ids live in cat_wid for the refresh)
// The factor is 1 iff every other member equals its dense_equal_to (the variable itself matches by
// construction of the bucket); n_others == 3 marks "never satisfied" (padding, or the variable
// occurring twice with different values).  eqA / eqB have 8 bits: on a 2-byte graph a row is a CAT
// row only if every dense_equal_to it stores is <= 255 (k_row_size); its other members may be wide.
__host__ __device__ inline uint32_t nb_pack_cat(int k, int eq_a, int eq_b, int n_others, int fixed)
{
    return (uint32_t)k | ((uint32_t)eq_a << 8) | ((uint32_t)eq_b << 16) | ((uint32_t)n_others << 24) | ((uint32_t)fixed << 26);
}

// Per-value energies of a CAT row: acc.add(k, w) for every satisfied incidence of bucket k.
template <class Acc, class T>
__device__ __forceinline__ void nb_cat_energies(const uint4 *__restrict__ qp, int n, uint32_t self,
                                                const T *__restrict__ vals, Acc &acc)
{
    for (int j = 0; j < n; j += 2) {
        uint4 q[2];
#pragma unroll
        for (int t = 0; t < 2; t++)
            q[t] = (j + t < n) ? nb_lds(qp + (size_t)(j + t) * 32) : make_uint4(self, self, nb_pack_cat(0, 0, 0, 3, 1), 0u);
        int xa[2], xb[2];
        float w[2];
#pragma unroll
        for (int t = 0; t < 2; t++) {
            xa[t] = (int)vals[q[t].x];
            xb[t] = (int)vals[q[t].y];
            w[t] = __uint_as_float(q[t].w);
        }
#pragma unroll
        for (int t = 0; t < 2; t++) {
            const uint32_t m = q[t].z;
            const int no = (int)((m >> 24) & 3u);
            const bool sat = no < 3 && (no < 1 || xa[t] == (int)((m >> 8) & 0xFFu)) && (no < 2 || xb[t] == (int)((m >> 16) & 0xFFu));
            if (sat) acc.add((int)(m & 0xFFu), w[t]);
        }
    }
}
