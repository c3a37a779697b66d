/*
 * nb_oracle.c -- CPU ORACLE for the numbskull Gibbs / weight-learning hot path.
 *
 * THIS IS TEST INFRASTRUCTURE, NOT PRODUCT CODE.  Only tests/, the smoke check
 * in __graft_entry__.py and the cpu_baseline / --impl reference legs of
 * bench.py may load it.  The product path (numbskull_b200/) never links,
 * imports or calls anything in this directory.
 *
 * It is a plain-C restatement of the reference's numba algorithm, operating on
 * the reference's own packed record arrays (numbskull/numbskulltypes.py:11-39)
 * so the same numpy buffers can be handed to the reference, to this oracle and
 * to the CUDA library.  Each function cites the reference lines it follows
 * (paths relative to the reference checkout).
 *
 * Parity pin: the random stream is MT19937 seeded by Knuth's LCG and turned
 * into 53-bit doubles exactly the way numba's runtime does it, with separate
 * "np" and "py" generators (np.random.rand in draw_sample, random.random in
 * sample_and_sgd).  With nthreads == 1 and the same seed this oracle therefore
 * reproduces the reference's count / var_value / weight_value arrays
 * bit-for-bit; tests/golden/ holds arrays produced by the real numba code
 * (tests/golden/make_golden.py) and tests/test_oracle_golden.py checks them.
 */
#include <math.h>
#include <pthread.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#pragma pack(push, 1)
typedef struct { uint8_t isFixed; double initialValue; } nbo_weight;            /*  9 B */
typedef struct { int8_t isEvidence; int64_t initialValue; int16_t dataType;
                 int64_t cardinality; int64_t vtf_offset; } nbo_variable;        /* 27 B */
typedef struct { int16_t factorFunction; int64_t weightId; double featureValue;
                 int64_t arity; int64_t ftv_offset; } nbo_factor;                /* 34 B */
typedef struct { int64_t vid; int64_t dense_equal_to; } nbo_ftv;                 /* 16 B */
typedef struct { int64_t value; int64_t factor_index_offset;
                 int64_t factor_index_length; } nbo_vtf;                         /* 24 B */
#pragma pack(pop)

/* ------------------------------------------------------------------ */
/* MT19937 (Matsumoto & Nishimura 1998), seeded/consumed like numba.   */
/* ------------------------------------------------------------------ */
#define MT_N 624
#define MT_M 397
typedef struct { uint32_t mt[MT_N]; int idx; } nbo_mt;

void nbo_mt_seed(nbo_mt *s, uint32_t seed)
{
    for (int i = 0; i < MT_N; i++) {
        s->mt[i] = seed;
        seed = 1812433253u * (seed ^ (seed >> 30)) + (uint32_t)i + 1u;
    }
    s->idx = MT_N;
}

static void mt_twist(nbo_mt *s)
{
    uint32_t *mt = s->mt;
    for (int i = 0; i < MT_N; i++) {
        uint32_t y = (mt[i] & 0x80000000u) | (mt[(i + 1) % MT_N] & 0x7fffffffu);
        uint32_t x = mt[(i + MT_M) % MT_N] ^ (y >> 1);
        if (y & 1u) x ^= 0x9908b0dfu;
        mt[i] = x;
    }
    s->idx = 0;
}

static uint32_t mt_u32(nbo_mt *s)
{
    if (s->idx >= MT_N) mt_twist(s);
    uint32_t y = s->mt[s->idx++];
    y ^= y >> 11;
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    y ^= y >> 18;
    return y;
}

double nbo_mt_double(nbo_mt *s)
{
    uint32_t a = mt_u32(s) >> 5, b = mt_u32(s) >> 6;
    return ((double)a * 67108864.0 + (double)b) / 9007199254740992.0;
}

/* Per-thread generator pair: np.random.* and random.* are distinct in numba. */
typedef struct { nbo_mt np; nbo_mt py; } nbo_rng;

void nbo_rng_seed(nbo_rng *r, uint32_t seed)
{
    nbo_mt_seed(&r->np, seed);
    nbo_mt_seed(&r->py, seed);
}

/* ------------------------------------------------------------------ */
/* Graph view: the arrays FactorGraph owns (factorgraph.py:30-73).     */
/* ------------------------------------------------------------------ */
typedef struct {
    const nbo_weight *weight;     int64_t n_weight;
    const nbo_variable *variable; int64_t n_var;
    const nbo_factor *factor;     int64_t n_factor;
    const nbo_ftv *fmap;          int64_t n_fmap;
    const nbo_vtf *vmap;          int64_t n_vmap;
    const int64_t *factor_index;  int64_t n_findex;
    const int64_t *cstart;        /* n_var + 1 */
    int64_t *count;
    int64_t *var_value;           /* copy 0 */
    int64_t *var_value_evid;      /* copy 0 */
    double *weight_value;         /* copy 0 */
} nbo_graph;

enum {
    F_NOOP = -1, F_IMPLY_NATURAL = 0, F_OR = 1, F_AND = 2, F_EQUAL = 3, F_ISTRUE = 4,
    F_LINEAR = 7, F_RATIO = 8, F_LOGICAL = 9, F_AND_CAT = 12, F_IMPLY_MLN = 13,
    F_OR_CAT = 14, F_EQUAL_CAT_CONST = 15, F_IMPLY_NATURAL_CAT = 16, F_IMPLY_MLN_CAT = 17,
    F_DP_CLASS_PRIOR = 18, F_DP_LF_PRIOR = 19, F_DP_LF_PROPENSITY = 20, F_DP_LF_ACCURACY = 21,
    F_DP_LF_CLASS_PROPENSITY = 22, F_DP_DEP_FIXING = 23, F_DP_DEP_REINFORCING = 24,
    F_DP_DEP_EXCLUSIVE = 25, F_DP_DEP_SIMILAR = 26, F_UFO = 30
};

/* Value of fmap slot l as eval_factor sees it: the sampled variable is forced
 * to `value`, everything else comes from the chain (inference.py:164-165 and
 * every other branch). */
static inline int64_t member_value(const nbo_ftv *fmap, int64_t l, int64_t var_samp,
                                   int64_t value, const int64_t *vals)
{
    int64_t vid = fmap[l].vid;
    return vid == var_samp ? value : vals[vid];
}

/* The three *_MLN/_CAT implication branches read the head through
 * var_value[var_copy][l] with l an fmap SLOT, not a variable id
 * (inference.py:243,277,292).  Restated as coded; out-of-range slots (numba
 * would read out of bounds) yield 0 and set *err = 2. */
static inline int64_t head_value_as_coded(const nbo_ftv *fmap, int64_t l, int64_t var_samp,
                                          int64_t value, const int64_t *vals,
                                          int64_t n_var, int *err)
{
    if (fmap[l].vid == var_samp) return value;
    if (l < 0 || l >= n_var) { if (err) *err = 2; return 0; }
    return vals[l];
}

/* inference.py:149-413 eval_factor.  Returns the factor function value as a
 * double (numba unifies the int/float returns to float64).  *err: 1 = factor
 * function not implemented (inference.py:410-413), 2 = see above. */
double nbo_eval_factor(const nbo_graph *g, int64_t factor_id, int64_t var_samp,
                       int64_t value, const int64_t *vals, int *err)
{
    const nbo_factor *fac = &g->factor[factor_id];
    const nbo_ftv *fmap = g->fmap;
    const int64_t s = fac->ftv_offset, e = s + fac->arity;
    int64_t l, v, head;

    switch (fac->factorFunction) {
    case F_NOOP:                                   /* :160-161 */
        return 0;
    case F_IMPLY_NATURAL:                          /* :162-176 */
        for (l = s; l < e; l++)
            if (member_value(fmap, l, var_samp, value, vals) == 0) return 0;
        head = member_value(fmap, e - 1, var_samp, value, vals);
        return head ? 1 : -1;
    case F_OR:                                     /* :177-183 */
        for (l = s; l < e; l++)
            if (member_value(fmap, l, var_samp, value, vals) == 1) return 1;
        return -1;
    case F_EQUAL:                                  /* :184-192 */
        v = member_value(fmap, s, var_samp, value, vals);
        for (l = s + 1; l < e; l++)
            if (member_value(fmap, l, var_samp, value, vals) != v) return -1;
        return 1;
    case F_AND:
    case F_ISTRUE:                                 /* :193-200 */
        for (l = s; l < e; l++)
            if (member_value(fmap, l, var_samp, value, vals) == 0) return -1;
        return 1;
    case F_LINEAR: {                               /* :201-211 */
        int64_t res = 0;
        head = member_value(fmap, e - 1, var_samp, value, vals);
        for (l = s; l < e - 1; l++)
            if (member_value(fmap, l, var_samp, value, vals) == head) res++;
        return (double)res;
    }
    case F_RATIO: {                                /* :212-222 */
        int64_t res = 1;
        head = member_value(fmap, e - 1, var_samp, value, vals);
        for (l = s; l < e - 1; l++)
            if (member_value(fmap, l, var_samp, value, vals) == head) res++;
        return log((double)res);
    }
    case F_LOGICAL:                                /* :223-231 */
        head = member_value(fmap, e - 1, var_samp, value, vals);
        for (l = s; l < e - 1; l++)
            if (member_value(fmap, l, var_samp, value, vals) == head) return 1;
        return 0;
    case F_IMPLY_MLN:                              /* :232-246 */
        for (l = s; l < e - 1; l++)
            if (member_value(fmap, l, var_samp, value, vals) == 0) return 1;
        head = head_value_as_coded(fmap, e - 1, var_samp, value, vals, g->n_var, err);
        return head ? 1 : 0;
    case F_AND_CAT:
    case F_EQUAL_CAT_CONST:                        /* :251-258 */
        for (l = s; l < e; l++)
            if (member_value(fmap, l, var_samp, value, vals) != fmap[l].dense_equal_to) return 0;
        return 1;
    case F_OR_CAT:                                 /* :259-265 */
        for (l = s; l < e; l++)
            if (member_value(fmap, l, var_samp, value, vals) == fmap[l].dense_equal_to) return 1;
        return -1;
    case F_IMPLY_NATURAL_CAT:                      /* :266-280 */
        for (l = s; l < e - 1; l++)
            if (member_value(fmap, l, var_samp, value, vals) != fmap[l].dense_equal_to) return 0;
        head = head_value_as_coded(fmap, e - 1, var_samp, value, vals, g->n_var, err);
        return head == fmap[e - 1].dense_equal_to ? 1 : -1;
    case F_IMPLY_MLN_CAT:                          /* :281-295 */
        for (l = s; l < e - 1; l++)
            if (member_value(fmap, l, var_samp, value, vals) != fmap[l].dense_equal_to) return 1;
        head = head_value_as_coded(fmap, e - 1, var_samp, value, vals, g->n_var, err);
        return head == fmap[e - 1].dense_equal_to ? 1 : 0;
    case F_DP_CLASS_PRIOR:                         /* :301-305 */
        return member_value(fmap, s, var_samp, value, vals) == 1 ? 1 : -1;
    case F_DP_LF_PRIOR:                            /* :306-315 */
        v = member_value(fmap, s, var_samp, value, vals);
        return v == 2 ? -1 : (v == 0 ? 0 : 1);
    case F_DP_LF_PROPENSITY: {                     /* :316-320 */
        int64_t abstain = g->variable[fmap[s].vid].cardinality - 1;
        return member_value(fmap, s, var_samp, value, vals) == abstain ? 0 : 1;
    }
    case F_DP_LF_ACCURACY: {                       /* :321-332 */
        int64_t y = member_value(fmap, s, var_samp, value, vals);
        int64_t lf = member_value(fmap, s + 1, var_samp, value, vals);
        int64_t abstain = g->variable[fmap[s + 1].vid].cardinality - 1;
        if (lf == abstain) return 0;
        return y == lf ? 1 : -1;
    }
    case F_DP_LF_CLASS_PROPENSITY: {               /* :333-347 */
        int64_t y = member_value(fmap, s, var_samp, value, vals);
        int64_t lf = member_value(fmap, s + 1, var_samp, value, vals);
        int64_t abstain = g->variable[fmap[s + 1].vid].cardinality - 1;
        if (lf == abstain) return 0;
        return y == 1 ? 1 : -1;
    }
    case F_DP_DEP_FIXING:                          /* :348-364 */
    case F_DP_DEP_REINFORCING: {                   /* :365-381 */
        int64_t y = member_value(fmap, s, var_samp, value, vals);
        int64_t l1 = member_value(fmap, s + 1, var_samp, value, vals);
        int64_t l2 = member_value(fmap, s + 2, var_samp, value, vals);
        int64_t abstain = g->variable[fmap[s + 1].vid].cardinality - 1;
        if (l1 == abstain) return l2 != 1 ? -1 : 0;
        if (fac->factorFunction == F_DP_DEP_FIXING) {
            if (l1 == 0 && l2 == 1 && y == 1) return 1;
            if (l1 == 1 && l2 == 0 && y == 0) return 1;
        } else {
            if (l1 == 0 && l2 == 0 && y == 0) return 1;
            if (l1 == 1 && l2 == 1 && y == 1) return 1;
        }
        return 0;
    }
    case F_DP_DEP_EXCLUSIVE: {                     /* :382-388 */
        int64_t l1 = member_value(fmap, s, var_samp, value, vals);
        int64_t l2 = member_value(fmap, s + 1, var_samp, value, vals);
        int64_t abstain = g->variable[fmap[s].vid].cardinality - 1;
        return (l1 == abstain || l2 == abstain) ? 0 : -1;
    }
    case F_DP_DEP_SIMILAR:                         /* :389-394 */
        return member_value(fmap, s, var_samp, value, vals) ==
               member_value(fmap, s + 1, var_samp, value, vals) ? 1 : 0;
    case F_UFO:                                    /* :399-405 */
        v = member_value(fmap, s, var_samp, value, vals);
        if (v == 0) return 0;
        return (double)member_value(fmap, s + v - 1, var_samp, value, vals);
    default:                                       /* :410-413 */
        if (err) *err = 1;
        return 0;
    }
}

/* inference.py:55-71 potential.  Note featureValue is NOT used here. */
double nbo_potential(const nbo_graph *g, int64_t var_samp, int64_t value,
                     const int64_t *vals, int *err)
{
    const nbo_variable *var = &g->variable[var_samp];
    int64_t off = var->dataType == 0 ? 0 : value;
    const nbo_vtf *vtf = &g->vmap[var->vtf_offset + off];
    double p = 0.0;
    for (int64_t k = vtf->factor_index_offset;
         k < vtf->factor_index_offset + vtf->factor_index_length; k++) {
        int64_t fid = g->factor_index[k];
        p += g->weight_value[g->factor[fid].weightId] *
             nbo_eval_factor(g, fid, var_samp, value, vals, err);
    }
    return p;
}

/* inference.py:36-52 draw_sample: exp, inclusive scan, one uniform, first
 * k with Z[k] >= z (np.argmax of an all-False mask is 0). */
static int64_t draw_sample(const nbo_graph *g, int64_t var_samp, const int64_t *vals,
                           double *Z, nbo_rng *rng, int *err)
{
    int64_t card = g->variable[var_samp].cardinality;
    for (int64_t k = 0; k < card; k++) Z[k] = exp(nbo_potential(g, var_samp, k, vals, err));
    for (int64_t k = 1; k < card; k++) Z[k] += Z[k - 1];
    double z = nbo_mt_double(&rng->np) * Z[card - 1];
    for (int64_t k = 0; k < card; k++)
        if (Z[k] >= z) return k;
    return 0;
}

/* inference.py:10-33 gibbsthread. */
int nbo_gibbsthread(const nbo_graph *g, int64_t shard, int64_t nshards, double *Z,
                    int sample_evidence, int burnin, nbo_rng *rng)
{
    int err = 0;
    int64_t nvar = g->n_var;
    int64_t start = (shard * nvar) / nshards, end = ((shard + 1) * nvar) / nshards;
    for (int64_t v = start; v < end; v++) {
        const nbo_variable *var = &g->variable[v];
        if (var->isEvidence == 4) continue;
        if (var->isEvidence == 0 || sample_evidence) {
            int64_t k = draw_sample(g, v, g->var_value, Z, rng, &err);
            g->var_value[v] = k;
            if (!burnin) {
                if (var->cardinality == 2) g->count[g->cstart[v]] += k;
                else g->count[g->cstart[v] + k] += 1;
            }
        }
    }
    return err;
}

static int cmp_i64(const void *a, const void *b)
{
    int64_t x = *(const int64_t *)a, y = *(const int64_t *)b;
    return (x > y) - (x < y);
}

/* learning.py:34-43 get_factor_id_range. */
static void bucket_range(const nbo_graph *g, int64_t v, int64_t val, int64_t *s, int64_t *e)
{
    const nbo_variable *var = &g->variable[v];
    const nbo_vtf *vtf = &g->vmap[var->vtf_offset + (var->dataType == 0 ? 0 : val)];
    *s = vtf->factor_index_offset;
    *e = *s + vtf->factor_index_length;
}

/* learning.py:46-125 sample_and_sgd. */
static void sample_and_sgd(const nbo_graph *g, int64_t v, double step, int regularization,
                           double reg_param, double truncation, double *Z, int64_t *fids,
                           int learn_non_evidence, nbo_rng *rng, int *err)
{
    const nbo_variable *var = &g->variable[v];
    int64_t evidence, proposal;
    if (var->isEvidence != 1) evidence = draw_sample(g, v, g->var_value_evid, Z, rng, err);
    else evidence = var->initialValue;
    g->var_value_evid[v] = evidence;
    proposal = draw_sample(g, v, g->var_value, Z, rng, err);
    g->var_value[v] = proposal;
    if (!learn_non_evidence && var->isEvidence != 1) return;

    int64_t s0, e0, s;
    bucket_range(g, v, evidence, &s0, &e0);
    if (evidence != proposal) {
        int64_t s1, e1;
        bucket_range(g, v, proposal, &s1, &e1);
        s = (e0 - s0) + (e1 - s1);
        memcpy(fids, g->factor_index + s0, (size_t)(e0 - s0) * sizeof(int64_t));
        memcpy(fids + (e0 - s0), g->factor_index + s1, (size_t)(e1 - s1) * sizeof(int64_t));
        qsort(fids, (size_t)s, sizeof(int64_t), cmp_i64);
    } else {
        s = e0 - s0;
        memcpy(fids, g->factor_index + s0, (size_t)s * sizeof(int64_t));
    }

    int truncate = 0;
    if (regularization == 1) truncate = nbo_mt_double(&rng->py) < 1.0 / truncation;

    int64_t last = -1;
    for (int64_t i = 0; i < s; i++) {
        int64_t fid = fids[i];
        if (fid == last) continue;
        last = fid;
        int64_t wid = g->factor[fid].weightId;
        if (g->weight[wid].isFixed) continue;
        double p0 = nbo_eval_factor(g, fid, v, evidence, g->var_value_evid, err);
        double p1 = nbo_eval_factor(g, fid, v, proposal, g->var_value, err);
        double gradient = (p1 - p0) * g->factor[fid].featureValue;
        double w = g->weight_value[wid];
        if (regularization == 2) {
            w *= 1.0 / (1.0 + reg_param * step);
            w -= step * gradient;
        } else if (regularization == 1) {
            w -= step * gradient;
            if (truncate) {
                double l1delta = reg_param * step * truncation;
                if (w > 0) { w = w - l1delta; if (w < 0) w = 0; }
                else       { w = w + l1delta; if (w > 0) w = 0; }
            }
        } else {
            w -= step * gradient;
        }
        g->weight_value[wid] = w;
    }
}

/* learning.py:12-31 learnthread. */
int nbo_learnthread(const nbo_graph *g, int64_t shard, int64_t nshards, double step,
                    int regularization, double reg_param, double truncation, double *Z,
                    int64_t *fids, int learn_non_evidence, nbo_rng *rng)
{
    int err = 0;
    int64_t nvar = g->n_var;
    int64_t start = (shard * nvar) / nshards, end = ((shard + 1) * nvar) / nshards;
    for (int64_t v = start; v < end; v++) {
        if (g->variable[v].isEvidence == 4) continue;
        sample_and_sgd(g, v, step, regularization, reg_param, truncation, Z, fids,
                       learn_non_evidence, rng, &err);
    }
    return err;
}

/* ------------------------------------------------------------------ */
/* Epoch drivers (factorgraph.py:13-24 run_pool, :129-208).            */
/* Threads own contiguous variable ranges and race on shared arrays    */
/* exactly like the reference's Hogwild pool.                          */
/* ------------------------------------------------------------------ */
typedef struct {
    const nbo_graph *g; int64_t shard, nshards; int learn;
    int sample_evidence, burnin;
    double step; int regularization; double reg_param, truncation; int learn_non_evidence;
    double *Z; int64_t *fids; nbo_rng *rng; int err;
} shard_job;

static void *shard_main(void *p)
{
    shard_job *j = (shard_job *)p;
    if (j->learn)
        j->err = nbo_learnthread(j->g, j->shard, j->nshards, j->step, j->regularization,
                                 j->reg_param, j->truncation, j->Z, j->fids,
                                 j->learn_non_evidence, j->rng);
    else
        j->err = nbo_gibbsthread(j->g, j->shard, j->nshards, j->Z, j->sample_evidence,
                                 j->burnin, j->rng);
    return NULL;
}

static int run_pool(shard_job *jobs, int nthreads)
{
    int err = 0;
    if (nthreads == 1) {
        shard_main(&jobs[0]);
    } else {
        pthread_t *t = (pthread_t *)malloc(sizeof(pthread_t) * (size_t)nthreads);
        for (int i = 0; i < nthreads; i++) pthread_create(&t[i], NULL, shard_main, &jobs[i]);
        for (int i = 0; i < nthreads; i++) pthread_join(t[i], NULL);
        free(t);
    }
    for (int i = 0; i < nthreads; i++) err |= jobs[i].err;
    return err;
}

typedef struct { int nthreads; int64_t maxcard, maxbucket; double *Z; int64_t *fids;
                 nbo_rng *rng; shard_job *jobs; } nbo_pool;

nbo_pool *nbo_pool_create(const nbo_graph *g, int nthreads, uint32_t seed)
{
    nbo_pool *p = (nbo_pool *)calloc(1, sizeof(nbo_pool));
    p->nthreads = nthreads;
    p->maxcard = 1; p->maxbucket = 1;
    for (int64_t i = 0; i < g->n_var; i++)
        if (g->variable[i].cardinality > p->maxcard) p->maxcard = g->variable[i].cardinality;
    for (int64_t i = 0; i < g->n_vmap; i++)
        if (g->vmap[i].factor_index_length > p->maxbucket) p->maxbucket = g->vmap[i].factor_index_length;
    p->Z = (double *)calloc((size_t)(nthreads * p->maxcard), sizeof(double));
    p->fids = (int64_t *)calloc((size_t)(nthreads * 2 * p->maxbucket), sizeof(int64_t));
    p->rng = (nbo_rng *)calloc((size_t)nthreads, sizeof(nbo_rng));
    p->jobs = (shard_job *)calloc((size_t)nthreads, sizeof(shard_job));
    /* thread 0 is the caller's thread in the reference (threads == 1 runs
     * inline); worker threads get their own streams. */
    for (int i = 0; i < nthreads; i++) nbo_rng_seed(&p->rng[i], seed + (uint32_t)i);
    return p;
}

void nbo_pool_destroy(nbo_pool *p)
{
    if (!p) return;
    free(p->Z); free(p->fids); free(p->rng); free(p->jobs); free(p);
}

/* factorgraph.py:129-175: `epochs` sweeps of gibbsthread over the pool. */
int nbo_gibbs_epochs(const nbo_graph *g, nbo_pool *p, int64_t epochs, int sample_evidence,
                     int burnin)
{
    int err = 0;
    for (int64_t ep = 0; ep < epochs; ep++) {
        for (int i = 0; i < p->nthreads; i++) {
            shard_job *j = &p->jobs[i];
            memset(j, 0, sizeof(*j));
            j->g = g; j->shard = i; j->nshards = p->nthreads; j->learn = 0;
            j->sample_evidence = sample_evidence; j->burnin = burnin;
            j->Z = p->Z + (size_t)i * (size_t)p->maxcard; j->rng = &p->rng[i];
        }
        err |= run_pool(p->jobs, p->nthreads);
    }
    return err;
}

/* factorgraph.py:188-206: learning epochs with stepsize *= decay; returns the
 * final stepsize through *stepsize. */
int nbo_learn_epochs(const nbo_graph *g, nbo_pool *p, int64_t epochs, double *stepsize,
                     double decay, int regularization, double reg_param, double truncation,
                     int learn_non_evidence)
{
    int err = 0;
    for (int64_t ep = 0; ep < epochs; ep++) {
        for (int i = 0; i < p->nthreads; i++) {
            shard_job *j = &p->jobs[i];
            memset(j, 0, sizeof(*j));
            j->g = g; j->shard = i; j->nshards = p->nthreads; j->learn = 1;
            j->step = *stepsize; j->regularization = regularization;
            j->reg_param = reg_param; j->truncation = truncation;
            j->learn_non_evidence = learn_non_evidence;
            j->Z = p->Z + (size_t)i * (size_t)p->maxcard;
            j->fids = p->fids + (size_t)i * 2 * (size_t)p->maxbucket;
            j->rng = &p->rng[i];
        }
        err |= run_pool(p->jobs, p->nthreads);
        *stepsize *= decay;
    }
    return err;
}

/* ------------------------------------------------------------------ */
/* dataloading.py:16-81 compute_var_map (integer work, bit-exact).     */
/* ------------------------------------------------------------------ */
void nbo_compute_var_map(nbo_variable *variables, int64_t n_var, const nbo_factor *factors,
                         int64_t n_factor, const nbo_ftv *fmap, int64_t n_fmap, nbo_vtf *vmap,
                         int64_t n_vmap, int64_t *factor_index, const uint8_t *domain_mask,
                         const int64_t *factors_to_skip, int64_t n_skip)
{
    /* :20-30 implicit domains */
    for (int64_t i = 0; i < n_var; i++) {
        if (variables[i].dataType == 0 || domain_mask[i]) continue;
        for (int64_t k = 0; k < variables[i].cardinality; k++)
            vmap[variables[i].vtf_offset + k].value = k;
    }
    /* :33-38 bucket lengths from every fmap entry */
    for (int64_t j = 0; j < n_fmap; j++) {
        int64_t vid = fmap[j].vid;
        int64_t val = variables[vid].dataType == 1 ? fmap[j].dense_equal_to : 0;
        vmap[variables[vid].vtf_offset + val].factor_index_length += 1;
    }
    /* :40-46 exclusive scan */
    int64_t last_len = 0, last_off = 0;
    for (int64_t i = 0; i < n_vmap; i++) {
        vmap[i].factor_index_offset = last_off + last_len;
        last_len = vmap[i].factor_index_length;
        last_off = vmap[i].factor_index_offset;
    }
    /* :48-65 scatter factor ids in factor order */
    int64_t *offsets = (int64_t *)malloc(sizeof(int64_t) * (size_t)(n_vmap > 0 ? n_vmap : 1));
    for (int64_t i = 0; i < n_vmap; i++) offsets[i] = vmap[i].factor_index_offset;
    int64_t fts = 0;
    for (int64_t i = 0; i < n_factor; i++) {
        if (fts < n_skip && factors_to_skip[fts] == i) { fts++; continue; }
        for (int64_t j = factors[i].ftv_offset; j < factors[i].ftv_offset + factors[i].arity; j++) {
            int64_t vid = fmap[j].vid;
            int64_t val = variables[vid].dataType == 1 ? fmap[j].dense_equal_to : 0;
            int64_t b = variables[vid].vtf_offset + val;
            factor_index[offsets[b]++] = i;
        }
    }
    free(offsets);
    /* :67-81 sort + unique each bucket; offsets are not compacted */
    for (int64_t i = 0; i < n_vmap; i++) {
        int64_t off = vmap[i].factor_index_offset, len = vmap[i].factor_index_length;
        qsort(factor_index + off, (size_t)len, sizeof(int64_t), cmp_i64);
        int64_t n = 0, last = -1;
        for (int64_t k = 0; k < len; k++) {
            int64_t fid = factor_index[off + k];
            if (fid == last) continue;
            last = fid;
            factor_index[off + n++] = fid;
        }
        vmap[i].factor_index_length = n;
    }
}

/* ------------------------------------------------------------------ */
/* Exact marginals by enumeration (tiny graphs only).  Uses            */
/* eval_factor(var_samp = -1), i.e. every member read from the state,  */
/* the way SURVEY.md section 4 pins the statistical tests.             */
/* out has cstart[n_var] entries laid out like `count` / `marginals`.  */
/* Evidence variables (isEvidence == 1) are clamped iff clamp_evidence.*/
/* ------------------------------------------------------------------ */
int nbo_exact_marginals(const nbo_graph *g, int clamp_evidence, double *out, double *logZ)
{
    int64_t n = g->n_var, total = g->cstart[n];
    int64_t *state = (int64_t *)calloc((size_t)(n > 0 ? n : 1), sizeof(int64_t));
    double *acc = (double *)calloc((size_t)(total > 0 ? total : 1), sizeof(double));
    double Zsum = 0.0;
    int err = 0;
    for (int64_t i = 0; i < n; i++)
        if (clamp_evidence && g->variable[i].isEvidence == 1) state[i] = g->variable[i].initialValue;
    for (;;) {
        double en = 0.0;
        for (int64_t f = 0; f < g->n_factor; f++)
            en += g->weight_value[g->factor[f].weightId] *
                  nbo_eval_factor(g, f, -1, 0, state, &err);
        double w = exp(en);
        Zsum += w;
        for (int64_t i = 0; i < n; i++) {
            if (g->variable[i].cardinality == 2) acc[g->cstart[i]] += w * (double)state[i];
            else acc[g->cstart[i] + state[i]] += w;
        }
        /* odometer over the free variables */
        int64_t i = 0;
        for (; i < n; i++) {
            if (clamp_evidence && g->variable[i].isEvidence == 1) continue;
            if (++state[i] < g->variable[i].cardinality) break;
            state[i] = 0;
        }
        if (i == n) break;
    }
    for (int64_t k = 0; k < total; k++) out[k] = acc[k] / Zsum;
    if (logZ) *logZ = log(Zsum);
    free(state); free(acc);
    return err;
}

int nbo_sizeof_rng(void) { return (int)sizeof(nbo_rng); }
int nbo_sizeof_graph(void) { return (int)sizeof(nbo_graph); }

/* ------------------------------------------------------------------ */
/* Counter-based streams of the CUDA library, restated from the        */
/* specification (Salmon et al., SC'11; Random123 constants) so that   */
/* tests can replay every draw of a sweep on the host.  The device     */
/* headers are deliberately NOT included: this is a second,            */
/* independent implementation.                                         */
/* ------------------------------------------------------------------ */
void nbo_philox4x32(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4])
{
    uint32_t x0 = ctr[0], x1 = ctr[1], x2 = ctr[2], x3 = ctr[3], k0 = key[0], k1 = key[1];
    for (int r = 0; r < 10; r++) {
        uint64_t a = (uint64_t)0xD2511F53u * x0, b = (uint64_t)0xCD9E8D57u * x2;
        uint32_t y0 = (uint32_t)(b >> 32) ^ x1 ^ k0, y1 = (uint32_t)b;
        uint32_t y2 = (uint32_t)(a >> 32) ^ x3 ^ k1, y3 = (uint32_t)a;
        x0 = y0; x1 = y1; x2 = y2; x3 = y3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = x0; out[1] = x1; out[2] = x2; out[3] = x3;
}

void nbo_philox2x32(const uint32_t ctr[2], uint32_t key, uint32_t out[2])
{
    uint32_t x0 = ctr[0], x1 = ctr[1];
    for (int r = 0; r < 10; r++) {
        uint64_t a = (uint64_t)0xD256D193u * x0;
        uint32_t y0 = (uint32_t)(a >> 32) ^ x1 ^ key;
        x1 = (uint32_t)a;
        x0 = y0;
        key += 0x9E3779B9u;
    }
    out[0] = x0; out[1] = x1;
}

/* 53-bit uniform in [0, 1): the top 53 bits of hi:lo */
double nbo_u53(uint32_t hi, uint32_t lo)
{
    return (double)((((uint64_t)hi << 32) | lo) >> 11) / 9007199254740992.0;
}

/* 32-bit key of the single-draw (Philox2x32) streams: seed, the epoch bits above 32 and the tag
 * mixed by the MurmurHash3 finaliser half, folded to 32 bits. */
uint32_t nbo_fold_key(uint64_t seed, uint64_t epoch, uint32_t tag)
{
    uint64_t x = seed ^ ((epoch >> 32) * 0x9E3779B97F4A7C15ull) ^ ((uint64_t)tag << 56);
    x ^= x >> 33;
    x *= 0xFF51AFD7ED558CCDull;
    x ^= x >> 33;
    return (uint32_t)x ^ (uint32_t)(x >> 32);
}

/* The single uniform of a record row: counter (id, low epoch word), folded key. */
double nbo_philox2x32_u53(uint32_t id, uint64_t epoch, uint64_t seed, uint32_t tag)
{
    uint32_t c[2] = {id, (uint32_t)epoch}, o[2];
    nbo_philox2x32(c, nbo_fold_key(seed, epoch, tag), o);
    return nbo_u53(o[0], o[1]);
}

/* The multi-draw stream of one (variable, epoch, tag): counter (id, low epoch word,
 * epoch bits 32..47 | tag << 24, block), key = seed; the four words of a block are read in
 * order, then block++. */
typedef struct { uint32_t c[3]; uint32_t key[2]; uint32_t block; uint32_t r[4]; int used; } nbo_stream;

void nbo_stream_init(nbo_stream *s, uint32_t id, uint64_t epoch, uint32_t tag, uint64_t seed)
{
    s->c[0] = id;
    s->c[1] = (uint32_t)epoch;
    s->c[2] = (uint32_t)((epoch >> 32) & 0xFFFFu) | (tag << 24);
    s->key[0] = (uint32_t)seed;
    s->key[1] = (uint32_t)(seed >> 32);
    s->block = 0;
    s->used = 4;
}

uint32_t nbo_stream_word(nbo_stream *s)
{
    if (s->used == 4) {
        uint32_t ctr[4] = {s->c[0], s->c[1], s->c[2], s->block++};
        nbo_philox4x32(ctr, s->key, s->r);
        s->used = 0;
    }
    return s->r[s->used++];
}

/* two words, the first one high: the 53-bit draw of small-cardinality rows */
double nbo_stream_next(nbo_stream *s)
{
    uint32_t hi = nbo_stream_word(s);
    return nbo_u53(hi, nbo_stream_word(s));
}

/* one word, centred: the per-value decisions of the reservoir */
double nbo_stream_next32(nbo_stream *s)
{
    return ((double)nbo_stream_word(s) + 0.5) / 4294967296.0;
}

int nbo_sizeof_stream(void) { return (int)sizeof(nbo_stream); }

/* ------------------------------------------------------------------ */
/* float64 decision rules.  Each returns the pick and, through         */
/* *margin, how far the uniform was from changing it (in units of the  */
/* uniform): a float32 implementation of the same rule may only pick   */
/* differently when the margin is of the order of its rounding.        */
/* ------------------------------------------------------------------ */
static double dmin(double a, double b) { return a < b ? a : b; }

/* Boolean rule: P(0) = 1 / (1 + exp(e1 - e0)), pick 0 iff u <= P(0) */
int64_t nbo_draw_bool(double e0, double e1, double u, double *margin)
{
    double p0 = 1.0 / (1.0 + exp(e1 - e0));
    *margin = fabs(u - p0);
    return u <= p0 ? 0 : 1;
}

/* inverse CDF (draw_sample, inference.py:36-52, maximum subtracted): the first k whose cumulative
 * mass reaches u * total; card - 1 if none does.  Margin: distance of u to the nearest boundary. */
int64_t nbo_draw_cdf(const double *e, int64_t card, double u, double *margin)
{
    double m = e[0], tot = 0.0, acc = 0.0;
    for (int64_t k = 1; k < card; k++) if (e[k] > m) m = e[k];
    for (int64_t k = 0; k < card; k++) tot += exp(e[k] - m);
    int64_t pick = -1;
    *margin = INFINITY;
    for (int64_t k = 0; k < card; k++) {
        acc += exp(e[k] - m);
        if (k < card - 1) *margin = dmin(*margin, fabs(acc / tot - u));
        if (pick < 0 && acc >= u * tot) pick = k;
    }
    return pick < 0 ? card - 1 : pick;
}

/* Weighted reservoir with a running maximum: group j (energy e, `mult` values) replaces the pick
 * when u * s < t, t = mult * exp(e - m) its mass and s the mass seen so far including it.  The first
 * group always takes the pick (its uniform is still consumed). */
typedef struct { double m, s; int empty; } nbo_reservoir;

static int reservoir_add(nbo_reservoir *r, double e, double mult, double u, double *margin)
{
    if (r->empty) { r->m = e; r->s = mult; r->empty = 0; return 1; }
    double t;
    if (e > r->m) { r->s = r->s * exp(r->m - e) + mult; r->m = e; t = mult; }
    else { t = mult * exp(e - r->m); r->s += t; }
    *margin = dmin(*margin, fabs(u - t / r->s));
    return u * r->s < t;
}

/* Streaming categorical draw.  nonempty == NULL: every value is its own group, in ascending order
 * (dataType 0 rows, warp rows).  Otherwise the values with nonempty[k] in ascending order, then ONE
 * group of the n_empty remaining values (energy 0), inside which a second uniform picks the
 * floor(u * n_empty)-th empty value. */
int64_t nbo_draw_reservoir(const double *e, int64_t card, const uint8_t *nonempty, nbo_stream *s, double *margin)
{
    nbo_reservoir r = {0.0, 0.0, 1};
    int64_t pick = 0, n_empty = 0;
    *margin = INFINITY;
    for (int64_t k = 0; k < card; k++) {
        if (nonempty && !nonempty[k]) { n_empty++; continue; }
        if (reservoir_add(&r, e[k], 1.0, nbo_stream_next32(s), margin)) pick = k;
    }
    if (n_empty > 0 && reservoir_add(&r, 0.0, (double)n_empty, nbo_stream_next32(s), margin)) {
        double x = nbo_stream_next32(s) * (double)n_empty;
        int64_t j = (int64_t)x;
        if (j > n_empty - 1) j = n_empty - 1;
        *margin = dmin(*margin, dmin(x - floor(x), ceil(x) - x) / (double)n_empty);
        for (int64_t k = 0; k < card; k++)
            if (!nonempty[k] && j-- == 0) { pick = k; break; }
    }
    return pick;
}

/* ------------------------------------------------------------------ */
/* Batched entries for the sweep replay.                               */
/* ------------------------------------------------------------------ */
/* potential(v, k) for every value of each listed variable, under chain 0 (var_value) or 1
 * (var_value_evid); variable ids[i] writes cardinality entries from out[off], off running. */
int nbo_energies(const nbo_graph *g, int chain, const int64_t *ids, int64_t n, double *out)
{
    int err = 0;
    const int64_t *vals = chain ? g->var_value_evid : g->var_value;
    int64_t off = 0;
    for (int64_t i = 0; i < n; i++) {
        int64_t card = g->variable[ids[i]].cardinality;
        for (int64_t k = 0; k < card; k++) out[off++] = nbo_potential(g, ids[i], k, vals, &err);
    }
    return err;
}

/* Row classes of the CUDA library, and the rule each one samples with:
 *   PAIR / FAST (0, 1): Boolean rule, one Philox2x32 uniform;
 *   CAT (2):            inverse CDF, one Philox2x32 uniform;
 *   GEN (3):            multi-draw stream: dataType 0 with cardinality <= 4 takes one 53-bit draw
 *                       (Boolean rule for cardinality 2, inverse CDF otherwise); other dataType 0
 *                       rows a reservoir over every value; dataType 1 rows a reservoir over the
 *                       values with a non-empty bucket, then the group of the empty ones;
 *   WARP (4):           multi-draw stream: one 53-bit draw as GEN for small dataType 0 rows,
 *                       otherwise a reservoir over every value;
 *   WIDE (5):           warp rows above cardinality 255: the GEN rule. */
enum { NBO_PAIR = 0, NBO_FAST = 1, NBO_CAT = 2, NBO_GEN = 3, NBO_WARP = 4, NBO_WIDE = 5 };

static int64_t draw_one(const nbo_graph *g, int64_t v, const double *e, int cls, uint32_t id, uint64_t seed,
                        uint64_t epoch, uint32_t tag, uint8_t *nonempty, double *margin)
{
    const nbo_variable *var = &g->variable[v];
    int64_t card = var->cardinality;
    if (cls == NBO_PAIR || cls == NBO_FAST)
        return nbo_draw_bool(e[0], e[1], nbo_philox2x32_u53(id, epoch, seed, tag), margin);
    if (cls == NBO_CAT) return nbo_draw_cdf(e, card, nbo_philox2x32_u53(id, epoch, seed, tag), margin);
    nbo_stream s;
    nbo_stream_init(&s, id, epoch, tag, seed);
    if (var->dataType == 0 && card <= 4) {
        double u = nbo_stream_next(&s);
        if (card == 2) return nbo_draw_bool(e[0], e[1], u, margin);
        return nbo_draw_cdf(e, card, u, margin);
    }
    if (var->dataType == 0 || cls == NBO_WARP) return nbo_draw_reservoir(e, card, NULL, &s, margin);
    for (int64_t k = 0; k < card; k++) nonempty[k] = g->vmap[var->vtf_offset + k].factor_index_length > 0;
    return nbo_draw_reservoir(e, card, nonempty, &s, margin);
}

/* Replays the draw of each listed variable from its float64 energies under `chain`.  cls[i] is
 * the row class of ids[i], rng_id[i] its stream id (low 32 bits of the global id). */
int nbo_replay_draws(const nbo_graph *g, int chain, const int64_t *ids, int64_t n, const int32_t *cls,
                     const uint32_t *rng_id, uint64_t seed, uint64_t epoch, uint32_t tag, int64_t *pick,
                     double *margin)
{
    int err = 0;
    const int64_t *vals = chain ? g->var_value_evid : g->var_value;
    int64_t maxcard = 1;
    for (int64_t i = 0; i < n; i++)
        if (g->variable[ids[i]].cardinality > maxcard) maxcard = g->variable[ids[i]].cardinality;
    double *e = (double *)malloc(sizeof(double) * (size_t)maxcard);
    uint8_t *ne = (uint8_t *)malloc((size_t)maxcard);
    for (int64_t i = 0; i < n; i++) {
        int64_t v = ids[i], card = g->variable[v].cardinality;
        for (int64_t k = 0; k < card; k++) e[k] = nbo_potential(g, v, k, vals, &err);
        pick[i] = draw_one(g, v, e, cls[i], rng_id[i], seed, epoch, tag, ne, &margin[i]);
    }
    free(e);
    free(ne);
    return err;
}

/* The first uniform of each listed stream: family 0 = Philox2x32 (record rows), 1 = the multi-draw
 * stream's 53-bit draw.  Used for the truncation draws of L1 learning. */
void nbo_first_uniforms(const uint32_t *rng_id, int64_t n, const int32_t *family, uint64_t seed, uint64_t epoch,
                        uint32_t tag, double *out)
{
    for (int64_t i = 0; i < n; i++) {
        if (family[i] == 0) { out[i] = nbo_philox2x32_u53(rng_id[i], epoch, seed, tag); continue; }
        nbo_stream s;
        nbo_stream_init(&s, rng_id[i], epoch, tag, seed);
        out[i] = nbo_stream_next(&s);
    }
}

/* learning.py:73-108 for a batch of variables whose evidence-chain value is ev[i] and free-chain
 * value prop[i]: every learnable factor of the buckets of ev and prop (once per factor) adds
 * (f(prop | var_value) - f(ev | var_value_evid)) * featureValue, rounded to 2^-20 units as the
 * library reduces it, to G_fix[weightId], and cnt_inc[i] to cnt[weightId]. */
int nbo_cell_gradients(const nbo_graph *g, const int64_t *ids, int64_t n, const int64_t *ev, const int64_t *prop,
                       const uint32_t *cnt_inc, int64_t *G_fix, int64_t *cnt)
{
    int err = 0;
    int64_t maxb = 1;
    for (int64_t i = 0; i < g->n_vmap; i++)
        if (g->vmap[i].factor_index_length > maxb) maxb = g->vmap[i].factor_index_length;
    int64_t *fids = (int64_t *)malloc(sizeof(int64_t) * (size_t)(2 * maxb));
    for (int64_t i = 0; i < n; i++) {
        int64_t v = ids[i], s0, e0, s1, e1, m;
        bucket_range(g, v, ev[i], &s0, &e0);
        memcpy(fids, g->factor_index + s0, (size_t)(e0 - s0) * sizeof(int64_t));
        m = e0 - s0;
        if (ev[i] != prop[i]) {
            bucket_range(g, v, prop[i], &s1, &e1);
            memcpy(fids + m, g->factor_index + s1, (size_t)(e1 - s1) * sizeof(int64_t));
            m += e1 - s1;
            qsort(fids, (size_t)m, sizeof(int64_t), cmp_i64);
        }
        int64_t last = -1;
        for (int64_t j = 0; j < m; j++) {
            int64_t fid = fids[j];
            if (fid == last) continue;
            last = fid;
            int64_t wid = g->factor[fid].weightId;
            if (g->weight[wid].isFixed) continue;
            double p1 = nbo_eval_factor(g, fid, v, prop[i], g->var_value, &err);
            double p0 = nbo_eval_factor(g, fid, v, ev[i], g->var_value_evid, &err);
            G_fix[wid] += llrint((p1 - p0) * g->factor[fid].featureValue * 1048576.0);
            cnt[wid] += cnt_inc[i];
        }
    }
    free(fids);
    return err;
}
