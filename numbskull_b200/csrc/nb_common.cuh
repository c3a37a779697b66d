// Internal declarations shared by the translation units of libnumbskull_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>

#include "../../include/numbskull_b200.h"

// ----------------------------------------------------------------------------
// error plumbing
// ----------------------------------------------------------------------------
void nb_set_error(const char *fmt, ...);

#define NB_CUDA(call)                                                                   \
    do {                                                                                \
        cudaError_t e_ = (call);                                                        \
        if (e_ != cudaSuccess) {                                                        \
            nb_set_error("CUDA error %s at %s:%d: %s", cudaGetErrorName(e_), __FILE__,  \
                         __LINE__, cudaGetErrorString(e_));                             \
            return NB_ERR_CUDA;                                                         \
        }                                                                               \
    } while (0)

#define NB_TRY(call)                       \
    do {                                   \
        int rc_ = (call);                  \
        if (rc_ != NB_OK) return rc_;      \
    } while (0)

#define NB_FAIL(code, ...)      \
    do {                        \
        nb_set_error(__VA_ARGS__); \
        return (code);          \
    } while (0)

// ----------------------------------------------------------------------------
// factor-function codes (dense 5-bit re-numbering of inference.py:74-146)
// ----------------------------------------------------------------------------
enum NbCode : int {
    C_NOOP = 0, C_IMPLY_NATURAL = 1, C_OR = 2, C_AND = 3, C_EQUAL = 4, C_ISTRUE = 5,
    C_LINEAR = 6, C_RATIO = 7, C_LOGICAL = 8, C_IMPLY_MLN = 9,
    C_AND_CAT = 10, C_OR_CAT = 11, C_EQUAL_CAT_CONST = 12, C_IMPLY_NATURAL_CAT = 13,
    C_IMPLY_MLN_CAT = 14,
    C_DP_CLASS_PRIOR = 15, C_DP_LF_PRIOR = 16, C_DP_LF_PROPENSITY = 17, C_DP_LF_ACCURACY = 18,
    C_DP_LF_CLASS_PROPENSITY = 19, C_DP_DEP_FIXING = 20, C_DP_DEP_REINFORCING = 21,
    C_DP_DEP_EXCLUSIVE = 22, C_DP_DEP_SIMILAR = 23, C_UFO = 24,
    C_UNKNOWN = 30,  // never emitted into a stream
    C_MARK = 31      // categorical bucket marker
};

__host__ __device__ inline int nb_code_of_func(int func)
{
    switch (func) {
    case -1: return C_NOOP;
    case 0: return C_IMPLY_NATURAL;
    case 1: return C_OR;
    case 2: return C_AND;
    case 3: return C_EQUAL;
    case 4: return C_ISTRUE;
    case 7: return C_LINEAR;
    case 8: return C_RATIO;
    case 9: return C_LOGICAL;
    case 12: return C_AND_CAT;
    case 13: return C_IMPLY_MLN;
    case 14: return C_OR_CAT;
    case 15: return C_EQUAL_CAT_CONST;
    case 16: return C_IMPLY_NATURAL_CAT;
    case 17: return C_IMPLY_MLN_CAT;
    case 18: return C_DP_CLASS_PRIOR;
    case 19: return C_DP_LF_PRIOR;
    case 20: return C_DP_LF_PROPENSITY;
    case 21: return C_DP_LF_ACCURACY;
    case 22: return C_DP_LF_CLASS_PROPENSITY;
    case 23: return C_DP_DEP_FIXING;
    case 24: return C_DP_DEP_REINFORCING;
    case 25: return C_DP_DEP_EXCLUSIVE;
    case 26: return C_DP_DEP_SIMILAR;
    case 30: return C_UFO;
    default: return C_UNKNOWN;
    }
}

// members carry a dense_equal_to word
__host__ __device__ inline bool nb_code_has_eq(int c) { return c >= C_AND_CAT && c <= C_IMPLY_MLN_CAT; }
// one extra trailing word: the as-coded "head alias" variable for the three
// implication functions that index var_value by fmap slot (inference.py:243,277,292),
// or the abstain value (cardinality - 1 of a fixed member) for the DP functions.
__host__ __device__ inline bool nb_code_has_extra(int c)
{
    return c == C_IMPLY_MLN || c == C_IMPLY_NATURAL_CAT || c == C_IMPLY_MLN_CAT ||
           (c >= C_DP_LF_PROPENSITY && c <= C_DP_DEP_EXCLUSIVE);
}
// member whose cardinality defines "abstain" (inference.py:319,327,342,356,373,387)
__host__ __device__ inline int nb_code_abstain_member(int c) { return (c == C_DP_LF_PROPENSITY || c == C_DP_DEP_EXCLUSIVE) ? 0 : 1; }

// ----------------------------------------------------------------------------
// Incidence-stream word formats.  A row (one variable) is a sequence of
// incidences, one per (variable, factor) pair of the reference's vmap bucket(s):
//   header | member words | [extra]? | [featureValue lo, hi]?
// compact header (1 word):  code:5 | feat:1 | fixed:1 | arity:5 | wid:20
// wide header (2 words):    wid:32 ; code:5 | feat:1 | fixed:1 | 0:1 | arity:24
// member word: NEW variable id; members of *_CAT functions are (id, dense_equal_to) pairs.
// A categorical variable's row has a MARK before each non-empty bucket:
//   compact: code=31 | value:27         wide: value ; code=31
// ----------------------------------------------------------------------------
#define NB_COMPACT_MAX_ARITY 31
#define NB_COMPACT_MAX_WID ((1u << 20) - 1)

struct NbHdr {
    int code, arity, feat, fixed;
    uint32_t wid;  // MARK: bucket value
};

__host__ __device__ inline uint32_t nb_pack_compact(int code, int feat, int fixed, int arity, uint32_t wid)
{
    return ((uint32_t)code << 27) | ((uint32_t)feat << 26) | ((uint32_t)fixed << 25) |
           ((uint32_t)arity << 20) | wid;
}
__host__ __device__ inline uint32_t nb_pack_wide_b(int code, int feat, int fixed, int arity)
{
    return ((uint32_t)code << 27) | ((uint32_t)feat << 26) | ((uint32_t)fixed << 25) | (uint32_t)arity;
}
__host__ __device__ inline uint32_t nb_pack_mark_compact(uint32_t value) { return ((uint32_t)C_MARK << 27) | value; }

// number of 32-bit words an incidence occupies
__host__ __device__ inline int nb_incidence_words(bool wide, int code, int arity, int feat)
{
    return (wide ? 2 : 1) + (feat ? 2 : 0) + arity * (nb_code_has_eq(code) ? 2 : 1) +
           (nb_code_has_extra(code) ? 1 : 0);
}

// vmeta word per (new) variable id: card:8 | isEvidence:4 | dataType:1 | valid:1 | fast:1 | row words:17
// (row words saturate at 2^17-1; warp-path rows take their length from wrow_ptr).  card = 0 marks a
// cardinality above 255 (2-byte graphs only): the real one is in nb_graph::d_vcard.  Device code
// reads cardinalities through NbCardOf (nb_eval.cuh), never NB_META_CARD directly.
#define NB_META_CARD(m) ((int)((m) & 0xFFu))
#define NB_META_EVID(m) ((int)(((m) >> 8) & 0xFu))
#define NB_META_DTYPE(m) ((int)(((m) >> 12) & 1u))
#define NB_META_VALID(m) ((int)(((m) >> 13) & 1u))
#define NB_META_FAST(m) ((int)(((m) >> 14) & 1u))
#define NB_META_ROWLEN(m) ((int)((m) >> 15))
#define NB_META_MAX_ROWLEN ((1u << 17) - 1)
__host__ __device__ inline uint32_t nb_pack_meta(int card, int evid, int dtype, int valid, int fast, uint32_t rowlen)
{
    if (rowlen > NB_META_MAX_ROWLEN) rowlen = NB_META_MAX_ROWLEN;
    return (uint32_t)card | ((uint32_t)(evid & 0xF) << 8) | ((uint32_t)dtype << 12) | ((uint32_t)valid << 13) |
           ((uint32_t)fast << 14) | (rowlen << 15);
}

// Row classes.  FAST: Boolean variable (dataType 0, cardinality 2) whose incidences all have
// arity <= 3 and a tabulable function -- sampled from the truth-table stream by k_gibbs_tt;
// GEN: any other row short enough for one thread; WARP: long rows, one per warp.
#define NB_CLASS_PAIR 0   /* FAST rows whose incidences all have at most one other member: 8-byte records */
#define NB_CLASS_FAST 1
#define NB_CLASS_CAT 2    /* categorical variable (card <= 32), AND_CAT / EQUAL_CAT_CONST factors of arity <= 3 */
#define NB_CLASS_GEN 3
#define NB_CLASS_WARP 4
#define NB_N_CLASSES 5
#define NB_CAT_MAX_CARD 32
// sort key: class:3 | colour:14 | id window:27 | row words:20
#define NB_KEY_CLASS(k) ((int)((k) >> 61))
#define NB_KEY_COLOR(k) ((int)(((k) >> 47) & 0x3FFF))
#define NB_KEY_WINDOW(k) ((int64_t)(((k) >> 20) & ((1ull << 27) - 1)))
#define NB_KEY_GROUP_BITS(k) ((k) >> 47)
#define NB_PAIR_MAX_WID ((1u << 22) - 1)
/* incidences per warp task: two per lane.  A task is a chain of dependent loads per incidence
   (offset -> header -> members -> values); with 1024 incidences a warp walked 32 of them back to
   back (230 us per colour on the KBC hubs, a tenth of the sweep) */
#define NB_WARP_TASK 64

// Variable values on the device.  The element width is a property of the graph, chosen at build
// time (nb_graph::value_bytes): 1 byte when every cardinality is <= 255 (nb_val_t), 2 bytes up to
// 65535 (nb_val16_t).  Kernels that read or write values are instantiated for both.
typedef uint8_t nb_val_t;
typedef uint16_t nb_val16_t;
#define NB_MAX_CARD 255          /* largest cardinality of a 1-byte graph (and of the vmeta card field) */
#define NB_MAX_CARD_WIDE 65535   /* largest cardinality of a 2-byte graph */

// ----------------------------------------------------------------------------
// device graph
// ----------------------------------------------------------------------------
struct NbColorRange {
    int32_t p_beg, p_end;  // PAIR rows [p_beg, p_end) in new ids (p_beg % 32 == 0)
    int32_t f_beg, f_end;  // FAST thread rows [f_beg, f_end) in new ids (f_beg % 32 == 0)
    int32_t c_beg, c_end;  // CAT rows
    int32_t t_beg, t_end;  // GEN thread rows [t_beg, t_end) in new ids (t_beg % 32 == 0)
    int32_t w_beg, w_end;  // warp-path rows, as indices into the warp-row arrays
    int32_t k_beg, k_end;  // their tasks (slices of at most NB_WARP_TASK incidences of one row)
    int64_t edges;         // bucket entries owned by this colour
    int64_t learn_visits_max;  // max over weights of gradient visits in this colour (dataType-0 upper bound)
};

struct nb_graph {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = true;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
#define NB_AUX_STREAMS 4
    cudaStream_t aux[NB_AUX_STREAMS] = {nullptr, nullptr, nullptr, nullptr};   // concurrent row classes of one colour
    cudaEvent_t ev_fork = nullptr, ev_join[NB_AUX_STREAMS] = {nullptr, nullptr, nullptr, nullptr};
    // Bit-packed mirror of the chain-0 values for the member gathers of the record kernels.  On an
    // all-Boolean graph whose value array no longer fits in L2 (200 M variables = 200 MB against
    // 126 MB) every second gather misses and costs a 32-byte DRAM sector for one byte; 1/8 of the
    // size stays resident.  Rebuilt from d_val[0] on entry to nb_gibbs_sweeps, kept current by the
    // kernels; the bytes stay authoritative for everything else.
    uint32_t *d_valbits = nullptr;
    bool bits_eligible = false;      // only PAIR / FAST / WARP rows, every variable Boolean
    bool use_bits = false;           // inside nb_gibbs_sweeps
    bool fan_out = false;             // nb_gibbs_sweeps on a single-GPU graph: run a colour's row classes concurrently

    // sizes
    int64_t V = 0, F = 0, W = 0, NFMAP = 0, NVMAP = 0, NFI = 0;
    int64_t n_edges = 0;        // sum of bucket lengths
    int64_t Vn = 0;             // padded new-id space (thread rows first, then warp rows)
    int64_t n_trows = 0;        // padded thread-row id space [0, n_trows)
    int64_t n_wrows = 0;        // warp rows occupy new ids [n_trows, n_trows + n_wrows)
    int64_t count_entries = 0;
    int n_colors = 0;
    bool wide = false;
    bool has_unknown_func = false;
    int64_t unknown_func_factor = -1;
    int unknown_func_id = 0;
    bool any_categorical = false;
    int max_card = 2;
    int max_arity = 0;
    int64_t jp_rounds = 0;
    int64_t device_bytes = 0;
    int64_t launches = 0;
    uint64_t epoch_counter = 0;
    // No tally exceeds tally_bound = tally_base + max over colours of tally_launches[c]: a variable is
    // tallied at most once per tallying launch of its colour (of its phase on partitioned graphs).
    // tally_base is the largest count installed by nb_set_counts (0 after nb_reset_counts).
    int64_t tally_bound = 0;
    int64_t tally_base = 0;
    std::vector<int64_t> tally_launches;   // [n_colors] tallying launches since the last reset / nb_set_counts
    int warp_row_words = 1024;
    int sigma_shift = 12;

    // ---- raw CSR in original ids (kept for the colouring / rebuilds) ----
    int8_t *d_v_evid = nullptr;      // [V]
    int32_t *d_v_card = nullptr;     // [V]
    int8_t *d_v_dtype = nullptr;     // [V]
    int32_t *d_v_init = nullptr;     // [V]
    int64_t *d_v_vtf = nullptr;      // [V]
    int64_t *d_b_off = nullptr;      // [NVMAP] bucket offset into factor_index
    int32_t *d_b_len = nullptr;      // [NVMAP]
    int32_t *d_fi = nullptr;         // [NFI] factor ids
    uint8_t *d_f_code = nullptr;     // [F]
    int32_t *d_f_wid = nullptr;      // [F]
    double *d_f_feat = nullptr;      // [F]
    int32_t *d_f_arity = nullptr;    // [F]
    int64_t *d_f_off = nullptr;      // [F]
    int32_t *d_m_vid = nullptr;      // [NFMAP]
    int32_t *d_m_eq = nullptr;       // [NFMAP] (only if any_categorical)
    int64_t *d_gid = nullptr;        // [V] global ids or null

    // ---- build intermediates (original ids) ----
    uint32_t *d_rowlen0 = nullptr;   // [V] row words
    uint32_t *d_ninc0 = nullptr;     // [V] incidences
    uint8_t *d_fast0 = nullptr;      // [V] FAST-class flag
    int32_t *d_cbase = nullptr;      // [V] JP colour window
    int32_t *d_cround = nullptr;     // [V] round in which a variable took its colour (natural-order mode)
    int32_t *d_blocker = nullptr;    // [V] the uncoloured higher-priority neighbour seen last (-1: none yet)
    int jp_mode = 0;                 // 0 = hashed priorities, 1 = natural order
    int jp_round_no = 0;
    unsigned long long *d_jpcnt = nullptr;
    uint64_t color_seed = 0;
    bool finalized = false;
    bool deferred = false;

    // ---- ordering ----
    int32_t *d_color = nullptr;      // [V] original ids
    int32_t *d_old2new = nullptr;    // [V]
    int32_t *d_new2old = nullptr;    // [Vn], -1 for padding
    uint32_t *d_rng_id = nullptr;    // [Vn] low 32 bits of the global id (Philox counter)

    // ---- per new-id variable data ----
    uint32_t *d_vmeta = nullptr;     // [Vn] packed meta incl. row length
    void *d_vinit = nullptr;         // [Vn] value_bytes each
    uint16_t *d_vcard = nullptr;     // [Vn] cardinalities of 2-byte graphs (nullptr on 1-byte graphs)
    uint32_t *d_cstart = nullptr;    // [Vn + 1] new-order count layout
    int64_t *d_cstart_old = nullptr; // [V + 1] reference count layout

    // ---- streams ----
    int64_t *d_slice_ptr = nullptr;  // [n_trows/32 + 1] QUAD (16-byte) offsets into d_twords
    uint32_t *d_twords = nullptr;    // SELL-32 thread-path stream: quad q of lane l at quad index ptr + q*32 + l
    int64_t n_twords = 0;
    int64_t n_prows = 0;             // PAIR rows occupy new ids [0, n_prows)
    int64_t *d_tt2_ptr = nullptr;    // [n_prows/32 + 1] quad offsets into d_tt2
    uint4 *d_tt2 = nullptr;          // pair stream: two 8-byte incidences {other, table:9 fixed:1 wid:22} per quad
    uint32_t *d_tt2_common = nullptr; // [n_prows/32] hoisted second word of a uniform slice (4 ids per quad), or NB_PAIR_NONE
    int64_t n_tt2_quads = 0;
    int32_t *d_count_b = nullptr;    // [Vn] tallies of the truth-table kernels (Boolean rows), indexed by new id
    int64_t n_frows = 0;             // PAIR + FAST rows occupy new ids [0, n_frows)
    int64_t n_crows = 0;             // CAT rows occupy new ids [n_frows, n_crows)
    int64_t *d_cat_ptr = nullptr;    // [(n_crows - n_frows)/32 + 1] quad offsets into d_cat
    uint4 *d_cat = nullptr;          // categorical records {other A, other B, k:8 eqA:8 eqB:8 nOthers:2 fixed:1, weight fp32}
    uint32_t *d_cat_wid = nullptr;   // weight id of every categorical record (weight refresh)
    int64_t n_cat_quads = 0;
    int64_t *d_tt_ptr = nullptr;     // [n_frows/32 + 1] quad offsets into d_tt
    uint4 *d_tt = nullptr;           // truth-table stream of the FAST rows (SELL-32, one quad per incidence)
    uint32_t *d_tt_base = nullptr;   // f(self = 0) tables, one word per quad (learning only)
    uint32_t *d_tt_wid = nullptr;    // weight id of every quad (learning + weight refresh; the quads inline the VALUE)
    uint64_t weights_version = 1;    // bumped whenever d_weight changes (nb_set_weights, learning)
    uint64_t tt_weights_version = 0; // version of the weights inlined in d_tt
    int64_t n_tt_quads = 0;
    int64_t *d_wrow_ptr = nullptr;   // [n_wrows + 1] word offsets into d_wwords
    uint32_t *d_wwords = nullptr;    // contiguous warp-path rows
    int64_t n_wwords = 0;
    int64_t *d_inc_ptr = nullptr;    // [n_wrows + 1] offsets into d_inc
    uint2 *d_inc = nullptr;          // per incidence of a warp row: (word offset in row, bucket value)
    int64_t n_inc = 0;
    // long rows are cut into tasks so that one hub variable is spread over many warps
    int32_t *d_wtask_row = nullptr;  // [n_wtasks] warp-row index
    int32_t *d_wtask_beg = nullptr;  // [n_wtasks] first incidence (relative to the row)
    int64_t *d_wtask_ptr = nullptr;  // [n_wrows + 1] tasks of each row
    double *d_wpart = nullptr;       // [n_wtasks][wpart_stride] partial energies
    int64_t n_wtasks = 0;
    int wpart_stride = 4;

    // ---- state ----
    void *d_val[2] = {nullptr, nullptr};  // [Vn] chain 0 = free, 1 = evidence (one allocation, val_stride elements apart)
    size_t val_stride = 0;
    int value_bytes = 1;             // element width of d_val / d_vinit: 1 (nb_val_t) or 2 (nb_val16_t)
    int32_t *d_count = nullptr;      // [count_entries] new-order layout
    double *d_weight = nullptr;      // [W]
    uint8_t *d_wfixed = nullptr;     // [W]

    // ---- learning scratch ----
    long long *d_grad = nullptr;     // [3][W] rotating fixed-point gradient sums by weight id (nb_learn.cu)
    uint32_t *d_nvis = nullptr;      // [3][W] visits (L2) / truncating visits (L1)
    int32_t *d_win_start = nullptr;  // device copy of win_start: the persistent learning kernel finds its cells' rows in it
    unsigned *d_learn_bar = nullptr; // grid barrier state of the persistent learning kernel
    uint8_t *d_long_rows = nullptr;  // [n_colors] truth-table rows of the colour are long: one warp per row

    // scratch for host transfers
    void *d_xfer = nullptr;
    size_t xfer_bytes = 0;
    void *h_pinned = nullptr;
    size_t pinned_bytes = 0;
    std::vector<cudaEvent_t> xfer_events;   // one per download chunk (nb_api.cu)
    void *d_flush = nullptr;
    size_t flush_bytes = 0;

    void *p2p = nullptr;               // NbP2P (nb_p2p.cu)
    bool halo_wait_off = false;        // launches of phases that never read a ghost skip the halo wait
    int64_t n_win = 0;                 // id windows (original id >> sigma_shift)
    std::vector<int32_t> win_start;    // [NB_N_CLASSES * (n_colors + 1)][n_win + 1] first new id of each window per group
    std::vector<uint8_t> learn_long_rows;  // host copy of d_long_rows
    std::vector<int64_t> learn_vmax;   // per colour: max gradient visits of one weight
    int learn_vmax_flag = -1;         // learn_non_evidence the bounds were computed for; -1 = none
    std::vector<uint8_t> h_wfixed;     // host copy of d_wfixed, fetched by the first nb_update_weights_fixed
    std::vector<NbColorRange> colors;
    std::vector<void *> allocs;
};

// the value arrays with their element type (T = nb_val_t on 1-byte graphs, nb_val16_t on 2-byte ones)
template <class T>
inline T *nb_vals(const nb_graph *g, int chain) { return (T *)g->d_val[chain]; }

// device allocation tracked by the graph
int nb_dev_alloc(nb_graph *g, void **p, size_t bytes, bool zero);
template <class T>
inline int nb_alloc(nb_graph *g, T **p, size_t n, bool zero = true)
{
    return nb_dev_alloc(g, (void **)p, n * sizeof(T), zero);
}
int nb_ensure_xfer(nb_graph *g, size_t bytes);
int nb_ensure_pinned(nb_graph *g, size_t bytes);

void nb_p2p_destroy(nb_graph *g);
void nb_p2p_wait_args(nb_graph *g, const volatile uint32_t **flags, const int32_t **neigh, int *n_neigh, uint32_t *phase,
                      int **error);

// build steps (nb_build.cu)
int nb_pack_value_bits(nb_graph *g);
int nb_build_device_graph(nb_graph *g, const nb_graph_desc *desc);
int nb_build_color_round(nb_graph *g, int64_t *remaining);
int nb_build_color_restart(nb_graph *g, int mode);
int nb_natural_round_cap(void);
void nb_release_color_scratch(nb_graph *g);
int nb_build_finalize(nb_graph *g);
int nb_refresh_inlined_weights(nb_graph *g);   // d_tt quads carry fp32 weight values: re-inline after a weight change
int nb_build_color_min_ids(nb_graph *g, int n_colors, int64_t *min_ids);
int nb_build_relabel_colors(nb_graph *g, const int32_t *map, int n);
int nb_learn_color(nb_graph *g, int color, int block, int n_blocks, double step, int regularization, double reg_param,
                   double truncation, int learn_non_evidence, uint64_t seed, uint64_t epoch);
int nb_learn_block_count(nb_graph *g, double step, int learn_non_evidence, int64_t batch_visits, int *n_blocks);
int nb_learn_cell_id_list(nb_graph *g, int color, int block, int n_blocks, int64_t *ids, int64_t *n);

// sweeps (nb_sweep.cu / nb_learn.cu)
int nb_launch_gibbs_color(nb_graph *g, int color, int burnin, int sample_evidence, uint64_t seed,
                          uint64_t epoch);
// NB_ERR_UNSUPPORTED when n_sweeps more tallying sweeps could take a tally past INT32_MAX
int nb_check_tally_room(const nb_graph *g, int burnin, int64_t n_sweeps);
int nb_run_learn(nb_graph *g, int64_t n_epochs, double *stepsize, double decay, int regularization,
                 double reg_param, double truncation, int learn_non_evidence, uint64_t seed,
                 int64_t batch_visits);
int nb_run_potentials(nb_graph *g, int chain, const int64_t *var_ids, int64_t n,
                      const int64_t *out_offsets, double *out, int64_t n_out);
int nb_run_potentials_records(nb_graph *g, int chain, const int64_t *var_ids, int64_t n,
                              const int64_t *out_offsets, double *out, int64_t n_out, int32_t *row_class);
