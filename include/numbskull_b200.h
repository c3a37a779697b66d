/*
 * numbskull_b200.h -- C ABI of the B200-native Gibbs / weight-learning hot path.
 *
 * This is the drop-in boundary (SURVEY.md section 8b).  In the reference the
 * seam is FactorGraph (numbskull/factorgraph.py:27-208): its constructor takes
 * the packed numpy record arrays declared in numbskull/numbskulltypes.py:11-39
 * and its burnIn/inference/learn methods hand those arrays to the numba
 * kernels through run_pool (factorgraph.py:13-24).  Every entry point below
 * replaces one of those hand-offs; the comment above each names the reference
 * lines it stands in for.  All pointers are plain host pointers unless a name
 * says "dev"; no torch / C++ types cross this boundary.
 *
 * Every function returns NB_OK (0) or an NB_ERR_* code; nb_last_error()
 * returns a human-readable message for the calling thread's last failure.
 * There is NO CPU fallback: without a CUDA device nb_graph_create fails with
 * NB_ERR_CUDA.
 */
#ifndef NUMBSKULL_B200_H
#define NUMBSKULL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NB_ABI_VERSION 1

enum {
    NB_OK = 0,
    NB_ERR_INVALID = 1,          /* malformed input (-> ValueError / AssertionError)        */
    NB_ERR_NOT_IMPLEMENTED = 2,  /* unknown factorFunction (inference.py:410-413)           */
    NB_ERR_CUDA = 3,             /* CUDA runtime failure or no device                        */
    NB_ERR_UNSUPPORTED = 4,      /* valid for the reference, outside this build's limits     */
    NB_ERR_NOMEM = 5
};

/* ---- host record layouts: numbskull/numbskulltypes.py:11-39, packed ---- */
#pragma pack(push, 1)
typedef struct { uint8_t isFixed; double initialValue; } nb_weight_rec;              /*  9 B */
typedef struct { int8_t isEvidence; int64_t initialValue; int16_t dataType;
                 int64_t cardinality; int64_t vtf_offset; } nb_variable_rec;          /* 27 B */
typedef struct { int16_t factorFunction; int64_t weightId; double featureValue;
                 int64_t arity; int64_t ftv_offset; } nb_factor_rec;                  /* 34 B */
typedef struct { int64_t vid; int64_t dense_equal_to; } nb_ftv_rec;                   /* 16 B */
typedef struct { int64_t value; int64_t factor_index_offset;
                 int64_t factor_index_length; } nb_vtf_rec;                           /* 24 B */
#pragma pack(pop)

typedef struct nb_graph nb_graph; /* opaque, owns all device memory of one factor graph */

/* What FactorGraph.__init__ receives (factorgraph.py:30-36) plus placement. */
typedef struct {
    const nb_weight_rec *weight;       int64_t n_weight;
    const nb_variable_rec *variable;   int64_t n_variable;
    const nb_factor_rec *factor;       int64_t n_factor;
    const nb_ftv_rec *fmap;            int64_t n_fmap;
    const nb_vtf_rec *vmap;            int64_t n_vmap;
    const int64_t *factor_index;       int64_t n_factor_index;
    int32_t device;                    /* CUDA ordinal                                     */
    uint64_t color_seed;               /* Jones-Plassmann priority seed                    */
    const int64_t *global_vid;         /* NULL, or per-variable global id (partitioned
                                          graphs: priorities and RNG streams are functions
                                          of the GLOBAL id so all ranks agree)             */
    int32_t warp_row_words;            /* rows longer than this go one-per-warp; 0 = default */
    int32_t sigma_shift;               /* SELL sorting window = 2^sigma_shift ids; 0 = default */
    const int32_t *preset_color;       /* NULL, or a valid colouring to adopt (n_variable)  */
    int32_t deferred_coloring;         /* != 0: stop after the upload; the caller drives
                                          nb_color_round (+ ghost colour exchange) and then
                                          nb_graph_finalize -- partitioned graphs             */
} nb_graph_desc;

typedef struct {
    int64_t n_variable, n_factor, n_weight, n_edges; /* n_edges = sum of bucket lengths     */
    int32_t n_colors;
    int32_t wide_headers;              /* 0 = 1-word incidence headers, 1 = 2-word          */
    int64_t n_thread_rows, n_warp_rows;
    int64_t stream_words;              /* 32-bit words in the incidence streams (with pad)  */
    int64_t device_bytes;              /* total device allocation                           */
    int64_t count_entries;             /* == cstart[n_variable]                              */
    int64_t jp_rounds;
    int64_t max_arity;                 /* largest factor arity (the natural-order colouring is only tried when <= 2) */
    int64_t n_pair_rows, n_fast_rows, n_cat_rows;   /* padded id ranges of the record row classes */
    int64_t tt_quads, tt2_quads;       /* 16-byte quads in the FAST / PAIR record streams   */
    int32_t value_bytes;               /* device value width: 1 (every cardinality <= 255) or 2 */
} nb_graph_info;

const char *nb_last_error(void);
int nb_abi_version(void);
int nb_device_count(int *count);

/* ---------------- host-side integer work (bit-exact) ---------------- */

/* numbskull.py:219-227 / :309-317 -- the per-variable Python loop that assigns
 * vtf_offset; returns the number of VarToFactor records through *n_vtf. */
int nb_assign_vtf_offsets(nb_variable_rec *variable, int64_t n_variable, int64_t *n_vtf);

/* dataloading.py:16-81 compute_var_map, in place, same outputs.  Unlike the
 * reference it bounds-checks every index (the reference's factors_to_skip
 * path overruns factor_index; here that returns NB_ERR_INVALID). */
int nb_compute_var_map(nb_variable_rec *variable, int64_t n_variable,
                       const nb_factor_rec *factor, int64_t n_factor,
                       const nb_ftv_rec *fmap, int64_t n_fmap,
                       nb_vtf_rec *vmap, int64_t n_vmap,
                       int64_t *factor_index, int64_t n_factor_index,
                       const uint8_t *domain_mask,
                       const int64_t *factors_to_skip, int64_t n_skip);

/* dataloading.py:103-123 / :126-156 / :159-187 / :190-237 -- big-endian
 * DeepDive binary parsers (graph.weights 17 B/rec, graph.variables 27 B/rec,
 * graph.domains, graph.factors variable-length). */
int nb_load_weights(const uint8_t *data, int64_t n_bytes, int64_t n_weight, nb_weight_rec *out);
int nb_load_variables(const uint8_t *data, int64_t n_bytes, int64_t n_variable,
                      nb_variable_rec *out);
int nb_load_domains(const uint8_t *data, int64_t n_bytes, uint8_t *domain_mask, nb_vtf_rec *vmap,
                    int64_t n_vmap, nb_variable_rec *variable, int64_t n_variable);
int nb_load_factors(const uint8_t *data, int64_t n_bytes, int64_t n_factor, nb_factor_rec *factor,
                    nb_ftv_rec *fmap, int64_t n_fmap, const uint8_t *domain_mask,
                    const nb_variable_rec *variable, int64_t n_variable, const nb_vtf_rec *vmap,
                    int64_t n_vmap);

/* Benchmark input generator: the KBC-style Boolean graph of BASELINE config 4 (SURVEY.md 8d;
 * numbskull_b200/synth.py kbc) written by host threads into caller-allocated record arrays --
 * the role ising/ising.cpp:88-200 plays for the reference.  mix3 = IMPLY / AND / OR factors per
 * variable; n_factor = nvar * (1 + sum mix3), n_fmap = nvar + 3 n_imp + 2 n_and + 3 n_or. */
int nb_synth_kbc(int64_t nvar, uint64_t seed, int64_t n_weights, double evidence_frac, int64_t window,
                 double far_frac, double hub_frac, double fixed_frac, const double *mix3,
                 nb_weight_rec *weight, nb_variable_rec *variable, nb_factor_rec *factor, int64_t n_factor,
                 nb_ftv_rec *fmap, int64_t n_fmap);
/* The same graph piecewise, for partitioned runs that never hold the whole graph: the weight table,
 * the variable records of listed global ids (NULL: 0 .. n-1), and the factors that touch the owner
 * block [lo, hi) in increasing global factor id with GLOBAL member ids (factor == NULL: only size the
 * arrays through *n_factor / *n_fmap). */
int nb_synth_kbc_weights(uint64_t seed, int64_t n_weights, double fixed_frac, nb_weight_rec *weight);
int nb_synth_kbc_variables(uint64_t seed, double evidence_frac, const int64_t *gids, int64_t n,
                           nb_variable_rec *variable);
int nb_synth_kbc_block(int64_t nvar, uint64_t seed, int64_t n_weights, int64_t window, double far_frac,
                       double hub_frac, const double *mix3, int64_t lo, int64_t hi, nb_factor_rec *factor,
                       int64_t *n_factor, nb_ftv_rec *fmap, int64_t *n_fmap);

/* Owner-block partitions (partition.extract_local, the role of the reference's per-minion graph
 * views, salt/src/messages.py:175-179): the ghost variables of block [lo, hi) in ascending global
 * id, and (rewrite != 0) fmap[].vid translated to local ids (owned v -> v - lo, ghost -> n_owned +
 * rank).  Two calls: ghosts == NULL returns the count. */
int nb_block_ghosts(nb_ftv_rec *fmap, int64_t n_fmap, int64_t nvar, int64_t lo, int64_t hi, int64_t *ghosts,
                    int64_t *n_ghosts, int rewrite);

/* The same for an arbitrary placement owner[v] (partition.extract_local_by_owner: an imported
 * partition -- salt/src/messages.py:175-179 -- or a locality-aware one): the factors with a member
 * owned by `rank` (order kept, ftv_offset renumbered), their members as local ids (owned first,
 * ghosts after, both in ascending global id) and global_vid[n_owned + n_ghost].  Two calls:
 * loc_factor == NULL returns the four counts. */
int nb_extract_local(const nb_factor_rec *factor, int64_t n_factor, const nb_ftv_rec *fmap, int64_t n_fmap,
                     const int32_t *owner, int64_t nvar, int32_t rank, int64_t *n_loc_factor, int64_t *n_loc_fmap,
                     int64_t *n_owned, int64_t *n_ghost, nb_factor_rec *loc_factor, nb_ftv_rec *loc_fmap,
                     int64_t *global_vid);

/* -------------------------- graph lifecycle -------------------------- */

/* FactorGraph.__init__ (factorgraph.py:30-73): builds the device-resident
 * SoA/CSR form, colours the variable conflict graph (Jones-Plassmann on the
 * GPU), reorders variables by (colour, row length) and lays the per-variable
 * incidence streams out in HBM.  State starts as the reference's: var_value =
 * var_value_evid = initialValue, weight_value = weight.initialValue, count = 0. */
int nb_graph_create(const nb_graph_desc *desc, nb_graph **out);
void nb_graph_destroy(nb_graph *g);          /* FactorGraph.clear (factorgraph.py:75-78) */
int nb_graph_get_info(const nb_graph *g, nb_graph_info *info);

/* Colour of every variable in ORIGINAL id order (-1 = not owned, isEvidence==4).
 * Parity hook for "no two same-colour variables share a factor". */
int nb_graph_get_colors(const nb_graph *g, int32_t *colors);
/* Device-side validity check of the colouring in use: number of ordered pairs of
 * owned variables that share a factor AND a colour (0 for a valid colouring). */
int nb_graph_check_coloring(nb_graph *g, int64_t *conflicts);
/* Bucket entries (factor-edge evaluations per sweep) owned by each colour; n_colors entries. */
int nb_graph_color_edges(const nb_graph *g, int64_t *edges_per_color);

/* ------------------- state exchange at call boundaries ------------------- */
/* The arrays are the reference's public ones (factorgraph.py:46-52):
 * chain 0 = var_value[var_copy], chain 1 = var_value_evid[var_copy] (int64, original
 * variable order); weight_value[weight_copy] (float64); count (int64, cstart layout). */
int nb_set_var_values(nb_graph *g, int chain, const int64_t *values);
int nb_get_var_values(nb_graph *g, int chain, int64_t *values);
int nb_set_weights(nb_graph *g, const double *weights);
int nb_get_weights(nb_graph *g, double *weights);
/* device-to-device copies of the weight table on the graph's stream (multi-GPU learning: the
 * per-epoch weight-delta all-reduce, numbskull_master.py:223-224, never touches the host) */
int nb_get_weights_dev(nb_graph *g, double *dev_weights);
int nb_set_weights_dev(nb_graph *g, const double *dev_weights);
int nb_reset_counts(nb_graph *g);
/* accumulate != 0: counts[i] += device tally (the reference's count is cumulative,
 * factorgraph.py:172-173); else counts[i] = device tally. */
int nb_get_counts(nb_graph *g, int64_t *counts, int accumulate);
/* Same, and in the same host pass marginals[i] = counts[i] / epochs (factorgraph.py:172-173). */
int nb_get_counts_marginals(nb_graph *g, int64_t *counts, int accumulate, double *marginals, double epochs);

/* marginals[i] = device tally / epochs without materialising the int64 count array
 * (factorgraph.py:172-173 when the caller only reads `marginals`). */
int nb_get_marginals(nb_graph *g, double *marginals, double epochs);
/* The device tallies in the reference's cstart layout at their natural width: *elem_bytes = 1, 2 or 4
 * (no tally exceeds the number of tallying sweeps since the last reset); `out` should be pinned
 * (nb_host_alloc) -- no host-side conversion at all. */
int nb_get_counts_compact(nb_graph *g, void *out, int64_t out_bytes, int32_t *elem_bytes);
/* Install `counts` (int64, cstart layout) as the device tallies: callers that edit `count` between
 * calls.  The device tallies are CUMULATIVE like the reference's count array (factorgraph.py:30-31
 * is never re-zeroed by inference()); nb_reset_counts zeroes them (FactorGraph.clear). */
int nb_set_counts(nb_graph *g, const int64_t *counts);
/* page-locked host memory for result arrays the library fills by DMA */
int nb_host_alloc(void **ptr, int64_t bytes);
int nb_host_free(void *ptr);

/* ------------------------------ hot path ------------------------------ */

/* inference.py:55-71 potential(), for parity tests: energies of every value of
 * the listed variables under the current state of `chain`; variable var_ids[i]
 * writes cardinality entries starting at out[out_offsets[i]]. */
int nb_potentials(nb_graph *g, int chain, const int64_t *var_ids, int64_t n,
                  const int64_t *out_offsets, double *out, int64_t n_out);

/* The same energies as the RECORD kernels compute them.  Boolean variables of the PAIR / FAST row
 * classes (sampled by k_gibbs_tt2 / k_gibbs_tt from 8- and 16-byte truth-table records) write
 * {0, potential(v,1) - potential(v,0)}; categorical variables of the CAT class (k_gibbs_cat) write
 * their fp32 per-value energies; variables of the generic classes write nothing.  row_class[i]
 * receives the class of var_ids[i] (0 PAIR, 1 FAST, 2 CAT, 3 GEN, 4 WARP).  The device code is the
 * very function each sweep kernel calls, so this pins the hot kernels to inference.py:55-71. */
int nb_potentials_records(nb_graph *g, int chain, const int64_t *var_ids, int64_t n,
                          const int64_t *out_offsets, double *out, int64_t n_out, int32_t *row_class);

/* run_pool(gibbsthread) x n_epochs (factorgraph.py:135-141 burnIn with
 * burnin != 0, :156-163 inference with burnin == 0): one chromatic Gibbs sweep
 * per epoch, one kernel launch per colour and row class.  Tallies into the
 * device count unless burnin.  `seed` keys the Philox streams. */
int nb_gibbs_sweeps(nb_graph *g, int64_t n_epochs, int burnin, int sample_evidence,
                    uint64_t seed);

/* run_pool(learnthread) x n_epochs with stepsize *= decay after each
 * (factorgraph.py:188-206); *stepsize is updated to the final value.
 * Both chains are sampled in one sweep; gradients are reduced by weight id
 * and applied once per mini-batch (a block of consecutive variable ids holding
 * at most `batch_visits` visits of any weight; 0 = default policy 0.25 / stepsize,
 * see DESIGN.md "learning"). */
int nb_learn_sweeps(nb_graph *g, int64_t n_epochs, double *stepsize, double decay,
                    int regularization, double reg_param, double truncation,
                    int learn_non_evidence, uint64_t seed, int64_t batch_visits);

/* ------------------------- measurement helpers ------------------------- */
/* CUDA-event timer on the stream the sweeps are launched on. */
int nb_timer_start(nb_graph *g);
int nb_timer_stop(nb_graph *g, float *milliseconds);
int nb_synchronize(nb_graph *g);
/* Number of kernel launches issued by this graph's sweeps so far. */
int nb_launch_count(const nb_graph *g, int64_t *launches);
/* Write `bytes` of device memory to evict L2 between timed iterations. */
int nb_flush_l2(nb_graph *g, int64_t bytes);

/* --------------------- partitioned (multi-GPU) graphs --------------------- */
/* Owner-computes partitioning (salt/src/numbskull_master.py:343,
 * numbskull_minion.py:185): non-owned members are local variables with
 * isEvidence == 4.  After each colour the owner's fresh values are shipped to
 * the ranks that hold them as ghosts (messages.py:1308-1319).  These calls
 * expose one colour phase at a time plus gather/scatter by local variable id
 * on DEVICE buffers so the host layer can put NCCL between them. */
int nb_gibbs_color_phase(nb_graph *g, int color, int burnin, int sample_evidence,
                         uint64_t seed, int64_t epoch);
/* values of `local_ids` (device int32, ORIGINAL local ids) of `chain` -> dev_out (uint8) */
int nb_gather_values_dev(nb_graph *g, int chain, const int32_t *dev_local_ids, int64_t n,
                         uint8_t *dev_out);
int nb_scatter_values_dev(nb_graph *g, int chain, const int32_t *dev_local_ids, int64_t n,
                          const uint8_t *dev_in);
/* Learning walks the graph in `n_blocks` blocks of consecutive variable ids (mini-batches) and,
 * inside a block, colour by colour.  nb_learn_blocks gives the block count the library would use
 * for this step size (partitioned graphs: take the MAX over ranks).  nb_learn_color_phase runs one
 * (block, colour) cell: both chains, gradient reduction by weight id, weight update; the caller
 * exchanges both chains' boundary values afterwards. */
int nb_learn_blocks(nb_graph *g, double stepsize, int learn_non_evidence, int64_t batch_visits, int *n_blocks);
int nb_learn_color_phase(nb_graph *g, int color, int block, int n_blocks, double stepsize, int regularization,
                         double reg_param, double truncation, int learn_non_evidence, uint64_t seed, int64_t epoch);
/* Parity hook: the ORIGINAL ids of the variables cell (block, colour) holds (`ids` has room for
 * n_variable entries; *n receives the count) -- which variables nb_learn_color_phase samples. */
int nb_learn_cell_ids(nb_graph *g, int color, int block, int n_blocks, int64_t *ids, int64_t *n);
/* Distributed Jones-Plassmann (graphs created with deferred_coloring): one round over the
 * owned, still uncoloured variables; ghosts are consulted through the colours last scattered
 * in.  *remaining != 0 iff an owned variable is still uncoloured after the round. */
int nb_color_round(nb_graph *g, int64_t *remaining);
/* (Re)start the colouring of a deferred graph: mode 0 = hashed priorities, 1 = natural order (the
 * smaller global id first; rounds are counted exactly, a colour taken in a round becomes visible in
 * the next).  The library's own policy, which partition.py reproduces across the ranks: hashed
 * first; if that needs more than 2 colours, natural order for at most nb_color_natural_round_cap()
 * rounds; keep the natural colouring only if it finished and uses fewer colours. */
int nb_color_restart(nb_graph *g, int mode);
int nb_color_natural_round_cap(void);
int nb_gather_colors_dev(nb_graph *g, const int32_t *dev_local_ids, int64_t n, int32_t *dev_out);
int nb_scatter_colors_dev(nb_graph *g, const int32_t *dev_local_ids, int64_t n, const int32_t *dev_in);
/* Colour order = visiting order.  Single-GPU graphs are relabelled so that colours are visited in
 * increasing order of the smallest variable id they contain (the chromatic analogue of the
 * reference's ascending-id scan); partitioned graphs do the same globally: min_ids[c] = smallest
 * GLOBAL id among this rank's owned variables of colour c (INT64_MAX if none), reduced with MIN
 * over the ranks by the caller, who then installs the permutation map[old colour] = new colour. */
int nb_color_min_ids(nb_graph *g, int n_colors, int64_t *min_ids);
int nb_relabel_colors(nb_graph *g, const int32_t *map, int n);
/* Orders the variables and lays out the streams once every variable has its colour. */
int nb_graph_finalize(nb_graph *g);
/* Peer-to-peer halo exchange (ranks = processes on one NVLink node).  Each rank exports CUDA-IPC
 * handles of its two value arrays and of a flag array (3 x 64 bytes), opens its neighbours',
 * and installs a plan: per colour, (owned local variable, peer rank, slot in the peer's value
 * array).  nb_p2p_exchange then pushes the colour's boundary values with NVLink peer stores and
 * runs a flag barrier with the neighbours in the same kernel -- no NCCL, no pack / unpack. */
int nb_p2p_export(nb_graph *g, int world, int rank, uint8_t *handles_3x64);
int nb_p2p_open(nb_graph *g, const uint8_t *handles_world_x3x64, const int32_t *neighbours, int n_neighbours);
int nb_p2p_local_slots(nb_graph *g, const int32_t *local_ids, int64_t n, int32_t *slots);
int nb_p2p_set_plan(nb_graph *g, int n_colors, const int64_t *color_ptr, const int32_t *src_local,
                    const int32_t *peer, const int32_t *dst_slot);
#define NB_P2P_NOWAIT 16 /* or-ed into chain_mask: signal only; the next sweep kernels wait in their prologue */
int nb_p2p_exchange(nb_graph *g, int color, int chain_mask);
int nb_p2p_wait(nb_graph *g);   /* block the stream until every neighbour reached the latest phase */
/* nb_gibbs_sweeps for a partitioned graph: per colour the sweep kernels and the halo push, launched
 * back to back from C (n_colors = the GLOBAL phase count).  mode bit 0: split-phase exchange
 * (NB_P2P_NOWAIT); bit 1: the colours were split with nb_split_colors -- the boundary phase 2c and
 * its push run on a high-priority side stream concurrently with the interior phase 2c + 1, so the
 * exchange is off the critical path. */
int nb_gibbs_sweeps_p2p(nb_graph *g, int64_t n_epochs, int burnin, int sample_evidence, uint64_t seed,
                        int n_colors, int mode);
/* Before nb_graph_finalize of a deferred graph: colour c becomes the phases 2c (ghosts and
 * `boundary_ids`, the owned variables other ranks hold copies of) and 2c + 1 (interior variables,
 * which never read a ghost).  Every rank must split (or none). */
int nb_split_colors(nb_graph *g, const int32_t *boundary_ids, int64_t n);
int nb_p2p_check(nb_graph *g);
/* unmap the peers' arrays; call on every rank, synchronise the ranks, then nb_graph_destroy */
int nb_p2p_close(nb_graph *g);
/* run the sweeps on a caller-owned CUDA stream (cudaStream_t as void*) */
int nb_set_stream(nb_graph *g, void *cuda_stream);
int nb_begin_epoch(nb_graph *g, int64_t *epoch); /* returns and advances the sweep counter */

#ifdef __cplusplus
}
#endif
#endif /* NUMBSKULL_B200_H */
