/*
 * sbn_b200.h -- C ABI of libsbn_b200.so: the B200-native replacement for the
 * BEAGLE-backed likelihood engine of phylovi/libsbn.
 *
 * Plain C, plain pointers and sizes; every pointer argument is HOST memory,
 * borrowed for the duration of the call (same ownership rule as the BEAGLE
 * calls it replaces).  All functions return 0 on success and a negative
 * SBNB_ERR_* code on failure; sbnb_last_error() returns a thread-local message
 * that the C++ glue turns into Failwith -> std::runtime_error -> Python
 * RuntimeError (reference src/sugar.hpp:67-78).  There is NO CPU fallback: if
 * no CUDA device is usable every entry point fails with SBNB_ERR_NO_DEVICE.
 *
 * The entry points mirror, one to one, the five batch methods of the
 * reference's `Engine` (src/engine.hpp:33-47, bodies src/engine.cpp:54-93),
 * which is the only caller of FatBeagle and therefore of BEAGLE.
 *
 * Conventions (identical to the reference's host objects):
 *  - taxa are numbered 0..n-1; node ids follow Node::Polish
 *    (src/node.cpp:341-357): leaves first, internal nodes in post-order, root
 *    last; a topology is its Node::ParentIdVector (src/node.cpp:413-424);
 *  - an unrooted tree has a trifurcating root and 2n-2 nodes; it is
 *    detrifurcated exactly as UnrootedTree::Detrifurcate does
 *    (src/unrooted_tree.cpp:27-37), so per-branch outputs have 2n-1 entries;
 *  - branch_lengths are indexed by node id (src/tree.hpp:54-55);
 *  - phylo-model parameters are one row per tree laid out by the reference's
 *    BlockSpecification: substitution block, then site block, then clock block
 *    (src/phylo_model.cpp:11-13); see sbnb_engine_param_block().
 */
#ifndef SBN_B200_H_
#define SBN_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum {
  SBNB_OK = 0,
  SBNB_ERR_INVALID_ARGUMENT = -1, /* bad sizes, malformed topology, unknown model */
  SBNB_ERR_NO_DEVICE = -2,        /* no usable CUDA device: there is no CPU path */
  SBNB_ERR_CUDA = -3,             /* a CUDA runtime call or kernel failed */
  SBNB_ERR_OUT_OF_MEMORY = -4,
  SBNB_ERR_MODEL = -5             /* parameter sanity failure (substitution_model.cpp:21-35) */
};

typedef struct sbnb_engine sbnb_engine; /* replaces Engine + its FatBeagles (engine.hpp:26-53) */
typedef struct sbnb_batch sbnb_batch;   /* one staged tree collection, device resident */

/* Thread-local description of the last failure on the calling thread. */
const char* sbnb_last_error(void);

/* Number of CUDA devices visible; <= 0 means the library cannot run. */
int sbnb_device_count(void);

/*
 * Replaces Engine::Engine (engine.cpp:10-46) + FatBeagle::FatBeagle
 * (fat_beagle.cpp:13-29): model specification strings as in
 * PhyloModelSpecification (phylo_model.hpp:13-17):
 *   substitution: "JC69" | "GTR" | "HKY"  (HKY is an addition; see DESIGN.md)
 *   site:         "constant" | "weibull+K" | "weibull" (K=4) | "gamma+K" | "gamma", each
 *                 optionally followed by "+I": a proportion p of invariable sites,
 *                 lik = (1 - p) L(rates / (1 - p)) + p I with I the summed frequencies of
 *                 the states every tip of the pattern allows (DESIGN.md, K2); p is the
 *                 last entry of the "entire site" block ("proportion invariant"), and any p
 *                 outside [0, 1) fails with SBNB_ERR_MODEL
 *   clock:        "none" | "strict"
 * tip_states is SitePattern::GetPatterns() flattened [taxon][pattern]
 * (site_pattern.hpp:46-50): 0..3 = A,C,G,T, anything >= 4 = gap/unknown.
 * pattern_weights is SitePattern::GetWeights().
 * device = CUDA ordinal.
 */
int sbnb_engine_create(const char* substitution, const char* site, const char* clock,
                       int32_t taxon_count, int64_t pattern_count, const uint8_t* tip_states,
                       const double* pattern_weights, int32_t device, sbnb_engine** out);
void sbnb_engine_destroy(sbnb_engine* engine);

/*
 * How the bytes of an alignment ([taxon][pattern]) encode its tips.
 *   SBNB_TIPS_STATES            0..3 = A,C,G,T, anything >= 4 = gap/unknown (the
 *                               reference's symbol table: degenerate nucleotides are gaps).
 *   SBNB_TIPS_NUCLEOTIDE_MASKS  the set of states a character allows: bit 0 = A, bit 1 = C,
 *                               bit 2 = G, bit 3 = T; 15 = missing (N X ? -), R = A|G = 5 and
 *                               so on.  A tip then enters the likelihood as the partial
 *                               vector of its bits (BEAGLE's tip partials).  0 and values
 *                               above 15 are refused with SBNB_ERR_INVALID_ARGUMENT.
 * An alignment of masks without a two- or three-state mask gives results bitwise identical
 * to the same alignment as states.
 */
enum { SBNB_TIPS_STATES = 0, SBNB_TIPS_NUCLEOTIDE_MASKS = 1 };
/* sbnb_engine_create with the tips in the given encoding (sbnb_engine_create is the
 * SBNB_TIPS_STATES case). */
int sbnb_engine_create_encoded(const char* substitution, const char* site, const char* clock,
                               int32_t taxon_count, int64_t pattern_count, const uint8_t* tips,
                               int32_t tip_encoding, const double* pattern_weights, int32_t device,
                               sbnb_engine** out);

/*
 * A device group: one engine over several GPUs of the box, replacing the
 * reference's thread_count FatBeagle instances and the thread pool that fans a
 * collection over them (engine.cpp:17-27, fat_beagle.hpp:119-149) -- one host thread
 * and one stream per device inside the library.  `devices` lists CUDA ordinals
 * (an ordinal may repeat).  shard_axis:
 *   SBNB_SHARD_TREES     every device evaluates a contiguous slice of the collection
 *                        (trees are independent; no exchange step);
 *   SBNB_SHARD_PATTERNS  every device walks all trees over its range of site patterns
 *                        and the raw per-tree sums are added across devices over
 *                        NVLink peer memory before one host finishing (for a tree
 *                        whose partials one device should not hold alone).
 * A group offers the one-call entry points (sbnb_log_likelihoods_*, sbnb_gradients_*);
 * the staged entry points below work on single-device engines.
 */
enum { SBNB_SHARD_TREES = 0, SBNB_SHARD_PATTERNS = 1 };
int sbnb_engine_create_multi(const char* substitution, const char* site, const char* clock,
                             int32_t taxon_count, int64_t pattern_count, const uint8_t* tip_states,
                             const double* pattern_weights, const int32_t* devices,
                             int32_t device_count, int32_t shard_axis, sbnb_engine** out);
/* sbnb_engine_create_multi with the tips in the given encoding (see sbnb_engine_create_encoded). */
int sbnb_engine_create_multi_encoded(const char* substitution, const char* site, const char* clock,
                                     int32_t taxon_count, int64_t pattern_count, const uint8_t* tips,
                                     int32_t tip_encoding, const double* pattern_weights,
                                     const int32_t* devices, int32_t device_count, int32_t shard_axis,
                                     sbnb_engine** out);
/*
 * How the "substitution_model" block of a gradient call (GTR: 8 entries, HKY: 4) is
 * computed.  The reference takes central differences of 16 full log-likelihood
 * evaluations per tree (fat_beagle.cpp:400-465, delta 1e-6 in stick-breaking
 * coordinates); SBNB_SUBSTITUTION_ANALYTIC (the default; or SBNB_SUBSTITUTION_GRADIENT=fd
 * in the environment for the other) computes the exact derivative inside the gradient
 * sweep: with P = V exp(Lambda tau) V^-1, dP/dtheta = V [(V^-1 dQ/dtheta V) o Phi(tau)] V^-1,
 * so the sweep only accumulates W_kl = sum of w/lik (V^T T)_k (V^-1 L)_l Phi_kl over edges,
 * categories and patterns (16 numbers per tree) and the host contracts them with
 * V^-1 dQ/dtheta V.  It differs from the reference's values by their O(delta^2)
 * truncation and O(eps/delta) rounding error.  SBNB_SUBSTITUTION_FINITE_DIFFERENCES
 * reproduces the reference's arithmetic.
 */
enum { SBNB_SUBSTITUTION_ANALYTIC = 0, SBNB_SUBSTITUTION_FINITE_DIFFERENCES = 1 };
int sbnb_engine_set_substitution_gradient(sbnb_engine* engine, int32_t mode);
/* Number of devices behind an engine (1 unless created with sbnb_engine_create_multi). */
int32_t sbnb_engine_device_count(const sbnb_engine* engine);

/* Engine::GetPhyloModelBlockSpecification (engine.hpp:31): total parameter
 * count K of one row, and (start, length) of a named block such as
 * "GTR rates", "frequencies", "kappa", "Weibull shape", "Gamma shape", "proportion invariant",
 * "clock rate", "entire substitution", "entire site", "entire clock".  Unknown key -> error. */
int32_t sbnb_engine_param_count(const sbnb_engine* engine);
int sbnb_engine_param_block(const sbnb_engine* engine, const char* key, int32_t* start,
                            int32_t* length);
int32_t sbnb_engine_category_count(const sbnb_engine* engine);

/* A tree collection in flat form. */
typedef struct {
  int32_t tree_count;
  int32_t node_count;           /* per tree: 2n-2 (trifurcating root) or 2n-1 (bifurcating) */
  const int32_t* parent_ids;    /* [tree_count][node_count-1]  Node::ParentIdVector */
  const double* branch_lengths; /* [tree_count][node_count]    Tree::branch_lengths_ */
  /* Rooted time trees only (RootedTree, rooted_tree.hpp); NULL otherwise. */
  const double* rates;         /* [tree_count][node_count-1]  RootedTree::rates_ */
  const double* node_heights;  /* [tree_count][node_count] */
  const double* node_bounds;   /* [tree_count][node_count] */
  const double* height_ratios; /* [tree_count][taxon_count-1] */
  int32_t rate_count;          /* 1 = strict clock, node_count-1 = one rate per branch */
} sbnb_tree_batch;

/* Per-tree results of a gradient call = the reference's PhyloGradient
 * (tree_gradient.hpp:10-19).  Any pointer may be NULL (that block is skipped);
 * blocks that the model does not define are left untouched. */
typedef struct {
  double* log_likelihood;     /* [T]                                            */
  double* branch_lengths;     /* [T][2n-1]   "branch_lengths"  (unrooted only)  */
  double* substitution_model; /* [T][8]      "substitution_model" (GTR; HKY: 4) */
  double* site_model;         /* [T][site entries] "site_model": the shape (categories > 1), then
                                 d/d proportion invariant (+I); 1 entry for every model without +I */
  double* ratios_root_height; /* [T][n-1]    "ratios_root_height" (rooted only) */
  double* clock_model;        /* [T][rate_count] "clock_model"    (rooted only) */
} sbnb_gradient_out;

/* ---- one-call entry points: what engine.cpp's five methods become --------- */

/* Engine::LogLikelihoods(UnrootedTreeCollection) (engine.cpp:54-60). */
int sbnb_log_likelihoods_unrooted(sbnb_engine* engine, const sbnb_tree_batch* trees,
                                  const double* params, int32_t rescaling,
                                  double* out_log_likelihoods);
/* Engine::LogLikelihoods(RootedTreeCollection) (engine.cpp:62-68): branch
 * lengths times rates, plus the log-determinant Jacobian (fat_beagle.cpp:82-104). */
int sbnb_log_likelihoods_rooted(sbnb_engine* engine, const sbnb_tree_batch* trees,
                                const double* params, int32_t rescaling,
                                double* out_log_likelihoods);
/* Engine::UnrootedLogLikelihoods(RootedTreeCollection) (engine.cpp:70-76). */
int sbnb_unrooted_log_likelihoods_of_rooted(sbnb_engine* engine, const sbnb_tree_batch* trees,
                                            const double* params, int32_t rescaling,
                                            double* out_log_likelihoods);
/*
 * Site log-likelihoods: for tree t and site pattern k of the engine's pattern range,
 * out_site[t][k] is the log site likelihood the walk adds into logL_t with weight w_k --
 * log(site likelihood) + (power-of-two exponent) ln 2 with rescaling, log((1 - p) L_k + p I_k)
 * with +I -- unweighted, so that sum_k w_k out_site[t][k] = logL_t up to summation order.
 * A pattern of weight 0 gets its value too; an unrescaled site that underflows gives -inf, as
 * its term in the sum would.  out_log_likelihoods ([T], or NULL) is bitwise what
 * sbnb_log_likelihoods_unrooted / _rooted return for the same input.  Rooted trees: the
 * values are for the branch lengths times the rates and exclude the log-det Jacobian, so
 * sum_k w_k out_site[t][k] = logL_t - logdetJ_t (sbnb_finish_log_likelihoods_rooted applied
 * to zeros gives logdetJ_t).  A device group fills the whole [T][pattern_count] matrix on
 * either shard axis.  For RELL / KH / SH / AU topology tests and PSIS-LOO / WAIC.
 */
int sbnb_site_log_likelihoods_unrooted(sbnb_engine* engine, const sbnb_tree_batch* trees,
                                       const double* params, int32_t rescaling,
                                       double* out_log_likelihoods, double* out_site);
int sbnb_site_log_likelihoods_rooted(sbnb_engine* engine, const sbnb_tree_batch* trees,
                                     const double* params, int32_t rescaling,
                                     double* out_log_likelihoods, double* out_site);
/* Engine::Gradients(UnrootedTreeCollection) (engine.cpp:78-84). */
int sbnb_gradients_unrooted(sbnb_engine* engine, const sbnb_tree_batch* trees,
                            const double* params, int32_t rescaling,
                            const sbnb_gradient_out* out);
/* Engine::Gradients(RootedTreeCollection) (engine.cpp:86-93). */
int sbnb_gradients_rooted(sbnb_engine* engine, const sbnb_tree_batch* trees,
                          const double* params, int32_t rescaling, const sbnb_gradient_out* out);

/* ---- staged entry points (same work split at the PCIe boundary) ----------- */

enum {
  SBNB_MODE_LOG_LIKELIHOOD = 0, /* post-order sweep + root reduction              */
  SBNB_MODE_BRANCH_GRADIENT = 1 /* + pre-order sweep + all 2n-2 edge derivatives  */
};

enum {
  SBNB_STAGE_ROOTED = 1,          /* RootedTree semantics: branch lengths scaled by rates */
  SBNB_STAGE_SUBSTITUTION_FD = 2, /* also stage the 2 x (5+3) perturbed models of the
                                     finite-difference substitution gradient
                                     (fat_beagle.cpp:400-465) as extra logL-only evaluations */
  SBNB_STAGE_SUBSTITUTION_ANALYTIC = 4, /* gradient runs also accumulate the 20 sums per tree of
                                     the analytic substitution gradient (see
                                     sbnb_engine_set_substitution_gradient); fetched with
                                     sbnb_batch_fetch_substitution_sums, they follow the rate
                                     gradients in the device result array */
  SBNB_STAGE_SITE_LOG_LIKELIHOODS = 8 /* log-likelihood runs also write the [T][P] site
                                     log-likelihoods (P = the engine's pattern range when
                                     staged; T x P doubles of device memory, allocated only
                                     with this flag); fetched with
                                     sbnb_batch_fetch_site_log_likelihoods */
};

/* Builds the per-tree traversal programs and eigen-systems on the host and
 * stages them in device memory. */
int sbnb_batch_stage(sbnb_engine* engine, const sbnb_tree_batch* trees, const double* params,
                     int32_t stage_flags, sbnb_batch** out);
/* Enqueues every kernel of one pass over the staged batch on the engine's
 * stream; does not copy or synchronise.  Results stay in device memory. */
int sbnb_batch_run(sbnb_engine* engine, sbnb_batch* batch, int32_t mode, int32_t rescaling);
/* Waits for the stream and copies results to the host: log_likelihoods
 * [sbnb_batch_evaluation_count()] = the T trees first, then (gradient runs of a
 * batch staged with SBNB_STAGE_SUBSTITUTION_FD) [T][2*coords] plus/minus
 * evaluations; if the last run was a gradient run, branch_gradients [T][2n-1]
 * (raw edge derivatives, before the fixed-node zeroing) and, when categories
 * > 1, rate_gradients [T][2n-1] (the same with d rate_c / d shape as scalers).
 * NULL pointers are skipped. */
int sbnb_batch_fetch(sbnb_engine* engine, sbnb_batch* batch, double* log_likelihoods,
                     double* branch_gradients, double* rate_gradients);
/* The analytic substitution-gradient sums of the last gradient run of a batch staged with
 * SBNB_STAGE_SUBSTITUTION_ANALYTIC: [T][20] = W (16, row-major) then R (4).  Sums over site
 * patterns: ranks that each hold a pattern range add them like the other raw results. */
int sbnb_batch_fetch_substitution_sums(sbnb_engine* engine, sbnb_batch* batch, double* sums);
/* The sums of the invariant class of the last gradient run of a +I model: [T][5] = D, then
 * E_A..E_T (DESIGN.md, K2; E only in batches staged with SBNB_STAGE_SUBSTITUTION_ANALYTIC, else 0).
 * Sums over site patterns: ranks that each hold a pattern range add them like the other raw
 * results (on the device they follow the substitution sums in the result array). */
int sbnb_batch_fetch_invariant_sums(sbnb_engine* engine, sbnb_batch* batch, double* sums);
/* The [T][P] site log-likelihoods (see sbnb_site_log_likelihoods_unrooted) of the last run of
 * a batch staged with SBNB_STAGE_SITE_LOG_LIKELIHOODS, P = the width of the pattern range it was
 * staged on (which a run requires unchanged).  SBNB_ERR_INVALID_ARGUMENT if the batch was staged
 * without the flag, has not been run, or was last run in gradient mode (gradient runs do not
 * write them). */
int sbnb_batch_fetch_site_log_likelihoods(sbnb_engine* engine, sbnb_batch* batch, double* out);
/* Device addresses of the raw result arrays sbnb_batch_fetch copies out
 * (fp64: [evaluation_count], [T][2n-1], [T][2n-1]), valid until the batch is
 * destroyed.  For site-pattern sharding: the ranks sum-all-reduce these in
 * place (NCCL, on the engine's stream, after sbnb_batch_run) and then fetch. */
int sbnb_batch_device_results(sbnb_batch* batch, void** log_likelihoods, void** branch_gradients,
                              void** rate_gradients);
void sbnb_batch_destroy(sbnb_engine* engine, sbnb_batch* batch);
int32_t sbnb_batch_evaluation_count(const sbnb_batch* batch);

/* Stream plumbing: the cudaStream_t (as void*) the engine launches on, so a
 * caller can bracket sbnb_batch_run with its own CUDA events; number of kernel
 * launches issued by this engine so far; algorithmic bytes of the last run
 * (SURVEY.md 8d model: (2n-2) U per logL, (10n-14) U per gradient, U = 32 C P). */
void* sbnb_engine_stream(sbnb_engine* engine);
int64_t sbnb_engine_launch_count(const sbnb_engine* engine);
double sbnb_batch_algorithmic_bytes(const sbnb_batch* batch, int32_t mode);
/* Cumulative bytes this engine has copied host->device and device->host
 * (staging goes through a page-locked arena, so these are DMA transfers). */
int sbnb_engine_transfer_bytes(const sbnb_engine* engine, int64_t* host_to_device,
                               int64_t* device_to_host);
/* Device time of the tree-walk kernel (the dominant kernel), measured with
 * CUDA events on the engine's stream around each launch made by
 * sbnb_batch_run: cumulative milliseconds and number of launches timed since
 * the last reset.  Waits for outstanding launches. */
int sbnb_engine_walk_timing(sbnb_engine* engine, double* total_ms, int64_t* samples,
                            int32_t reset);

/* Restrict this engine to the pattern range [begin, end) of the alignment it
 * was created with (site-pattern sharding across GPUs: every rank stages the
 * same trees, computes partial sums over its range, and the caller
 * sum-all-reduces log-likelihoods and edge derivatives). */
int sbnb_engine_set_pattern_range(sbnb_engine* engine, int64_t begin, int64_t end);

/* ---- host finishing, split out for site-pattern sharding ------------------ */

/*
 * The O(n) host tail of FatBeagle::Gradient (fat_beagle.cpp:467-545) applied to
 * the RAW sums sbnb_batch_fetch returns: fixed-node zeroing of the branch
 * gradient, central differences of the substitution gradient, the site-model
 * contraction (fat_beagle.cpp:389-398) and, for rooted trees, the ratio /
 * root-height and clock gradients (rooted_gradient_transforms.cpp).  All three
 * inputs are sums over site patterns, so ranks that each hold a pattern range
 * sum-all-reduce them and call this once; sbnb_gradients_* is exactly
 * stage + run + fetch + this.  Needs no device.  with_substitution_fd says
 * whether log_likelihoods carries the [T][2 * coords] finite-difference
 * evaluations after the T base values (batch staged with SBNB_STAGE_SUBSTITUTION_FD).
 */
int sbnb_finish_gradients(const char* substitution, const char* site, const char* clock,
                          int32_t taxon_count, const sbnb_tree_batch* trees, int32_t rooted,
                          int32_t with_substitution_fd, const double* log_likelihoods,
                          const double* branch_gradients, const double* rate_gradients,
                          const sbnb_gradient_out* out);
/* The same host tail for a batch staged with SBNB_STAGE_SUBSTITUTION_ANALYTIC: the
 * "substitution_model" block is < W, V^-1 dQ/dtheta V > + d pi/d theta . R from the (reduced)
 * substitution sums and the parameter rows; everything else as sbnb_finish_gradients. */
int sbnb_finish_gradients_analytic(const char* substitution, const char* site, const char* clock,
                                   int32_t taxon_count, const sbnb_tree_batch* trees, int32_t rooted,
                                   const double* params, const double* log_likelihoods,
                                   const double* branch_gradients, const double* rate_gradients,
                                   const double* substitution_sums, const sbnb_gradient_out* out);
/* The host tail for a +I site model, which the two entries above refuse (they have no
 * d/d proportion invariant): everything as sbnb_finish_gradients_analytic, with the [T][5]
 * sums of sbnb_batch_fetch_invariant_sums; substitution_sums may be NULL (no
 * "substitution_model" block is then written).  The site-model row is [shape | proportion
 * invariant]: d logL / dp = D + sum over edges of tau g / (1 - p). */
int sbnb_finish_gradients_invariant(const char* substitution, const char* site, const char* clock,
                                    int32_t taxon_count, const sbnb_tree_batch* trees, int32_t rooted,
                                    const double* params, const double* log_likelihoods,
                                    const double* branch_gradients, const double* rate_gradients,
                                    const double* substitution_sums, const double* invariant_sums,
                                    const sbnb_gradient_out* out);
/* Adds the log-determinant Jacobian of the height-ratio transform
 * (fat_beagle.cpp:82-94) to already reduced rooted log-likelihoods, in place. */
int sbnb_finish_log_likelihoods_rooted(int32_t taxon_count, const sbnb_tree_batch* trees,
                                       double* log_likelihoods);

/* ---- host-only diagnostics (no device needed; used by the CPU test-suite) -- */

/* The traversal programs generated for one topology.  post_ops / pre_ops
 * receive (taxon_count-1) records of 8 int32 each:
 *   post: {node, child0, child1, dst_slot, child0_slot, child1_slot, flags, 0}
 *   pre:  {node, child0, child1, pre_slot, child0_dst_slot, child1_dst_slot, flags, 0}
 * flags: 1 = child0 is a leaf, 2 = child1 is a leaf, 4 = node is the root.
 * slots[0..1] = stack depth of the post-order / pre-order walk. */
int sbnb_debug_tree_program(const int32_t* parent_ids, int32_t node_count, int32_t taxon_count,
                            int32_t* post_ops, int32_t* pre_ops, int32_t* slots);

/* The model tables built from one parameter row: eigenvectors[16],
 * inverse_eigenvectors[16], eigenvalues[4], frequencies[4], q[16] (row-major),
 * then category rates / weights / rate derivatives (category_count each; with +I the rates
 * and their derivatives divided by 1 - proportion invariant). */
int sbnb_debug_model_tables(const char* substitution, const char* site, const char* clock,
                            const double* param_row, double* eigenvectors,
                            double* inverse_eigenvectors, double* eigenvalues, double* frequencies,
                            double* q, double* category_rates, double* category_weights,
                            double* category_rate_derivatives);

/* The host part of the analytic substitution-parameter gradient for one parameter
 * row: per gradient coordinate theta (GTR: 5 rate + 3 frequency stick-breaking
 * coordinates; HKY: kappa + 3), B_theta = V^-1 (dQ/dtheta) V as b[theta][16] (row-major)
 * and d pi / d theta as dfreqs[theta][4]; *count = number of coordinates. */
int sbnb_debug_substitution_derivatives(const char* substitution, const char* site, const char* clock,
                                        const double* param_row, double* b, double* dfreqs,
                                        int32_t* count);

#ifdef __cplusplus
}
#endif

#endif /* SBN_B200_H_ */
