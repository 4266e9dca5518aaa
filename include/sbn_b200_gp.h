/*
 * sbn_b200_gp.h -- C ABI of the generalized-pruning (GP) engine of libsbn_b200.so:
 * the B200-native replacement for phylovi/libsbn's GPEngine (src/gp_engine.hpp,
 * src/gp_engine.cpp), which executes GPOperation programs (src/gp_operation.hpp)
 * on partial likelihood vectors (PLVs) of the subsplit DAG.
 *
 * The reference keeps its PLVs in an mmapped file (src/mmapped_plv.hpp) and
 * interprets one std::variant op at a time on the host with Eigen
 * (GPEngine::ProcessOperations, gp_engine.cpp:167-171).  Here the PLVs live in
 * HBM for the life of the engine and a whole program is executed by ONE
 * persistent kernel launch: the host-side scheduler (GPDAG, unchanged) flattens
 * its GPOperationVector into int32 words and hands it over.
 *
 * Same conventions as sbn_b200.h: plain C, host pointers borrowed for the call,
 * 0 on success / negative SBNB_ERR_* on failure, sbnb_last_error() for the
 * message, no CPU fallback.  The reference's Assert/Failwith conditions inside
 * ops (non-finite PLV after Multiply, negative PLV entry, rescaled stationary
 * distribution, dest rescaling too large; gp_engine.cpp:70-71, 89-90, 115,
 * 300-301) surface as SBNB_ERR_GP_ASSERT with the reference's message.
 */
#ifndef SBN_B200_GP_H_
#define SBN_B200_GP_H_

#include <stddef.h>
#include <stdint.h>

#include "sbn_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

enum { SBNB_ERR_GP_ASSERT = -6 };

typedef struct sbnb_gp_engine sbnb_gp_engine; /* replaces GPEngine (gp_engine.hpp:20-207) */

/*
 * Program encoding: a flat int32 stream, one record per GPOperation
 * (gp_operation.hpp:25-171), record = opcode followed by its size_t fields in
 * declaration order:
 */
enum {
  SBNB_GP_ZERO_PLV = 0,                  /* dest                                  */
  SBNB_GP_SET_TO_STATIONARY = 1,         /* dest, root_gpcsp_idx                  */
  SBNB_GP_INCREMENT_WITH_EVOLVED = 2,    /* dest, gpcsp, src                      */
  SBNB_GP_MULTIPLY = 3,                  /* dest, src1, src2                      */
  SBNB_GP_LIKELIHOOD = 4,                /* dest, child, parent                   */
  SBNB_GP_OPTIMIZE_BRANCH_LENGTH = 5,    /* leafward, rootward, gpcsp             */
  SBNB_GP_UPDATE_SBN_PROBABILITIES = 6,  /* start, stop                           */
  SBNB_GP_RESET_MARGINAL_LIKELIHOOD = 7, /* (no fields)                           */
  SBNB_GP_INCREMENT_MARGINAL = 8,        /* stationary_times_prior, rootsplit, p  */
  SBNB_GP_PREP_FOR_MARGINALIZATION = 9   /* dest, count, src[count]               */
};

/*
 * GPEngine::GPEngine (gp_engine.cpp:9-46).  tip_states is
 * SitePattern::GetPatterns() flattened [taxon][pattern] (0..3, >= 4 = gap), from
 * which the first taxon_count PLVs are initialised (InitializePLVsWithSitePatterns,
 * gp_engine.cpp:268-286); pattern_weights is SitePattern::GetWeights(); site_count
 * is SitePattern::SiteCount().  sbn_prior (q), unconditional_node_probabilities and
 * inverted_sbn_prior may be NULL (the reference's unit test passes empty vectors);
 * their lengths are gpcsp_count, node_count and gpcsp_count.  Branch lengths start
 * at 0.1 (gp_engine.hpp:84).  The substitution model is JC69, as in the reference
 * (gp_engine.hpp:143-154).
 */
int sbnb_gp_create(int32_t taxon_count, int64_t pattern_count, const uint8_t* tip_states,
                   const double* pattern_weights, int64_t site_count, int32_t plv_count,
                   int32_t gpcsp_count, double rescaling_threshold, const double* sbn_prior,
                   const double* unconditional_node_probabilities, int32_t node_count,
                   const double* inverted_sbn_prior, int32_t device, sbnb_gp_engine** out);
/* sbnb_gp_create with the tips in the given encoding (SBNB_TIPS_*, sbn_b200.h;
 * sbnb_gp_create is the SBNB_TIPS_STATES case).  With SBNB_TIPS_NUCLEOTIDE_MASKS a leaf
 * PLV entry is bit s of the tip's mask, in every category; 15 is the all-ones gap. */
int sbnb_gp_create_encoded(int32_t taxon_count, int64_t pattern_count, const uint8_t* tips,
                           int32_t tip_encoding, const double* pattern_weights, int64_t site_count,
                           int32_t plv_count, int32_t gpcsp_count, double rescaling_threshold,
                           const double* sbn_prior, const double* unconditional_node_probabilities,
                           int32_t node_count, const double* inverted_sbn_prior, int32_t device,
                           sbnb_gp_engine** out);
void sbnb_gp_destroy(sbnb_gp_engine* engine);

/*
 * The substitution model behind every transition matrix and the stationary distribution.
 * The reference's GPEngine is hard-wired to JC69 (gp_engine.hpp:143-154; SURVEY.md 8f-4); this
 * is an addition.  `substitution` and `params` as in the "entire substitution" block of a
 * phylo_model_params row (sbn_b200.h): "JC69" (no parameters, the default), "GTR" (6 rates,
 * then 4 frequencies; substitution_model.cpp:39-80) or "HKY" (4 frequencies, then kappa:
 * sub-blocks in key order, block_specification.cpp:10-21).
 * Takes effect with the next call; PLVs computed before are not touched.
 */
int sbnb_gp_set_substitution_model(sbnb_gp_engine* engine, const char* substitution, const double* params,
                                   int32_t param_count);

/*
 * Rate categories (SURVEY.md 8f-4; an addition, the reference's GPEngine has one rate): `site`
 * and `params` as in the "entire site" block of a phylo_model_params row -- "constant",
 * "weibull+K" (shape; the median discretisation of site_model.cpp:37-62) or "gamma+K" (shape),
 * K = 1, 2, 4 or 8.  Every PLV becomes [pattern][category][4] (sbnb_gp_get_plv returns
 * pattern_count * K * 4 doubles), every transition matrix P(r_c t) per category, every site
 * likelihood the proportion-weighted sum over the categories; the op programs do not change.
 * RESETS the PLVs and rescaling counts to their state after sbnb_gp_create.
 */
int sbnb_gp_set_site_model(sbnb_gp_engine* engine, const char* site, const double* params, int32_t param_count);
int32_t sbnb_gp_category_count(const sbnb_gp_engine* engine);

/* GPEngine::ProcessOperations (gp_engine.cpp:167-171): the whole program in one
 * kernel launch; returns after it has finished. */
int sbnb_gp_process_operations(sbnb_gp_engine* engine, const int32_t* program, int64_t word_count);

/*
 * The schedule the device runs for `program` (host only, no device needed; what
 * sbnb_gp_process_operations does first):
 *   - a run of adjacent IncrementWithWeightedEvolvedPLV records into one PLV (a node's
 *     increments, gp_dag.cpp:264-290) becomes one record of internal kind 10 -- dest, n,
 *     (gpcsp, src) x n, n <= 4 -- whose sources are loaded together and added in the
 *     reference's order; when the PLV's last writer is a ZeroPLV nobody has read since, the
 *     record (or the single increment) carries bit 30 of word 0 ("fresh": the sum starts from
 *     0, dest is not loaded: 0 + x = x exactly) and that ZeroPLV carries bit 30 too (it only
 *     clears the rescaling count);
 *   - the records are re-ordered by dependency level -- an op's level is one more than the
 *     highest level of the ops it must follow (read after write, write after write, write
 *     after read over PLVs, rescaling counts, q, branch lengths, log-likelihood rows, the
 *     log-marginal vector) -- and inside a level by kind, so that every value is computed
 *     by the same arithmetic as in the reference's sequential order
 *     (GPEngine::ProcessOperations, gp_engine.cpp:167-171);
 *   - word 0 of the first record of a run of mutually independent records of one kind
 *     carries the run length in bits 8..15 (the interpreter issues their loads together);
 *     the opcode is word 0 & 0xff;
 *   - bit 16 of word 0 of an increment (bit 16 + u for source u of a kind-10 record) marks a rootward
 *     source: a PLV that carries the stationary distribution (SetToStationaryDistribution, and every
 *     PLV computed from one), which evolves as P(t)^T r -- P(t) is not symmetric unless the
 *     frequencies are equal.  The directions follow the program in its order, starting from no
 *     rootward PLV (sbnb_gp_process_operations starts from what the engine's earlier programs left).
 * out must hold word_count words; *out_word_count (<= word_count) of them are written.
 */
int sbnb_gp_schedule_program(int32_t plv_count, int32_t gpcsp_count, const int32_t* program,
                             int64_t word_count, int32_t* out, int64_t* out_word_count);

/* gp_engine.cpp:193-209. */
int sbnb_gp_set_branch_lengths(sbnb_gp_engine* engine, const double* branch_lengths);
int sbnb_gp_set_branch_lengths_to_constant(sbnb_gp_engine* engine, double branch_length);
int sbnb_gp_get_branch_lengths(sbnb_gp_engine* engine, double* out);
int sbnb_gp_reset_log_marginal_likelihood(sbnb_gp_engine* engine);
int sbnb_gp_get_log_marginal_likelihood(sbnb_gp_engine* engine, double* out);
/* GetPerGPCSPLogLikelihoods(start, length) (gp_engine.cpp:213-220): rows of the
 * log-likelihood matrix times the pattern weights. */
int sbnb_gp_get_per_gpcsp_log_likelihoods(sbnb_gp_engine* engine, int32_t start, int32_t length,
                                          double* out);
/* GetPerGPCSPComponentsOfFullLogMarginal (gp_engine.cpp:222-225). */
int sbnb_gp_get_per_gpcsp_components_of_full_log_marginal(sbnb_gp_engine* engine, double* out);
/* GetLogLikelihoodMatrix (gp_engine.cpp:227-229): [gpcsp_count][pattern_count] row-major. */
int sbnb_gp_get_log_likelihood_matrix(sbnb_gp_engine* engine, double* out);
/* GetSBNParameters (gp_engine.cpp:235) and its setter. */
int sbnb_gp_get_sbn_parameters(sbnb_gp_engine* engine, double* out);
int sbnb_gp_set_sbn_parameters(sbnb_gp_engine* engine, const double* q);
/* GetHybridMarginals (gp_engine.cpp:231-233) and a setter for values computed elsewhere. */
int sbnb_gp_get_hybrid_marginals(sbnb_gp_engine* engine, double* out);
int sbnb_gp_set_hybrid_marginals(sbnb_gp_engine* engine, const double* values);

/* LogLikelihoodAndDerivative (gp_engine.cpp:244-266): out[0] = log likelihood of
 * the op's edge at its current branch length, out[1] = its derivative. */
int sbnb_gp_log_likelihood_and_derivative(sbnb_gp_engine* engine, int32_t leafward, int32_t rootward,
                                          int32_t gpcsp, double* out);
/* SetTransitionMatrixToHaveBranchLength + GetTransitionMatrix (gp_engine.cpp:173-176),
 * computed on the device; out = 16 doubles row-major. */
int sbnb_gp_transition_matrix(sbnb_gp_engine* engine, double branch_length, double* out);

/*
 * CalculateQuartetHybridLikelihoods (gp_engine.cpp:396-452).  Each tip list is
 * count records of 3 int32 {tip_node_id, plv_idx, gpcsp_idx}
 * (quartet_hybrid_request.hpp).  out receives
 * rootward_count * sister_count * rotated_count * sorted_count log likelihoods in
 * the reference's loop order.  sbnb_gp_process_quartet_hybrid_request additionally
 * stores their LogSum in the hybrid marginal of central_gpcsp (gp_engine.cpp:454-460).
 */
int sbnb_gp_quartet_hybrid_likelihoods(sbnb_gp_engine* engine, int32_t central_gpcsp,
                                       const int32_t* rootward_tips, int32_t rootward_count,
                                       const int32_t* sister_tips, int32_t sister_count,
                                       const int32_t* rotated_tips, int32_t rotated_count,
                                       const int32_t* sorted_tips, int32_t sorted_count, double* out);
int sbnb_gp_process_quartet_hybrid_request(sbnb_gp_engine* engine, int32_t central_gpcsp,
                                           const int32_t* rootward_tips, int32_t rootward_count,
                                           const int32_t* sister_tips, int32_t sister_count,
                                           const int32_t* rotated_tips, int32_t rotated_count,
                                           const int32_t* sorted_tips, int32_t sorted_count);

/* Diagnostics: one PLV ([pattern][4], the reference's column-major 4 x P block,
 * mmapped_plv.hpp:15-41), the per-PLV rescaling counts, kernels launched so far,
 * and the device time (ms, CUDA events) of the last process_operations call. */
int sbnb_gp_get_plv(sbnb_gp_engine* engine, int32_t plv_idx, double* out);
int sbnb_gp_get_rescaling_counts(sbnb_gp_engine* engine, int32_t* out);
int64_t sbnb_gp_launch_count(const sbnb_gp_engine* engine);
double sbnb_gp_last_kernel_ms(const sbnb_gp_engine* engine);
/* The interpreter's launch plan for the current shape (patterns x categories, PLV and GPCSP
 * counts), for tests that claim a regime: out[0] threads per CTA, out[1] CTAs, out[2] 1 when a
 * multi-CTA grid runs as one thread-block cluster, out[3] 1 when the transition matrices and q
 * live in shared memory (0: global memory), out[4] 1 when the per-warp rescaling counts live in
 * shared memory (0: global memory), out[5] doubles of UpdateSBNProbabilities scratch. */
int sbnb_gp_debug_launch_plan(const sbnb_gp_engine* engine, int32_t* out);

#ifdef __cplusplus
}
#endif

#endif /* SBN_B200_GP_H_ */
