/*
 * sbn_b200_patterns.h -- C ABI of the site-pattern compression of libsbn_b200.so:
 * the B200-native replacement for phylovi/libsbn's SitePattern::Compress
 * (src/site_pattern.cpp:77-115) with its DNA symbol table (site_pattern.cpp:15-45),
 * the step that turns an alignment into the (patterns, weights) pair every
 * likelihood engine is built from (SURVEY.md 8f, item 3).
 *
 * The reference walks the alignment column by column on the host, hashing each
 * column (a std::vector<int>) into an unordered_map.  Here the alignment goes to
 * the device once; columns are symbolised and hashed, de-duplicated through an
 * open-addressing table, verified byte for byte against their representative,
 * and emitted -- all in HBM-bound byte/integer kernels.
 *
 * Result.  The same SET of (pattern, weight) pairs as the reference.  The
 * reference's ORDER is the iteration order of a libstdc++ unordered_map (hash
 * and bucket-count dependent, SURVEY.md 8c); ours is the order of first
 * appearance in the alignment, which is deterministic.  Log-likelihoods do not
 * depend on the order.
 *
 * Same conventions as sbn_b200.h: plain C, host pointers borrowed for the call,
 * 0 on success / negative SBNB_ERR_* on failure, sbnb_last_error() for the
 * message, no CPU fallback.
 */
#ifndef SBN_B200_PATTERNS_H_
#define SBN_B200_PATTERNS_H_

#include <stddef.h>
#include <stdint.h>

#include "sbn_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/*
 * sequences: taxon_count rows of site_count characters (no terminators),
 *   row t = the sequence of the taxon with leaf id t
 *   (taxon_number_to_sequence, site_pattern.cpp:82-86).
 * out_patterns: capacity taxon_count * site_count bytes; filled as
 *   [taxon][pattern_count] (row pitch = the returned pattern count) with symbols
 *   0..3 = A C G T and 4 = gap / unknown / degenerate, as GetSymbolTable maps them.
 * out_weights: capacity site_count doubles; the multiplicity of each pattern.
 * out_device_ms: if not NULL, the device time of the kernels (CUDA events).
 * A character outside the symbol table fails with the reference's message
 * "Symbol 'c' not known." (site_pattern.cpp:47-55).
 */
int sbnb_compress_site_patterns(int32_t taxon_count, int64_t site_count, const char* sequences,
                                int32_t device, uint8_t* out_patterns, double* out_weights,
                                int64_t* out_pattern_count, double* out_device_ms);
/*
 * sbnb_compress_site_patterns with the output in the given tip encoding (SBNB_TIPS_*,
 * sbn_b200.h; sbnb_compress_site_patterns is the SBNB_TIPS_STATES case).  With
 * SBNB_TIPS_NUCLEOTIDE_MASKS the characters map through the IUPAC table, upper and lower
 * case: A C G T = 1 2 4 8, U = T, R Y S W K M B D H V = the masks of the states they allow,
 * N X ? - = 15; columns that differ only in degenerate codes are different patterns.
 */
int sbnb_compress_site_patterns_encoded(int32_t taxon_count, int64_t site_count, const char* sequences,
                                        int32_t tip_encoding, int32_t device, uint8_t* out_patterns,
                                        double* out_weights, int64_t* out_pattern_count,
                                        double* out_device_ms);

#ifdef __cplusplus
}
#endif

#endif /* SBN_B200_PATTERNS_H_ */
