/*
 * libhmsbeagle/beagle.h -- the INNER drop-in boundary of libsbn_b200: the subset
 * of the BEAGLE C API that phylovi/libsbn links against.
 *
 * BEAGLE (beagle-dev/beagle-lib, branch hmc-clock, unpinned: reference
 * README.md:16-19, SConstruct:187-197) is a third-party dependency that is NOT
 * vendored in the reference tree.  This header declares the 17 C entry points,
 * 2 structs and the flag / return-code enums that the reference calls (all call
 * sites: src/fat_beagle.cpp; flag names: src/beagle_flag_names.hpp:22-54; python
 * enum: src/pylibsbn.cpp:448-475), so that the UNMODIFIED reference host code
 * compiles against it, plus one standard BEAGLE call the reference does not make,
 * beagleGetSiteLogLikelihoods (per-pattern log-likelihoods for topology tests and
 * model comparison).  Two libraries
 * implement this ABI:
 *   - libsbn_b200/csrc/beagle_shim.cu -> libhmsbeagle_b200.so: every call runs on
 *     the B200 (the product's compatibility path: relink, nothing else changes);
 *   - oracle/beagle_cpu.cpp: the CPU restatement used only as the test oracle (the 17
 *     calls the reference makes; not beagleGetSiteLogLikelihoods).
 * The performance path is the outer boundary, include/sbn_b200.h.
 *
 * Written from the reference's call sites and the published BEAGLE API
 * description; bit positions follow the name table in
 * src/beagle_flag_names.hpp:22-54.
 */
#ifndef SBNB_LIBHMSBEAGLE_BEAGLE_H_
#define SBNB_LIBHMSBEAGLE_BEAGLE_H_

#ifdef __cplusplus
extern "C" {
#endif

enum BeagleReturnCodes {
  BEAGLE_SUCCESS = 0,
  BEAGLE_ERROR_GENERAL = -1,
  BEAGLE_ERROR_OUT_OF_MEMORY = -2,
  BEAGLE_ERROR_UNIDENTIFIED_EXCEPTION = -3,
  BEAGLE_ERROR_UNINITIALIZED_INSTANCE = -4,
  BEAGLE_ERROR_OUT_OF_RANGE = -5,
  BEAGLE_ERROR_NO_RESOURCE = -6,
  BEAGLE_ERROR_NO_IMPLEMENTATION = -7,
  BEAGLE_ERROR_FLOATING_POINT = -8
};

/* Bit k of the flag word is entry k of beagle_flag_names.hpp:22-54. */
enum BeagleFlags {
  BEAGLE_FLAG_PRECISION_SINGLE = 1L << 0,
  BEAGLE_FLAG_PRECISION_DOUBLE = 1L << 1,
  BEAGLE_FLAG_COMPUTATION_SYNCH = 1L << 2,
  BEAGLE_FLAG_COMPUTATION_ASYNCH = 1L << 3,
  BEAGLE_FLAG_EIGEN_REAL = 1L << 4,
  BEAGLE_FLAG_EIGEN_COMPLEX = 1L << 5,
  BEAGLE_FLAG_SCALING_MANUAL = 1L << 6,
  BEAGLE_FLAG_SCALING_AUTO = 1L << 7,
  BEAGLE_FLAG_SCALING_ALWAYS = 1L << 8,
  BEAGLE_FLAG_SCALERS_RAW = 1L << 9,
  BEAGLE_FLAG_SCALERS_LOG = 1L << 10,
  BEAGLE_FLAG_VECTOR_SSE = 1L << 11,
  BEAGLE_FLAG_VECTOR_NONE = 1L << 12,
  BEAGLE_FLAG_THREADING_OPENMP = 1L << 13,
  BEAGLE_FLAG_THREADING_NONE = 1L << 14,
  BEAGLE_FLAG_PROCESSOR_CPU = 1L << 15,
  BEAGLE_FLAG_PROCESSOR_GPU = 1L << 16,
  BEAGLE_FLAG_PROCESSOR_FPGA = 1L << 17,
  BEAGLE_FLAG_PROCESSOR_CELL = 1L << 18,
  BEAGLE_FLAG_PROCESSOR_PHI = 1L << 19,
  BEAGLE_FLAG_INVEVEC_STANDARD = 1L << 20,
  BEAGLE_FLAG_INVEVEC_TRANSPOSED = 1L << 21,
  BEAGLE_FLAG_FRAMEWORK_CUDA = 1L << 22,
  BEAGLE_FLAG_FRAMEWORK_OPENCL = 1L << 23,
  BEAGLE_FLAG_VECTOR_AVX = 1L << 24,
  BEAGLE_FLAG_SCALING_DYNAMIC = 1L << 25,
  BEAGLE_FLAG_PROCESSOR_OTHER = 1L << 26,
  BEAGLE_FLAG_FRAMEWORK_CPU = 1L << 27,
  BEAGLE_FLAG_PARALLELOPS_STREAMS = 1L << 28,
  BEAGLE_FLAG_PARALLELOPS_GRID = 1L << 29,
  BEAGLE_FLAG_THREADING_CPP = 1L << 30
};

enum BeagleOpCodes { BEAGLE_OP_COUNT = 7, BEAGLE_OP_NONE = -1 };

typedef struct {
  int resourceNumber;
  char* resourceName;
  char* implName;
  char* implDescription;
  long flags;
} BeagleInstanceDetails;

/* One partial-likelihood update; used by both the post-order
 * (fat_beagle.cpp:327-342) and the pre-order (fat_beagle.cpp:344-362) passes. */
typedef struct {
  int destinationPartials;
  int destinationScaleWrite;
  int destinationScaleRead;
  int child1Partials;
  int child1TransitionMatrix;
  int child2Partials;
  int child2TransitionMatrix;
} BeagleOperation;

/* fat_beagle.cpp:247-251 */
int beagleCreateInstance(int tipCount, int partialsBufferCount, int compactBufferCount,
                         int stateCount, int patternCount, int eigenBufferCount,
                         int matrixBufferCount, int categoryCount, int scaleBufferCount,
                         int* resourceList, int resourceCount, long preferenceFlags,
                         long requirementFlags, BeagleInstanceDetails* returnInfo);
/* fat_beagle.cpp:32 */
int beagleFinalizeInstance(int instance);
/* fat_beagle.cpp:261 -- states >= stateCount mean "missing". */
int beagleSetTipStates(int instance, int tipIndex, const int* inStates);
/* fat_beagle.cpp:268 -- [pattern][state], replicated over categories. */
int beagleSetTipPartials(int instance, int tipIndex, const double* inPartials);
/* fat_beagle.cpp:323 -- [category][pattern][state]. */
int beagleSetPartials(int instance, int bufferIndex, const double* inPartials);
/* fat_beagle.cpp:263,270 */
int beagleSetPatternWeights(int instance, const double* inPatternWeights);
/* fat_beagle.cpp:277 */
int beagleSetCategoryWeights(int instance, int categoryWeightsIndex,
                             const double* inCategoryWeights);
/* fat_beagle.cpp:278 */
int beagleSetCategoryRates(int instance, const double* inCategoryRates);
/* fat_beagle.cpp:289 */
int beagleSetStateFrequencies(int instance, int stateFrequenciesIndex,
                              const double* inStateFrequencies);
/* fat_beagle.cpp:290-293 -- row-major eigenvectors / inverse eigenvectors. */
int beagleSetEigenDecomposition(int instance, int eigenIndex,
                                const double* inEigenVectors,
                                const double* inInverseEigenVectors,
                                const double* inEigenValues);
/* fat_beagle.cpp:307-313 */
int beagleUpdateTransitionMatrices(int instance, int eigenIndex,
                                   const int* probabilityIndices,
                                   const int* firstDerivativeIndices,
                                   const int* secondDerivativeIndices,
                                   const double* edgeLengths, int count);
/* fat_beagle.cpp:129 -- [category][i][j]. */
int beagleSetDifferentialMatrix(int instance, int matrixIndex, const double* inMatrix);
/* fat_beagle.cpp:54,122 */
int beagleResetScaleFactors(int instance, int cumulativeScaleIndex);
/* fat_beagle.cpp:60-63,139-141 */
int beagleUpdatePartials(int instance, const BeagleOperation* operations,
                         int operationCount, int cumulativeScaleIndex);
/* fat_beagle.cpp:149-151 */
int beagleUpdatePrePartials(int instance, const BeagleOperation* operations,
                            int operationCount, int cumulativeScaleIndex);
/* fat_beagle.cpp:157-166 */
int beagleCalculateEdgeDerivatives(int instance, const int* postBufferIndices,
                                   const int* preBufferIndices,
                                   const int* derivativeMatrixIndices,
                                   const int* categoryWeightsIndices, int count,
                                   double* outDerivatives, double* outSumDerivatives,
                                   double* outSumSquaredDerivatives);
/* fat_beagle.cpp:65-68,170-173 */
int beagleCalculateRootLogLikelihoods(int instance, const int* bufferIndices,
                                      const int* categoryWeightsIndices,
                                      const int* stateFrequenciesIndices,
                                      const int* cumulativeScaleIndices, int count,
                                      double* outSumLogLikelihood);

/* ---- a standard BEAGLE call the reference does not make ---------------------------------- */

/* The per-pattern log-likelihoods of the most recent beagleCalculateRootLogLikelihoods on the
 * instance (cumulative scale factors included, pattern weights not): patternCount doubles.
 * An error before any root call.  (Declared extern, apart from the 17 calls above.) */
extern int beagleGetSiteLogLikelihoods(int instance, double* outLogLikelihoods);

#ifdef __cplusplus
}
#endif

#endif /* SBNB_LIBHMSBEAGLE_BEAGLE_H_ */
