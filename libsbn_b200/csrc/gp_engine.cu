// GP engine of libsbn_b200: the device-resident replacement for the reference's
// GPEngine (src/gp_engine.hpp, src/gp_engine.cpp) and the C ABI of
// include/sbn_b200_gp.h.
//
// Design.  Every GP operation except three acts on site patterns independently,
// so a thread owns one site pattern for the WHOLE program: one persistent kernel
// interprets the op stream, and all data hazards between ops (op i + 1 reads the PLV
// op i wrote) are same-thread hazards that need no barrier.  The PLVs stay in HBM/L2
// ([plv][pattern][state], the reference's memory order, mmapped_plv.hpp:15-41), 32
// bytes per (PLV, pattern).  The three cross-pattern couplings are reductions:
//   * Multiply's finite check, min/max scan and conditional rescale
//     (gp_engine.cpp:111-117, 288-320) -- one reduction of two integer keys per op
//     instead of the reference's three full passes;
//   * OptimizeBranchLength's objective (gp_engine.cpp:326-345): Brent's control
//     flow runs redundantly in every thread on identical, deterministically
//     reduced objective values, so no host round trip happens inside the search;
//   * UpdateSBNProbabilities' per-GPCSP weighted sums (gp_engine.cpp:136-153).
// Scalars (rescaling counts per warp, q, the transition matrices of all GPCSPs) live in
// shared memory; every CTA keeps its own copies and computes the same values.
//
// At DS1 size an op is a chain of latencies, not arithmetic or bandwidth (measured: 0.13
// instructions per cycle per warp, fixed-latency and scoreboard stalls), so the work is
// arranged to shorten that chain:
//   * the patterns are spread over several CTAs on different SMs (934 patterns: 8 CTAs of
//     128 threads), which share nothing but the reductions -- exchanged through an
//     LL-style mailbox in L2 (8-byte words carrying their own epoch flag: one round
//     trip, no grid-wide barrier);
//   * P(t) of every GPCSP is computed once per launch by half-warps and kept current by
//     OptimizeBranchLength (every thread evaluating V exp(Lambda t) V^-1 for itself was
//     ~290 fp64 instructions per op);
//   * the host re-orders the program by dependency level (CompileProgram) and marks runs
//     of independent ops of one kind as batches, whose loads are in flight together and
//     whose reductions share one exchange.
//
// There is no CPU path in this file.

#include <cooperative_groups.h>
#include <cuda_runtime.h>

#include <cmath>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "../../include/sbn_b200_gp.h"
#include "common.hpp"
#include "device_common.cuh"
#include "model.hpp"

namespace cg = cooperative_groups;


namespace sbnb {

namespace {

constexpr int kGpMaxBlockThreads = 256;
constexpr int kGpBlockThreads = 128;      // one pattern per thread ...
constexpr int kGpGridBlockThreads = 256;  // ... until the resident CTAs cannot hold them all
constexpr size_t kGpSmemBudget = 200 * 1024;  // dynamic shared memory of the interpreter
constexpr int kGpScratchDoubles = 256;
constexpr size_t kGpProgramCacheSize = 16;

// Status word written by the interpreter when a reference Assert would fire.
enum GpFault : int {
  kGpOk = 0,
  kGpFaultDestRescaling = 1,     // gp_engine.cpp:70-71
  kGpFaultRescaledStationary = 2,  // gp_engine.cpp:89-90
  kGpFaultNotFinite = 3,         // gp_engine.cpp:115
  kGpFaultNegative = 4,          // gp_engine.cpp:300-301
  kGpFaultBadProgram = 5,
  kGpFaultBarrierTimeout = 6  // a CTA of a multi-block launch never posted its partial results
};

struct GpParams {
  int64_t pattern_count;
  int32_t plv_count, gpcsp_count;
  // rate categories (a power of two <= kGpMaxCategories; 1 = the reference's GPEngine): the
  // lanes of a pattern's categories are adjacent, every PLV is [pattern][category][4]
  int32_t categories, log2_categories;
  double rates[8], proportions[8];
  double* plvs;             // [plv][pattern][category][4]
  int32_t* counts;          // [block][warp][plv]  rescaling counts, one identical copy per warp
  double* branch_lengths;   // [gpcsp]
  double* q;                // [gpcsp]
  const double* hybrid;     // [gpcsp]
  double* log_likelihoods;  // [gpcsp][pattern]
  double* log_marginal;     // [pattern]
  const double* weights;    // [pattern]
  const int32_t* program;
  int64_t word_count;
  double threshold, log_threshold;
  double* exchange;  // [2][blocks][2 kGpReduceValues] 8-byte words: cross-block reduction mailboxes
  int32_t* status;   // [2] = fault code, op index
  int32_t cluster_exchange;  // the grid is one thread-block cluster: reductions through distributed shared memory
  double* matrix_cache;  // [gpcsp][16]: where the interpreter keeps P(t_g) when shared memory cannot
  double evec[16], ivec[16], eval[4], freqs[4];
};

// gp_engine.hpp:88-98
constexpr double kMinLogBranchLength = -13.9;
constexpr double kMaxLogBranchLength = 1.1;
constexpr int kSignificantDigits = 6;
constexpr int kMaxBrentIterations = 1000;

__device__ __forceinline__ void LoadState(const double* plv, int64_t pattern, double (&x)[4]) {
  const double2* src = reinterpret_cast<const double2*>(plv + pattern * 4);
  const double2 v0 = src[0], v1 = src[1];
  x[0] = v0.x, x[1] = v0.y, x[2] = v1.x, x[3] = v1.y;
}
__device__ __forceinline__ void StoreState(double* plv, int64_t pattern, const double (&x)[4]) {
  double2* dst = reinterpret_cast<double2*>(plv + pattern * 4);
  dst[0] = make_double2(x[0], x[1]);
  dst[1] = make_double2(x[2], x[3]);
}

// P = V diag(exp(lambda t)) V^-1 (gp_engine.cpp:173-176); with `derivative`,
// V diag(lambda exp(lambda t)) V^-1 (gp_engine.cpp:178-185).
__device__ __forceinline__ void TransitionMatrix(const GpParams& p, double t, bool derivative,
                                                 double (&m)[16]) {
  double d[4];
#pragma unroll
  for (int k = 0; k < 4; k++) {
    d[k] = exp(t * p.eval[k]);
    if (derivative) d[k] *= p.eval[k];
  }
#pragma unroll
  for (int i = 0; i < 4; i++)
#pragma unroll
    for (int j = 0; j < 4; j++) {
      double sum = 0.0;
#pragma unroll
      for (int k = 0; k < 4; k++) sum += (p.evec[i * 4 + k] * d[k]) * p.ivec[k * 4 + j];
      m[i * 4 + j] = sum;
    }
}

// a^T M b
__device__ __forceinline__ double Bilinear(const double (&a)[4], const double (&m)[16],
                                           const double (&b)[4]) {
  double total = 0.0;
#pragma unroll
  for (int i = 0; i < 4; i++) {
    const double row = fma(m[i * 4 + 3], b[3], fma(m[i * 4 + 2], b[2], fma(m[i * 4 + 1], b[1], m[i * 4] * b[0])));
    total = fma(a[i], row, total);
  }
  return total;
}

// numerical_utils.hpp:36-52
__device__ __forceinline__ double LogAdd(double x, double y) {
  if (y > x) {
    const double t = x;
    x = y;
    y = t;
  }
  if (x == -INFINITY) return x;
  const double neg_diff = y - x;
  if (neg_diff < -36.04365338911715 /* LOG_EPS = log(DBL_EPSILON) */) return x;
  return x + log(1.0 + exp(neg_diff));
}

// Deterministic reductions over every thread of the launch.  Each returns the
// same bits in every thread.
//   Inside a CTA: one barrier per reduction; the per-warp mailboxes are double-buffered --
// a warp that writes buffer b for reduction r + 2 has passed the barrier of reduction r + 1,
// which every warp reaches only after it has read buffer b in reduction r.
//   Across CTAs (all co-resident: cooperative launch): no grid-wide barrier.  Every CTA posts
// its partial results as 8-byte words {epoch : 32 | half of a double : 32} -- a 64-bit store
// is single-copy atomic, so a word that shows the epoch carries its data (the LL protocol of
// collective libraries) -- and polls the words of all CTAs: ONE L2 round trip after the last
// CTA has posted, against several microseconds of a cooperative-groups grid sync.  The
// mailboxes alternate with the epoch's parity: a CTA can post epoch r + 2 only after every
// CTA has posted r + 1, i.e. after every CTA has read r.
//   A grid of at most 8 CTAs (DS1: 934 patterns = 8 x 128 threads) is launched as ONE
// thread-block cluster and the same words travel through distributed shared memory instead:
// a CTA stores its words straight into every peer's shared memory (st.shared::cluster through
// mapa addresses) and polls its own -- no L2 round trip per poll; 5 % off the DS1 Brent sweep.
// compute-sanitizer's racecheck reports exactly these store / poll pairs (the protocol IS a
// benign race on a self-validating word); SBNB_GP_NO_CLUSTER=1 selects the L2 path.
constexpr int kGpMaxGridBlocks = 160;
constexpr int kGpClusterBlocks = 8;  // a grid of at most this many CTAs is launched as one thread-block cluster
constexpr int kGpMaxCategories = 8;
constexpr int kGpChain = 4;                        // sources of one fused accumulation
constexpr int kGpFlag = 1 << 30;                   // word 0: ZeroPLV clears the count only / an accumulation starts fresh
constexpr int SBNB_GP_INTERNAL_EVOLVE_SUM = 10;    // dest, n, (gpcsp, src) x n: produced by CompileProgram only
#ifndef SBNB_GP_BATCH_OPS
#define SBNB_GP_BATCH_OPS 2
#endif
constexpr int kGpBatch = SBNB_GP_BATCH_OPS;                        // ops of one batch whose loads are in flight together
constexpr int kGpReduceValues = 2 * kGpBatch;      // values one reduction carries
constexpr int kGpSpinLimit = 1 << 21;  // polls before a CTA gives up (a lost peer must not hang the device)

// Order-preserving map of a double onto an unsigned 64-bit key (negative values below
// positive ones, -0 just below +0, +inf and NaNs with a clear sign bit on top): maxima over
// site patterns are taken on keys with integer compares and the warp-wide REDUX
// instruction instead of a chain of NaN-aware fmax sequences.
__device__ __forceinline__ unsigned long long SortableKey(double x) {
  const long long bits = __double_as_longlong(x);
  return static_cast<unsigned long long>(bits ^ ((bits >> 63) | static_cast<long long>(0x8000000000000000ull)));
}
__device__ __forceinline__ double FromSortableKey(unsigned long long key) {
  const long long bits = static_cast<long long>(key);
  return __longlong_as_double(bits < 0 ? (bits & 0x7fffffffffffffffll) : ~bits);
}

struct Reducer {
  const GpParams& p;
  bool multi_block;
  unsigned long long (*smem)[kGpMaxBlockThreads / 32][kGpReduceValues];  // [2][warp][value]
  unsigned long long (*landed)[kGpReduceValues];  // [block][value] values of the other CTAs as they arrive
  int* abort_flag;        // shared: a poll timed out
  // the grid is one thread-block cluster: [parity][source CTA][word] in EVERY CTA's shared memory
  // (peers store their words here directly), else NULL and the words go through p.exchange in L2
  unsigned long long (*cluster_words)[kGpClusterBlocks][2 * kGpReduceValues];
  uint32_t epoch = 0;
  int block_round = 0;    // alternates the per-warp mailboxes
  bool dead = false;

  // bits[0..COUNT): doubles that are summed (KEYS = false) or unsigned keys whose maximum is
  // taken (KEYS = true), over every thread of the launch, in a fixed order.
  template <int COUNT, bool KEYS>
  __device__ void Exchange(unsigned long long (&bits)[COUNT]) {
    static_assert(COUNT <= kGpReduceValues, "more values than a mailbox slot holds");
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps = (blockDim.x + 31) >> 5;
    auto combine = [](unsigned long long a, unsigned long long b) -> unsigned long long {
      if (KEYS) return a > b ? a : b;
      return static_cast<unsigned long long>(
          __double_as_longlong(__longlong_as_double(static_cast<long long>(a)) + __longlong_as_double(static_cast<long long>(b))));
    };
#pragma unroll
    for (int i = 0; i < COUNT; i++) {
      if (KEYS) {
        const unsigned hi = __reduce_max_sync(0xffffffffu, static_cast<unsigned>(bits[i] >> 32));
        const unsigned lo = __reduce_max_sync(
            0xffffffffu, static_cast<unsigned>(bits[i] >> 32) == hi ? static_cast<unsigned>(bits[i]) : 0u);
        bits[i] = (static_cast<unsigned long long>(hi) << 32) | lo;
      } else {
#pragma unroll
        for (int m = 16; m >= 1; m >>= 1) bits[i] = combine(bits[i], __shfl_xor_sync(0xffffffffu, bits[i], m));
      }
    }
    unsigned long long(*box)[kGpReduceValues] = smem[block_round & 1];
    block_round++;
    if (lane == 0) {
#pragma unroll
      for (int i = 0; i < COUNT; i++) box[warp][i] = bits[i];
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < COUNT; i++) {
      unsigned long long total = box[0][i];
      for (int w = 1; w < warps; w++) total = combine(total, box[w][i]);
      bits[i] = total;
    }
    if (multi_block && !dead) {
      epoch++;
      if (cluster_words != nullptr) {
        // Distributed shared memory: a word is stored straight into every peer's shared memory
        // (~200 cycles) and each CTA polls its OWN shared memory -- no L2 round trip per poll.
        unsigned long long(*const words)[2 * kGpReduceValues] = cluster_words[epoch & 1];
        if (threadIdx.x < 2 * COUNT) {
          unsigned long long mine = bits[0];
#pragma unroll
          for (int i = 1; i < COUNT; i++) mine = (static_cast<int>(threadIdx.x >> 1) == i) ? bits[i] : mine;
          const unsigned half = (threadIdx.x & 1) ? static_cast<unsigned>(mine >> 32) : static_cast<unsigned>(mine);
          const unsigned long long word = (static_cast<unsigned long long>(epoch) << 32) | half;
          const uint32_t local = static_cast<uint32_t>(__cvta_generic_to_shared(&words[blockIdx.x][threadIdx.x]));
          for (unsigned b = 0; b < gridDim.x; b++) {
            uint32_t remote;
            asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(local), "r"(b));
            asm volatile("st.relaxed.cluster.shared::cluster.u64 [%0], %1;" ::"r"(remote), "l"(word) : "memory");
          }
        }
        const int count = static_cast<int>(gridDim.x) * 2 * COUNT;
        for (int w = threadIdx.x; w < count; w += blockDim.x) {
          const int b = w / (2 * COUNT), j = w % (2 * COUNT);
          // (store and load are both relaxed at cluster scope on one naturally aligned 64-bit word:
          //  a word that shows the epoch carries its data; nothing else is ordered by it)
          const uint32_t src = static_cast<uint32_t>(__cvta_generic_to_shared(&words[b][j]));
          unsigned long long got;
          asm volatile("ld.relaxed.cluster.shared::cta.u64 %0, [%1];" : "=l"(got) : "r"(src) : "memory");
          for (int spins = 0; static_cast<uint32_t>(got >> 32) != epoch && spins < kGpSpinLimit; spins++)
            asm volatile("ld.relaxed.cluster.shared::cta.u64 %0, [%1];" : "=l"(got) : "r"(src) : "memory");
          if (static_cast<uint32_t>(got >> 32) != epoch) *abort_flag = 1;
          reinterpret_cast<uint32_t*>(landed[b])[j] = static_cast<uint32_t>(got);
        }
      } else {
        unsigned long long* const mailbox = reinterpret_cast<unsigned long long*>(p.exchange) +
                                            static_cast<size_t>(epoch & 1) * gridDim.x * (2 * kGpReduceValues);
        if (threadIdx.x < 2 * COUNT) {
          unsigned long long mine = bits[0];
#pragma unroll
          for (int i = 1; i < COUNT; i++) mine = (static_cast<int>(threadIdx.x >> 1) == i) ? bits[i] : mine;
          const unsigned half = (threadIdx.x & 1) ? static_cast<unsigned>(mine >> 32) : static_cast<unsigned>(mine);
          *reinterpret_cast<volatile unsigned long long*>(mailbox + blockIdx.x * (2 * kGpReduceValues) + threadIdx.x) =
              (static_cast<unsigned long long>(epoch) << 32) | half;
        }
        const int words = static_cast<int>(gridDim.x) * 2 * COUNT;
        for (int w = threadIdx.x; w < words; w += blockDim.x) {
          const int b = w / (2 * COUNT), j = w % (2 * COUNT);
          const volatile unsigned long long* src = mailbox + b * (2 * kGpReduceValues) + j;
          unsigned long long got = *src;
          for (int spins = 0; static_cast<uint32_t>(got >> 32) != epoch && spins < kGpSpinLimit; spins++) got = *src;
          if (static_cast<uint32_t>(got >> 32) != epoch) *abort_flag = 1;
          reinterpret_cast<uint32_t*>(landed[b])[j] = static_cast<uint32_t>(got);
        }
      }
      __syncthreads();
      // (the next write into `landed` comes after the next reduction's first barrier, which
      //  every thread reaches only after these reads)
      if (*abort_flag) {
        dead = true;
        if (threadIdx.x == 0) {
          p.status[0] = kGpFaultBarrierTimeout;
          p.status[1] = static_cast<int32_t>(epoch);
        }
      }
#pragma unroll
      for (int i = 0; i < COUNT; i++) {
        unsigned long long total = landed[0][i];
        for (unsigned b = 1; b < gridDim.x; b++) total = combine(total, landed[b][i]);
        bits[i] = total;
      }
    }
  }
  template <int COUNT>
  __device__ void MaxKeys(unsigned long long (&keys)[COUNT]) {
    Exchange<COUNT, true>(keys);
  }
  __device__ double Sum(double v) {
    unsigned long long bits[1] = {static_cast<unsigned long long>(__double_as_longlong(v))};
    Exchange<1, false>(bits);
    return __longlong_as_double(static_cast<long long>(bits[0]));
  }
  template <int COUNT>
  __device__ void Sums(double (&values)[COUNT]) {
    unsigned long long bits[COUNT];
#pragma unroll
    for (int i = 0; i < COUNT; i++) bits[i] = static_cast<unsigned long long>(__double_as_longlong(values[i]));
    Exchange<COUNT, false>(bits);
#pragma unroll
    for (int i = 0; i < COUNT; i++) values[i] = __longlong_as_double(static_cast<long long>(bits[i]));
  }
  // Every thread of the launch has got here.
  __device__ void Barrier() { Sum(0.0); }
};

// P_c(t) = V diag(exp(lambda r_c t)) V^-1 for every rate category c, computed by one warp into
// out[c][16]: lane (c, k) = ((lane >> 2) % C, lane & 3) evaluates one exponential, the
// elements are assembled from shuffles.  Same operation order per element as
// TransitionMatrix (with one category, t r_0 = t exactly).
__device__ __forceinline__ void WarpCategoryMatrices(const GpParams& p, double t, double* out) {
  const int lane = threadIdx.x & 31, C = p.categories;
  const double mine = exp((t * p.rates[(lane >> 2) & (C - 1)]) * p.eval[lane & 3]);
  const int rounds = (16 * C + 31) / 32;
  for (int r = 0; r < rounds; r++) {
    const int idx = r * 32 + lane;
    const int c = (idx >> 4) & (C - 1), i = (idx >> 2) & 3, j = idx & 3;
    double sum = 0.0;
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const double d = __shfl_sync(0xffffffffu, mine, c * 4 + k);
      sum += (p.evec[i * 4 + k] * d) * p.ivec[k * 4 + j];
    }
    if (idx < 16 * C) out[idx] = sum;
  }
}

// Shared-memory plan of the interpreter (dynamic; what does not fit stays in global memory).
struct GpSmemPlan {
  int32_t program_words;  // the op program, staged once (0: read from global memory)
  int32_t matrices;       // P_c(t_g) of every GPCSP + a copy of q: [gpcsp][category][16], [gpcsp]
  int32_t counts;         // rescaling counts, one copy per warp: [warp][plv]
  int32_t scratch;        // doubles of UpdateSBNProbabilities scratch
  size_t bytes;
};

// SINGLE: every thread owns at most one site pattern (the launch has at least as many threads
// as patterns) -- the pattern loops of the ops disappear.
template <bool SINGLE>
__device__ __forceinline__ void GpInterpretBody(const GpParams& p, const GpSmemPlan& plan,
                                                unsigned long long (*cluster_words)[kGpClusterBlocks][2 * kGpReduceValues]) {
  extern __shared__ __align__(16) unsigned char gp_smem[];
  __shared__ unsigned long long reduce_smem[2][kGpMaxBlockThreads / 32][kGpReduceValues];
  __shared__ unsigned long long landed_smem[kGpMaxGridBlocks][kGpReduceValues];
  __shared__ int abort_flag;
  __shared__ __align__(16) double warp_matrix_smem[kGpMaxBlockThreads / 32][kGpMaxCategories * 16];
  if (threadIdx.x == 0) abort_flag = 0;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps = (blockDim.x + 31) >> 5;
  const int G = p.gpcsp_count, C = p.categories;
  // ---- carve-up: [matrices | q | scratch | counts | program]
  double* const matrices_smem = reinterpret_cast<double*>(gp_smem);
  double* const q_smem = matrices_smem + (plan.matrices ? static_cast<size_t>(G) * C * 16 : 0);
  double* const scratch = q_smem + (plan.matrices ? G : 0);
  int32_t* const counts_smem = reinterpret_cast<int32_t*>(scratch + plan.scratch);
  int32_t* const program_smem = counts_smem + (plan.counts ? static_cast<size_t>(warps) * p.plv_count : 0);

  // The op program is a dependency chain: every op starts by reading its own words.  A
  // program that fits is staged in shared memory once, so that read is an LDS instead of
  // a global round trip per op.
  const int32_t* program = p.program;
  if (plan.program_words > 0) {
    for (int64_t w = threadIdx.x; w < p.word_count; w += blockDim.x) program_smem[w] = p.program[w];
    program = program_smem;
  }
  // Transition matrices of all GPCSPs at their current branch lengths: computed once per
  // launch by half-warps, kept current by OptimizeBranchLength.  (Every thread of the CTA
  // evaluating V exp(Lambda t) V^-1 for itself cost ~290 fp64 instructions per op -- on
  // ONE SM's fp64 pipe that was most of an op's 2 us.)
  double* const matrices = plan.matrices ? matrices_smem : p.matrix_cache;
  double* const q = plan.matrices ? q_smem : p.q;
  for (int g = warp; g < G; g += warps) WarpCategoryMatrices(p, p.branch_lengths[g], matrices + static_cast<size_t>(g) * C * 16);
  if (plan.matrices)
    for (int g = threadIdx.x; g < G; g += blockDim.x) q_smem[g] = p.q[g];
  // Warps drift apart between reductions, so a shared copy of the rescaling
  // counts could show a lagging warp a value from its future; every warp keeps
  // (updated by its lane 0) its own copy.  Matrices and q are only written right after a
  // barrier of the same op, which orders the write after every older read -- by one warp /
  // one thread per entry -- and a CTA barrier publishes them (racecheck-clean).
  int32_t* const counts =
      plan.counts ? counts_smem + static_cast<size_t>(warp) * p.plv_count
                  : p.counts + (static_cast<size_t>(blockIdx.x) * (kGpMaxBlockThreads / 32) + warp) * p.plv_count;
  if (plan.counts)
    for (int i = lane; i < p.plv_count; i += 32) counts[i] = p.counts[i];
  // (the first copy in global memory is what the getters and the other kernels read)
  const bool mirrors_counts = plan.counts && blockIdx.x == 0 && warp == 0;
  auto set_count = [&](int index, int value) {  // (warp-uniform call sites: one lane writes the warp's copy)
    __syncwarp();  // (the other lanes' reads of older ops)
    if (lane == 0) {
      counts[index] = value;
      if (mirrors_counts) p.counts[index] = value;
    }
    __syncwarp();
  };
  __syncthreads();

  Reducer reduce{p, gridDim.x > 1, reduce_smem, landed_smem, &abort_flag, p.cluster_exchange ? cluster_words : nullptr};
  const int64_t P = p.pattern_count;
  // A thread owns (pattern, category) pairs e = pattern * C + category: first, first + stride, ...
  // (SINGLE: at most `first`).  Block sizes are multiples of 32 and C divides 32, so the
  // category of a thread's pairs is always the same, and the C lanes of a pattern sit side
  // by side in one warp.
  const int64_t E = P << p.log2_categories;
  const int64_t first = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  const int64_t step = SINGLE ? E : stride;
  const int my_category = static_cast<int>(first) & (C - 1);
  const double my_proportion = p.proportions[my_category];
  // sum over the categories of a pattern (every lane of the warp takes part)
  auto category_sum = [&](double value) -> double {
    for (int m = 1; m < C; m <<= 1) value += __shfl_xor_sync(0xffffffffu, value, m);
    return value;
  };
  auto plv = [&](int index) -> double* { return p.plvs + static_cast<size_t>(index) * E * 4; };
  auto fault = [&](int code, int64_t pc) {
    if (first == 0) {
      p.status[0] = code;
      p.status[1] = static_cast<int32_t>(pc);
    }
  };
  auto load_matrix = [&](int gpcsp, double (&m)[16]) {
    const double2* src = reinterpret_cast<const double2*>(matrices + (static_cast<size_t>(gpcsp) * C + my_category) * 16);
#pragma unroll
    for (int x = 0; x < 8; x++) {
      const double2 v = src[x];
      m[2 * x] = v.x, m[2 * x + 1] = v.y;
    }
  };
  // P_c(t) of this lane's category, for every lane of the warp (through the warp's scratch).
  auto warp_transition_matrix = [&](double t, double (&m)[16]) {
    double* const mine = warp_matrix_smem[warp];
    __syncwarp();  // (the previous evaluation's reads)
    WarpCategoryMatrices(p, t, mine);
    __syncwarp();
    const double2* src = reinterpret_cast<const double2*>(mine + my_category * 16);
#pragma unroll
    for (int x = 0; x < 8; x++) {
      const double2 v = src[x];
      m[2 * x] = v.x, m[2 * x + 1] = v.y;
    }
  };
  // sum_k w_k (log(rootward_k^T P(t) leafward_k) + count_log): the general form of
  // OptimizeBranchLength's objective (any number of patterns per thread).
  auto edge_log_likelihood = [&](const double* rootward, const double* leafward, double t,
                                 double count_log) -> double {
    double m[16];
    warp_transition_matrix(t, m);
    double local = 0.0;
    for (int64_t base = first - lane; base < E; base += stride) {  // (warp-uniform: the category sum shuffles)
      const int64_t e = base + lane;
      double r[4] = {1.0, 1.0, 1.0, 1.0}, l[4] = {1.0, 1.0, 1.0, 1.0};
      if (e < E) {
        LoadState(rootward, e, r);
        LoadState(leafward, e, l);
      }
      const double likelihood = category_sum(Bilinear(r, m, l) * my_proportion);
      if (e < E && my_category == 0) local = fma(p.weights[e >> p.log2_categories], log(likelihood) + count_log, local);
    }
    return reduce.Sum(local);
  };

  int64_t pc = 0;
  while (pc < p.word_count && !reduce.dead) {
    // Word 0 of a record: opcode | batch << 8.  A batch is a run of `batch` records of the
    // same kind that the host found mutually independent (CompileProgram below): their
    // loads are issued together, and their reductions travel in one exchange.
    const int word0 = program[pc];
    const int opcode = word0 & 0xff;
    const int batch = max((word0 >> 8) & 0xff, 1);
    switch (opcode) {
      case SBNB_GP_ZERO_PLV: {  // gp_engine.cpp:48-51
        const double zero[4] = {0.0, 0.0, 0.0, 0.0};
        for (int u = 0; u < batch; u++) {
          const int dest = program[pc + 2 * u + 1];
          // (flagged: the next writer overwrites the whole PLV without reading it -- count only)
          if (!(program[pc + 2 * u] & kGpFlag))
            for (int64_t k = first; k < E; k += step) StoreState(plv(dest), k, zero);
          set_count(dest, 0);
        }
        pc += 2 * batch;
        break;
      }
      case SBNB_GP_SET_TO_STATIONARY: {  // gp_engine.cpp:53-62
        for (int u = 0; u < batch; u++) {
          const int dest = program[pc + 3 * u + 1], root = program[pc + 3 * u + 2];
          const double prior = q[root];
          const double x[4] = {prior * p.freqs[0], prior * p.freqs[1], prior * p.freqs[2], prior * p.freqs[3]};
          for (int64_t k = first; k < E; k += step) StoreState(plv(dest), k, x);
          set_count(dest, 0);
        }
        pc += 3 * batch;
        break;
      }
      case SBNB_GP_INCREMENT_WITH_EVOLVED: {  // gp_engine.cpp:64-82
        double* dest_plv[kGpBatch];
        const double* src_plv[kGpBatch];
        int gpcsp[kGpBatch];
        double factor[kGpBatch];
        bool fresh[kGpBatch];  // the sum starts from 0: dest is not loaded
        int faulty = -1;  // (no return inside the unrolled loops: they must stay unrolled for the arrays to be registers)
#pragma unroll
        for (int u = 0; u < kGpBatch; u++) {
          if (u < batch) {
            const int dest = program[pc + 4 * u + 1], src = program[pc + 4 * u + 3];
            gpcsp[u] = program[pc + 4 * u + 2];
            fresh[u] = (program[pc + 4 * u] & kGpFlag) != 0;
            dest_plv[u] = plv(dest);
            src_plv[u] = plv(src);
            const int difference = counts[src] - counts[dest];
            if (difference < 0 && faulty < 0) faulty = u;
            factor[u] = q[gpcsp[u]];
            if (difference > 0) factor[u] *= pow(p.threshold, static_cast<double>(difference));
          }
        }
        if (faulty >= 0) {
          fault(kGpFaultDestRescaling, pc + 4 * faulty);
          return;
        }
        for (int64_t k = first; k < E; k += step) {
          double s[kGpBatch][4], d[kGpBatch][4];
#pragma unroll
          for (int u = 0; u < kGpBatch; u++) {
            if (u < batch) {
              LoadState(src_plv[u], k, s[u]);
              if (fresh[u]) {
                d[u][0] = d[u][1] = d[u][2] = d[u][3] = 0.0;
              } else {
                LoadState(dest_plv[u], k, d[u]);
              }
            }
          }
#pragma unroll
          for (int u = 0; u < kGpBatch; u++) {
            if (u < batch) {
              double m[16];
              load_matrix(gpcsp[u], m);
#pragma unroll
              for (int i = 0; i < 4; i++)
                d[u][i] += factor[u] * fma(m[i * 4 + 3], s[u][3],
                                           fma(m[i * 4 + 2], s[u][2], fma(m[i * 4 + 1], s[u][1], m[i * 4] * s[u][0])));
              StoreState(dest_plv[u], k, d[u]);
              // (keeps the next op's matrix loads from being hoisted above this point: four
              //  matrices live at once cost 128 registers and spill)
              asm volatile("" ::: "memory");
            }
          }
        }
        pc += 4 * batch;
        break;
      }
      case SBNB_GP_INTERNAL_EVOLVE_SUM: {  // a run of gp_engine.cpp:64-82 into one PLV (CompileProgram)
        const int dest = program[pc + 1], sources = program[pc + 2];
        const bool fresh = (word0 & kGpFlag) != 0;
        double* const dest_plv = plv(dest);
        const double* src_plv[kGpChain];
        int gpcsp[kGpChain];
        double factor[kGpChain];
        int faulty = -1;
#pragma unroll
        for (int u = 0; u < kGpChain; u++) {
          if (u < sources) {
            gpcsp[u] = program[pc + 3 + 2 * u];
            const int src = program[pc + 4 + 2 * u];
            src_plv[u] = plv(src);
            const int difference = counts[src] - counts[dest];
            if (difference < 0 && faulty < 0) faulty = u;
            factor[u] = q[gpcsp[u]];
            if (difference > 0) factor[u] *= pow(p.threshold, static_cast<double>(difference));
          }
        }
        if (faulty >= 0) {
          fault(kGpFaultDestRescaling, pc);
          return;
        }
        for (int64_t k = first; k < E; k += step) {
          double s[kGpChain][4], d[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
          for (int u = 0; u < kGpChain; u++)
            if (u < sources) LoadState(src_plv[u], k, s[u]);
          if (!fresh) LoadState(dest_plv, k, d);
#pragma unroll
          for (int u = 0; u < kGpChain; u++) {  // (added in the reference's order)
            if (u < sources) {
              double m[16];
              load_matrix(gpcsp[u], m);
#pragma unroll
              for (int i = 0; i < 4; i++)
                d[i] += factor[u] * fma(m[i * 4 + 3], s[u][3], fma(m[i * 4 + 2], s[u][2], fma(m[i * 4 + 1], s[u][1], m[i * 4] * s[u][0])));
              asm volatile("" ::: "memory");
            }
          }
          StoreState(dest_plv, k, d);
        }
        pc += 3 + 2 * sources;
        break;
      }
      case SBNB_GP_MULTIPLY: {  // gp_engine.cpp:111-117 + RescalePLVIfNeeded 298-320
        double* dest_plv[kGpBatch];
        const double *a_plv[kGpBatch], *b_plv[kGpBatch];
        // per op, as sortable keys: the largest entry, and (complemented) the smallest
        unsigned long long keys[2 * kGpBatch];
#pragma unroll
        for (int u = 0; u < kGpBatch; u++) {
          keys[2 * u] = keys[2 * u + 1] = 0;
          if (u < batch) {
            dest_plv[u] = plv(program[pc + 4 * u + 1]);
            a_plv[u] = plv(program[pc + 4 * u + 2]);
            b_plv[u] = plv(program[pc + 4 * u + 3]);
          }
        }
        for (int64_t k = first; k < E; k += step) {
          double a[kGpBatch][4], b[kGpBatch][4];
#pragma unroll
          for (int u = 0; u < kGpBatch; u++) {
            if (u < batch) {
              LoadState(a_plv[u], k, a[u]);
              LoadState(b_plv[u], k, b[u]);
            }
          }
#pragma unroll
          for (int u = 0; u < kGpBatch; u++) {
            if (u < batch) {
              double d[4];
#pragma unroll
              for (int i = 0; i < 4; i++) {
                d[i] = a[u][i] * b[u][i];
                const unsigned long long key = SortableKey(d[i]);
                keys[2 * u] = key > keys[2 * u] ? key : keys[2 * u];
                keys[2 * u + 1] = ~key > keys[2 * u + 1] ? ~key : keys[2 * u + 1];
              }
              StoreState(dest_plv[u], k, d);
            }
          }
        }
        if (batch == 1) {
          unsigned long long pair[2] = {keys[0], keys[1]};
          reduce.MaxKeys<2>(pair);
          keys[0] = pair[0], keys[1] = pair[1];
        } else {
          reduce.MaxKeys<2 * kGpBatch>(keys);
        }
        int faulty = -1, fault_code = kGpOk;
#pragma unroll
        for (int u = 0; u < kGpBatch; u++) {
          if (u < batch && faulty < 0) {
            // (keys of +inf and NaN sit above every finite value; a thread without a pattern left 0)
            if (keys[2 * u] >= SortableKey(INFINITY)) {
              faulty = u, fault_code = kGpFaultNotFinite;
            } else if (keys[2 * u + 1] != 0 && ~keys[2 * u + 1] < SortableKey(-0.0)) {
              faulty = u;
              fault_code = ~keys[2 * u + 1] <= SortableKey(-INFINITY) ? kGpFaultNotFinite : kGpFaultNegative;
            }
          }
        }
        if (faulty >= 0) {
          fault(fault_code, pc + 4 * faulty);
          return;
        }
#pragma unroll
        for (int u = 0; u < kGpBatch; u++) {
          if (u < batch) {
            const int dest = program[pc + 4 * u + 1], src1 = program[pc + 4 * u + 2], src2 = program[pc + 4 * u + 3];
            int count = counts[src1] + counts[src2];
            double max_entry = keys[2 * u] == 0 ? 0.0 : FromSortableKey(keys[2 * u]);
            if (max_entry != 0.0 && max_entry < p.threshold) {
              int rescaling = 0;
              while (max_entry < p.threshold) {
                max_entry /= p.threshold;
                rescaling++;
              }
              const double divisor = pow(p.threshold, static_cast<double>(rescaling));
              for (int64_t k = first; k < E; k += step) {
                double d[4];
                LoadState(dest_plv[u], k, d);
#pragma unroll
                for (int i = 0; i < 4; i++) d[i] /= divisor;
                StoreState(dest_plv[u], k, d);
              }
              count += rescaling;
            }
            set_count(dest, count);
          }
        }
        pc += 4 * batch;
        break;
      }
      case SBNB_GP_LIKELIHOOD: {  // gp_engine.cpp:119-123, gp_engine.hpp:198-206
        const double *parent_plv[kGpBatch], *child_plv[kGpBatch];
        double* row[kGpBatch];
        int dest[kGpBatch];
        double count_log[kGpBatch];
#pragma unroll
        for (int u = 0; u < kGpBatch; u++) {
          if (u < batch) {
            dest[u] = program[pc + 4 * u + 1];
            const int child = program[pc + 4 * u + 2], parent = program[pc + 4 * u + 3];
            parent_plv[u] = plv(parent);
            child_plv[u] = plv(child);
            row[u] = p.log_likelihoods + static_cast<size_t>(dest[u]) * P;
            count_log[u] = static_cast<double>(counts[parent]) * p.log_threshold +
                           static_cast<double>(counts[child]) * p.log_threshold;
          }
        }
        for (int64_t base = first - lane; base < E; base += step) {  // (warp-uniform: the category sum shuffles)
          const int64_t k = base + lane;
          const bool on = k < E;
          double a[kGpBatch][4], b[kGpBatch][4];
#pragma unroll
          for (int u = 0; u < kGpBatch; u++) {
#pragma unroll
            for (int i = 0; i < 4; i++) a[u][i] = b[u][i] = 1.0;
            if (u < batch && on) {
              LoadState(parent_plv[u], k, a[u]);
              LoadState(child_plv[u], k, b[u]);
            }
          }
#pragma unroll
          for (int u = 0; u < kGpBatch; u++) {
            if (u < batch) {
              double m[16];
              load_matrix(dest[u], m);
              const double likelihood = category_sum(Bilinear(a[u], m, b[u]) * my_proportion);
              if (on && my_category == 0) row[u][k >> p.log2_categories] = log(likelihood) + count_log[u];
              asm volatile("" ::: "memory");
            }
          }
        }
        pc += 4 * batch;
        break;
      }
      case SBNB_GP_OPTIMIZE_BRANCH_LENGTH: {  // gp_engine.cpp:326-345, optimization.hpp:10-115
        const int leafward = program[pc + 1], rootward = program[pc + 2], gpcsp = program[pc + 3];
        const double count_log = static_cast<double>(counts[rootward]) * p.log_threshold +
                                 static_cast<double>(counts[leafward]) * p.log_threshold;
        // The thread's own patterns stay in registers for the whole search when there are at
        // most kOwn of them (the matrix form r^T P(t) l of the reference, gp_engine.cpp:244-266:
        // evaluated in the eigenbasis instead -- 4 fma per pattern -- the objective differs in
        // its last bits, and on the DS1 DAG that was enough to send one of Brent's searches
        // down another path: a 7e-5 relative change in the sum of the branch lengths after six
        // sweeps; measured, and dropped for 12 % of the sweep's time).
        constexpr int kOwn = SINGLE ? 1 : 2;
        const bool own_cover = E <= kOwn * stride;
        double r[kOwn][4], l[kOwn][4], weight[kOwn];
        if (own_cover) {
#pragma unroll
          for (int s = 0; s < kOwn; s++) {
            const int64_t k = first + s * stride;
            weight[s] = 0.0;
#pragma unroll
            for (int i = 0; i < 4; i++) r[s][i] = l[s][i] = 1.0;  // (no pattern: log of a positive number x weight 0)
            if (k < E) {
              LoadState(plv(rootward), k, r[s]);
              LoadState(plv(leafward), k, l[s]);
              if (my_category == 0) weight[s] = p.weights[k >> p.log2_categories];
            }
          }
        }
        auto f = [&](double log_branch_length) -> double {
          const double t = exp(log_branch_length);
          if (!own_cover) return -edge_log_likelihood(plv(rootward), plv(leafward), t, count_log);
          double m[16];
          warp_transition_matrix(t, m);
          double local = 0.0;
#pragma unroll
          for (int s = 0; s < kOwn; s++)
            local = fma(weight[s], log(category_sum(Bilinear(r[s], m, l[s]) * my_proportion)) + count_log, local);
          return -reduce.Sum(local);
        };
        const double current_log_branch_length = log(p.branch_lengths[gpcsp]);
        const double current_value = f(current_log_branch_length);
        // ---- Brent's minimiser, transcribed control flow (boost/math/tools/minima.hpp
        //      as copied into optimization.hpp)
        double min = kMinLogBranchLength, max = kMaxLogBranchLength;
        const double tolerance = ldexp(1.0, 1 - kSignificantDigits);
        double x, w, v, u, delta, delta2, fu, fv, fw, fx, mid, fract1, fract2;
        const double golden = 0.3819660f;
        x = w = v = max;
        fw = fv = fx = f(x);
        delta2 = delta = 0;
        int count = kMaxBrentIterations;
        do {
          mid = (min + max) / 2;
          fract1 = tolerance * fabs(x) + tolerance / 4;
          fract2 = 2 * fract1;
          if (fabs(x - mid) <= (fract2 - (max - min) / 2)) break;
          if (fabs(delta2) > fract1) {
            double r = (x - w) * (fx - fv);
            double qq = (x - v) * (fx - fw);
            double pp = (x - v) * qq - (x - w) * r;
            qq = 2 * (qq - r);
            if (qq > 0) pp = -pp;
            qq = fabs(qq);
            const double td = delta2;
            delta2 = delta;
            if ((fabs(pp) >= fabs(qq * td / 2)) || (pp <= qq * (min - x)) || (pp >= qq * (max - x))) {
              delta2 = (x >= mid) ? min - x : max - x;
              delta = golden * delta2;
            } else {
              delta = pp / qq;
              u = x + delta;
              if (((u - min) < fract2) || ((max - u) < fract2))
                delta = (mid - x) < 0 ? -fabs(fract1) : fabs(fract1);
            }
          } else {
            delta2 = (x >= mid) ? min - x : max - x;
            delta = golden * delta2;
          }
          u = (fabs(delta) >= fract1) ? (x + delta) : (delta > 0 ? (x + fabs(fract1)) : (x - fabs(fract1)));
          fu = f(u);
          if (fu <= fx) {
            if (u >= x)
              min = x;
            else
              max = x;
            v = w;
            w = x;
            x = u;
            fv = fw;
            fw = fx;
            fx = fu;
          } else {
            if (u < x)
              min = u;
            else
              max = u;
            if ((fu <= fw) || (w == x)) {
              v = w;
              w = u;
              fv = fw;
              fw = fu;
            } else if ((fu <= fv) || (v == x) || (v == w)) {
              v = u;
              fv = fu;
            }
          }
        } while (--count);
        // "Numerical optimization sometimes yields new nllk > current nllk."
        // (every warp has passed the last evaluation's barrier: nobody still reads the old values)
        const double new_length = (fx > current_value) ? exp(current_log_branch_length) : exp(x);
        p.branch_lengths[gpcsp] = new_length;
        if (warp == 0) WarpCategoryMatrices(p, new_length, matrices + static_cast<size_t>(gpcsp) * C * 16);
        __syncthreads();
        pc += 4;
        break;
      }
      case SBNB_GP_UPDATE_SBN_PROBABILITIES: {  // gp_engine.cpp:136-153
        const int start = program[pc + 1], stop = program[pc + 2];
        const int length = stop - start;
        auto set_q = [&](int g, double value) {  // (by one thread of the CTA; the caller synchronises)
          q[g] = value;
          if (plan.matrices && blockIdx.x == 0) p.q[g] = value;  // (the copy the getters read)
        };
        if (length == 1) {
          reduce.Barrier();  // lagging warps may still be reading q in an older op
          if (threadIdx.x == 0) set_q(start, 1.0);
          __syncthreads();
        } else if (length > 1) {
          // (a lagging warp may still be reading the scratch values of an older op)
          __syncthreads();
          bool use_hybrid = true;
          for (int g = start; g < stop; g++) use_hybrid = use_hybrid && (p.hybrid[g] > -INFINITY);
          // weighted sum of a GPCSP's per-pattern log likelihoods
          auto row_sum = [&](int g) -> double {
            const double* row = p.log_likelihoods + static_cast<size_t>(g) * P;
            double local = 0.0;
            for (int64_t e = first; e < E; e += stride)
              if (my_category == 0) local = fma(row[e >> p.log2_categories], p.weights[e >> p.log2_categories], local);
            return reduce.Sum(local);
          };
          // log of the unnormalised posterior per GPCSP, folded with LogAdd in index order;
          // kept for the second pass when the scratch holds the range (every thread writes
          // the same bits)
          const bool keep = length <= plan.scratch;
          double log_norm = 0.0;
          for (int g0 = start; g0 < stop; g0 += 4) {
            // (four rows per exchange; every sum is reduced in the same order as one at a time)
            double sums[4] = {0.0, 0.0, 0.0, 0.0};
            if (!use_hybrid) {
#pragma unroll
              for (int u = 0; u < 4; u++) {
                if (g0 + u < stop) {
                  const double* row = p.log_likelihoods + static_cast<size_t>(g0 + u) * P;
                  // (a pattern's values are read by the thread that wrote them: its category-0 lane)
                  for (int64_t e = first; e < E; e += stride)
                    if (my_category == 0) sums[u] = fma(row[e >> p.log2_categories], p.weights[e >> p.log2_categories], sums[u]);
                }
              }
              reduce.Sums(sums);
            }
#pragma unroll
            for (int u = 0; u < 4; u++) {
              const int g = g0 + u;
              if (g < stop) {
                const double value = (use_hybrid ? p.hybrid[g] : sums[u]) + log(q[g]);
                if (keep && threadIdx.x == 0) scratch[g - start] = value;
                log_norm = (g == start) ? value : LogAdd(log_norm, value);
              }
            }
          }
          if (keep) {
            // every thread must have read q[start..stop) before anyone overwrites it
            reduce.Barrier();
            for (int g = start + static_cast<int>(threadIdx.x); g < stop; g += blockDim.x)
              set_q(g, exp(scratch[g - start] - log_norm));
            __syncthreads();
          } else {
            // too long for the scratch: the second pass recomputes the same values (identical bits)
            for (int g = start; g < stop; g++) {
              const double updated = exp((use_hybrid ? p.hybrid[g] : row_sum(g)) + log(q[g]) - log_norm);
              reduce.Barrier();
              if (threadIdx.x == 0) set_q(g, updated);
              __syncthreads();
            }
          }
        }
        pc += 3;
        break;
      }
      case SBNB_GP_RESET_MARGINAL_LIKELIHOOD: {  // gp_engine.cpp:84-86
        // (by the thread that accumulates the pattern in IncrementMarginalLikelihood: its category-0 lane)
        for (int64_t e = first; e < E; e += stride)
          if (my_category == 0) p.log_marginal[e >> p.log2_categories] = -INFINITY;
        pc += 1;
        break;
      }
      case SBNB_GP_INCREMENT_MARGINAL: {  // gp_engine.cpp:88-109
        const int stationary = program[pc + 1], rootsplit = program[pc + 2], leafward = program[pc + 3];
        if (counts[stationary] != 0) {
          fault(kGpFaultRescaledStationary, pc);
          return;
        }
        const double count_log = static_cast<double>(counts[leafward]) * p.log_threshold;
        const double log_prior = log(q[rootsplit]);
        double* row = p.log_likelihoods + static_cast<size_t>(rootsplit) * P;
        for (int64_t base = first - lane; base < E; base += stride) {  // (warp-uniform: the category sum shuffles)
          const int64_t e = base + lane;
          double a[4] = {1.0, 1.0, 1.0, 1.0}, b[4] = {1.0, 1.0, 1.0, 1.0};
          if (e < E) {
            LoadState(plv(stationary), e, a);
            LoadState(plv(leafward), e, b);
          }
          const double site = category_sum(fma(a[3], b[3], fma(a[2], b[2], fma(a[1], b[1], a[0] * b[0]))) * my_proportion);
          if (e < E && my_category == 0) {
            const int64_t k = e >> p.log2_categories;
            const double value = log(site) + count_log;
            p.log_marginal[k] = LogAdd(p.log_marginal[k], value);
            row[k] = value - log_prior;
          }
        }
        pc += 4;
        break;
      }
      case SBNB_GP_PREP_FOR_MARGINALIZATION: {  // gp_engine.cpp:155-165
        const int dest = program[pc + 1], src_count = program[pc + 2];
        int minimum = counts[program[pc + 3]];
        for (int i = 1; i < src_count; i++) minimum = min(minimum, counts[program[pc + 3 + i]]);
        set_count(dest, minimum);
        pc += 3 + src_count;
        break;
      }
      default:
        fault(kGpFaultBadProgram, pc);
        return;
    }
  }
}
// The interpreter's launch.  With p.cluster_exchange the grid is ONE thread-block cluster (at most
// kGpClusterBlocks CTAs) and the cross-CTA reductions travel through distributed shared memory:
// a CTA's words live in shared memory (zeroed here), every CTA of the cluster has started before
// anyone stores into a peer (first cluster barrier), and no CTA exits while a peer might still
// store into it (second cluster barrier: every path of the body, faults and time-outs included,
// returns here).
template <bool SINGLE>
__global__ void __launch_bounds__(kGpMaxBlockThreads, 1) GpInterpretKernel(const GpParams p, const GpSmemPlan plan) {
  __shared__ __align__(8) unsigned long long cluster_words[2][kGpClusterBlocks][2 * kGpReduceValues];
  if (p.cluster_exchange) {
    for (int w = threadIdx.x; w < 2 * kGpClusterBlocks * 2 * kGpReduceValues; w += blockDim.x)
      (&cluster_words[0][0][0])[w] = 0;
    asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
  }
  GpInterpretBody<SINGLE>(p, plan, cluster_words);
  if (p.cluster_exchange)
    asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}


// GetLogMarginalLikelihood, GetPerGPCSPLogLikelihoods: rows[r] . weights, one block per row.
__global__ void GpWeightedRowSumsKernel(const double* rows, const double* weights, int64_t P, double* out) {
  __shared__ double smem[32];
  const double* row = rows + static_cast<size_t>(blockIdx.x) * P;
  double local = 0.0;
  for (int64_t k = threadIdx.x; k < P; k += blockDim.x) local = fma(row[k], weights[k], local);
#pragma unroll
  for (int m = 16; m >= 1; m >>= 1) local += __shfl_xor_sync(0xffffffffu, local, m);
  if ((threadIdx.x & 31) == 0) smem[threadIdx.x >> 5] = local;
  __syncthreads();
  if (threadIdx.x == 0) {
    double total = 0.0;
    for (int w = 0; w < (blockDim.x + 31) / 32; w++) total += smem[w];
    out[blockIdx.x] = total;
  }
}

// LogLikelihoodAndDerivative (gp_engine.cpp:244-266), one block.  With rate categories the site
// likelihood is sum_c p_c r_c^T P(r_c t) l_c and its derivative in t sum_c p_c r_c r_c^T Q P(r_c t) l_c.
__global__ void GpLogLikelihoodAndDerivativeKernel(const GpParams p, int leafward, int rootward, int gpcsp,
                                                   double* out) {
  __shared__ double smem[32][2];
  const int64_t P = p.pattern_count;
  const int C = p.categories;
  const double t = p.branch_lengths[gpcsp];
  const double count_log = static_cast<double>(p.counts[rootward]) * p.log_threshold +
                           static_cast<double>(p.counts[leafward]) * p.log_threshold;
  const double* rootward_plv = p.plvs + static_cast<size_t>(rootward) * P * C * 4;
  const double* leafward_plv = p.plvs + static_cast<size_t>(leafward) * P * C * 4;
  double log_likelihood = 0.0, derivative = 0.0;
  for (int64_t k = threadIdx.x; k < P; k += blockDim.x) {
    double likelihood = 0.0, slope = 0.0;
    for (int c = 0; c < C; c++) {
      double m[16], dm[16], r[4], l[4];
      TransitionMatrix(p, t * p.rates[c], false, m);
      TransitionMatrix(p, t * p.rates[c], true, dm);
      LoadState(rootward_plv, k * C + c, r);
      LoadState(leafward_plv, k * C + c, l);
      likelihood += p.proportions[c] * Bilinear(r, m, l);
      slope += p.proportions[c] * p.rates[c] * Bilinear(r, dm, l);
    }
    log_likelihood = fma(p.weights[k], log(likelihood) + count_log, log_likelihood);
    derivative = fma(p.weights[k], slope / likelihood, derivative);
  }
#pragma unroll
  for (int s = 16; s >= 1; s >>= 1) {
    log_likelihood += __shfl_xor_sync(0xffffffffu, log_likelihood, s);
    derivative += __shfl_xor_sync(0xffffffffu, derivative, s);
  }
  if ((threadIdx.x & 31) == 0) smem[threadIdx.x >> 5][0] = log_likelihood, smem[threadIdx.x >> 5][1] = derivative;
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0.0, b = 0.0;
    for (int w = 0; w < (blockDim.x + 31) / 32; w++) a += smem[w][0], b += smem[w][1];
    out[0] = a;
    out[1] = b;
  }
}

__global__ void GpTransitionMatrixKernel(const GpParams p, double branch_length, double* out) {
  double m[16];
  TransitionMatrix(p, branch_length, false, m);
  if (threadIdx.x == 0)
    for (int i = 0; i < 16; i++) out[i] = m[i];
}

// CalculateQuartetHybridLikelihoods (gp_engine.cpp:396-452): one block per
// (rootward, sister, rotated, sorted) combination; every combination recomputes
// the short chain of 4 x 4 products for its patterns instead of materialising
// the reference's four scratch PLVs.
struct GpQuartetParams {
  const int32_t* tips;  // records of 3 int32: rootward, then sister, rotated, sorted lists
  int32_t rootward_count, sister_count, rotated_count, sorted_count;
  int32_t central_gpcsp;
  const double* unconditional_node_probabilities;
  const double* inverted_sbn_prior;
};
__global__ void GpQuartetKernel(const GpParams p, const GpQuartetParams qp, double* out, int32_t* status) {
  __shared__ double smem[32];
  const int64_t P = p.pattern_count;
  int index = blockIdx.x;
  const int sorted_i = index % qp.sorted_count;
  index /= qp.sorted_count;
  const int rotated_i = index % qp.rotated_count;
  index /= qp.rotated_count;
  const int sister_i = index % qp.sister_count;
  const int rootward_i = index / qp.sister_count;
  const int32_t* rootward = qp.tips + 3 * rootward_i;
  const int32_t* sister = qp.tips + 3 * (qp.rootward_count + sister_i);
  const int32_t* rotated = qp.tips + 3 * (qp.rootward_count + qp.sister_count + rotated_i);
  const int32_t* sorted = qp.tips + 3 * (qp.rootward_count + qp.sister_count + qp.rotated_count + sorted_i);
  if (p.counts[rootward[1]] != 0 || p.counts[sister[1]] != 0 || p.counts[rotated[1]] != 0 ||
      p.counts[sorted[1]] != 0) {
    if (threadIdx.x == 0) status[0] = 1;  // "Rescaling not implemented in CalculateQuartetHybridLikelihoods."
    return;
  }
  const int C = p.categories;
  double m_rootward[16], m_sister[16], m_central[16], m_rotated[16], m_sorted[16];
  auto matrices_of = [&](int c) {
    const double rate = p.rates[c];
    TransitionMatrix(p, p.branch_lengths[rootward[2]] * rate, false, m_rootward);
    TransitionMatrix(p, p.branch_lengths[sister[2]] * rate, false, m_sister);
    TransitionMatrix(p, p.branch_lengths[qp.central_gpcsp] * rate, false, m_central);
    TransitionMatrix(p, p.branch_lengths[rotated[2]] * rate, false, m_rotated);
    TransitionMatrix(p, p.branch_lengths[sorted[2]] * rate, false, m_sorted);
  };
  if (C == 1) matrices_of(0);
  auto apply = [](const double (&m)[16], const double (&x)[4], double (&y)[4]) {
#pragma unroll
    for (int i = 0; i < 4; i++)
      y[i] = fma(m[i * 4 + 3], x[3], fma(m[i * 4 + 2], x[2], fma(m[i * 4 + 1], x[1], m[i * 4] * x[0])));
  };
  const double log_rootward_tip_prior = log(qp.unconditional_node_probabilities[rootward[0]]);
  const size_t plv_doubles = static_cast<size_t>(P) * C * 4;
  double local = 0.0;
  for (int64_t k = threadIdx.x; k < P; k += blockDim.x) {
    double likelihood = 0.0;
    for (int c = 0; c < C; c++) {
      if (C > 1) matrices_of(c);  // (rate categories: not the reference's path; the matrices are per category)
      const int64_t e = k * C + c;
      double x[4], root_plv[4], y[4], r_s[4], q_s[4], r_sorted[4];
      LoadState(p.plvs + rootward[1] * plv_doubles, e, x);
      apply(m_rootward, x, root_plv);
      LoadState(p.plvs + sister[1] * plv_doubles, e, x);
      apply(m_sister, x, y);
#pragma unroll
      for (int i = 0; i < 4; i++) r_s[i] = root_plv[i] * y[i];
      apply(m_central, r_s, q_s);
      LoadState(p.plvs + rotated[1] * plv_doubles, e, x);
      apply(m_rotated, x, y);
#pragma unroll
      for (int i = 0; i < 4; i++) r_sorted[i] = q_s[i] * y[i];
      LoadState(p.plvs + sorted[1] * plv_doubles, e, x);
      likelihood += p.proportions[c] * Bilinear(r_sorted, m_sorted, x);
    }
    local = fma(p.weights[k], log(likelihood) - log_rootward_tip_prior, local);
  }
#pragma unroll
  for (int s = 16; s >= 1; s >>= 1) local += __shfl_xor_sync(0xffffffffu, local, s);
  if ((threadIdx.x & 31) == 0) smem[threadIdx.x >> 5] = local;
  __syncthreads();
  if (threadIdx.x == 0) {
    double total = 0.0;
    for (int w = 0; w < (blockDim.x + 31) / 32; w++) total += smem[w];
    const double non_sequence = log(qp.inverted_sbn_prior[rootward[2]] * p.q[sister[2]] * p.q[rotated[2]] *
                                    p.q[sorted[2]]);
    out[blockIdx.x] = non_sequence + total;
  }
}

const char* FaultMessage(int code) {
  switch (code) {
    case kGpFaultDestRescaling:
      return "dest_ rescaling too large in IncrementWithWeightedEvolvedPLV";
    case kGpFaultRescaledStationary:
      return "Surprise! Rescaled stationary distribution in IncrementMarginalLikelihood";
    case kGpFaultNotFinite:
      return "Multiply dest_ is not finite";
    case kGpFaultNegative:
      return "PLV with negative entry passed to RescalePLVIfNeeded";
    case kGpFaultBarrierTimeout:
      return "libsbn_b200: a thread block of the GP interpreter never reached a reduction (device barrier timed out)";
    default:
      return "Malformed GP operation program";
  }
}

}  // namespace

}  // namespace sbnb

using namespace sbnb;

namespace {

// The op program as the interpreter runs it.  The reference's schedules are long
// sequences in which most neighbours do not depend on each other (DS1 DAG: the 1410 ops that
// populate the PLVs form 66 dependency levels), and on the device an op is a chain of
// latencies, not of arithmetic.  So the program is re-ordered by dependency level -- an op's
// level is one more than the highest level among the ops it must follow (read after write,
// write after write, write after read, over PLVs, rescaling counts, q, branch lengths,
// log-likelihood rows and the log-marginal vector) -- and, inside a level, by kind; runs of
// one kind become batches whose loads the interpreter issues together and whose reductions
// share one exchange.  Ops of one level are independent, so every value is computed by the
// same arithmetic in the same order as in the reference's sequence: bit-identical results.
struct CompiledProgram {
  std::vector<int32_t> source;  // the caller's words (cache key)
  std::vector<int32_t> words;   // what the device runs
  std::vector<std::pair<int32_t, int32_t>> origin;  // (word offset in `words`, word offset in `source`) per op
  DeviceArray<int32_t> device;
  uint64_t last_used = 0;
};

}  // namespace

struct sbnb_gp_engine {
  int device = 0;
  int sm_count = 0;
  int32_t taxon_count = 0, plv_count = 0, gpcsp_count = 0, node_count = 0;
  int64_t pattern_count = 0, site_count = 0;
  int blocks = 1, threads = 32;
  bool no_cluster = false;  // SBNB_GP_NO_CLUSTER: multi-CTA launches use the L2 mailboxes even when a cluster would do
  cudaStream_t stream = nullptr;
  cudaEvent_t begin = nullptr, end = nullptr;
  GpParams params{};
  DeviceArray<double> plvs, branch_lengths, q, hybrid, log_likelihoods, log_marginal, weights, exchange, scalars,
      node_probabilities, inverted_prior;
  DeviceArray<double> matrix_cache;
  std::vector<uint8_t> host_tips;  // [taxon][pattern], for re-initialising the PLVs when the site model changes
  bool tip_masks = false;          // host_tips are nucleotide masks (SBNB_TIPS_NUCLEOTIDE_MASKS), not states
  DeviceArray<int32_t> counts, program, status, tips;
  // programs seen before (the reference regenerates the same few schedules call after call)
  std::vector<std::unique_ptr<CompiledProgram>> compiled;
  uint64_t program_clock = 0;
  GpSmemPlan plan{};  // the per-engine part (matrices, counts, scratch); the program is fitted per launch
  bool has_node_probabilities = false;
  int64_t launch_count = 0;
  double last_kernel_ms = 0.0;

  ~sbnb_gp_engine() {
    if (begin) cudaEventDestroy(begin);
    if (end) cudaEventDestroy(end);
    if (stream) cudaStreamDestroy(stream);
  }
};

namespace {

void CompileProgram(int32_t plv_count, int32_t gpcsp_count, const int32_t* program, int64_t word_count,
                    CompiledProgram* out);
void SetCategories(sbnb_gp_engine* e, int categories, const double* rates, const double* proportions);

void Bind(sbnb_gp_engine* e) { SBNB_CUDA(cudaSetDevice(e->device)); }

void CopyOut(sbnb_gp_engine* e, double* host, const double* device, size_t count) {
  SBNB_CUDA(cudaMemcpyAsync(host, device, count * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
  SBNB_CUDA(cudaStreamSynchronize(e->stream));
}

struct GpShape {
  int32_t plv_count, gpcsp_count;
};
void CheckPlv(const GpShape& e, int index) { Require(index >= 0 && index < e.plv_count, "PLV index out of range."); }
void CheckGpcsp(const GpShape& e, int index) {
  Require(index >= 0 && index < e.gpcsp_count, "GPCSP index out of range.");
}
void CheckPlv(const sbnb_gp_engine* e, int index) { CheckPlv(GpShape{e->plv_count, e->gpcsp_count}, index); }
void CheckGpcsp(const sbnb_gp_engine* e, int index) { CheckGpcsp(GpShape{e->plv_count, e->gpcsp_count}, index); }

// Host-side validation of a program: every index in range, records complete.
void ValidateProgram(const GpShape& e, const int32_t* program, int64_t words) {
  int64_t pc = 0;
  while (pc < words) {
    const int opcode = program[pc];
    auto need = [&](int64_t count) { Require(pc + count <= words, "Truncated GP operation record."); };
    switch (opcode) {
      case SBNB_GP_ZERO_PLV:
        need(2);
        CheckPlv(e, program[pc + 1]);
        pc += 2;
        break;
      case SBNB_GP_SET_TO_STATIONARY:
        need(3);
        CheckPlv(e, program[pc + 1]);
        CheckGpcsp(e, program[pc + 2]);
        pc += 3;
        break;
      case SBNB_GP_INCREMENT_WITH_EVOLVED:
        need(4);
        CheckPlv(e, program[pc + 1]);
        CheckGpcsp(e, program[pc + 2]);
        CheckPlv(e, program[pc + 3]);
        pc += 4;
        break;
      case SBNB_GP_MULTIPLY:
        need(4);
        for (int i = 1; i <= 3; i++) CheckPlv(e, program[pc + i]);
        pc += 4;
        break;
      case SBNB_GP_LIKELIHOOD:
        need(4);
        CheckGpcsp(e, program[pc + 1]);
        CheckPlv(e, program[pc + 2]);
        CheckPlv(e, program[pc + 3]);
        pc += 4;
        break;
      case SBNB_GP_OPTIMIZE_BRANCH_LENGTH:
        need(4);
        CheckPlv(e, program[pc + 1]);
        CheckPlv(e, program[pc + 2]);
        CheckGpcsp(e, program[pc + 3]);
        pc += 4;
        break;
      case SBNB_GP_UPDATE_SBN_PROBABILITIES:
        need(3);
        Require(program[pc + 1] >= 0 && program[pc + 1] <= program[pc + 2] && program[pc + 2] <= e.gpcsp_count,
                "UpdateSBNProbabilities range out of bounds.");
        pc += 3;
        break;
      case SBNB_GP_RESET_MARGINAL_LIKELIHOOD:
        pc += 1;
        break;
      case SBNB_GP_INCREMENT_MARGINAL:
        need(4);
        CheckPlv(e, program[pc + 1]);
        CheckGpcsp(e, program[pc + 2]);
        CheckPlv(e, program[pc + 3]);
        pc += 4;
        break;
      case SBNB_GP_PREP_FOR_MARGINALIZATION: {
        need(3);
        CheckPlv(e, program[pc + 1]);
        const int count = program[pc + 2];
        Require(count > 0, "Empty src_vector in PrepForMarginalization");
        need(3 + count);
        for (int i = 0; i < count; i++) CheckPlv(e, program[pc + 3 + i]);
        pc += 3 + count;
        break;
      }
      default:
        Fail(SBNB_ERR_INVALID_ARGUMENT, "Unknown GP opcode " + std::to_string(opcode) + ".");
    }
  }
}

// Where in the caller's program the op at `offset` of the compiled program came from.
int32_t OriginalOffset(const CompiledProgram& compiled, int32_t offset) {
  for (const auto& entry : compiled.origin)
    if (entry.first == offset) return entry.second;
  return offset;
}

void WeightedRowSums(sbnb_gp_engine* e, const double* rows, int row_count, double* host_out) {
  if (row_count == 0) return;
  e->scalars.Reserve(std::max<size_t>(row_count, 64));
  GpWeightedRowSumsKernel<<<row_count, 256, 0, e->stream>>>(rows, e->weights.get(), e->pattern_count,
                                                            e->scalars.get());
  SBNB_CUDA(cudaGetLastError());
  e->launch_count++;
  CopyOut(e, host_out, e->scalars.get(), row_count);
}

std::vector<int32_t> PackTips(const int32_t* a, int na, const int32_t* b, int nb, const int32_t* c, int nc,
                              const int32_t* d, int nd) {
  std::vector<int32_t> out;
  auto append = [&](const int32_t* tips, int count) { out.insert(out.end(), tips, tips + 3 * count); };
  append(a, na), append(b, nb), append(c, nc), append(d, nd);
  return out;
}

void QuartetLikelihoods(sbnb_gp_engine* e, int32_t central, const int32_t* rootward, int32_t rootward_count,
                        const int32_t* sister, int32_t sister_count, const int32_t* rotated, int32_t rotated_count,
                        const int32_t* sorted, int32_t sorted_count, std::vector<double>* out) {
  Bind(e);
  CheckGpcsp(e, central);
  Require(e->has_node_probabilities,
          "Quartet hybrid likelihoods need unconditional_node_probabilities and inverted_sbn_prior.");
  Require(rootward_count >= 0 && sister_count >= 0 && rotated_count >= 0 && sorted_count >= 0,
          "Negative tip count.");
  const int64_t total = static_cast<int64_t>(rootward_count) * sister_count * rotated_count * sorted_count;
  out->assign(total, 0.0);
  if (total == 0) return;
  Require((rootward && sister && rotated && sorted), "NULL tip list.");
  const std::vector<int32_t> tips =
      PackTips(rootward, rootward_count, sister, sister_count, rotated, rotated_count, sorted, sorted_count);
  for (size_t i = 0; i < tips.size(); i += 3) {
    Require(tips[i] >= 0 && tips[i] < e->node_count, "Quartet tip node id out of range.");
    CheckPlv(e, tips[i + 1]);
    CheckGpcsp(e, tips[i + 2]);
  }
  e->tips.Upload(tips.data(), tips.size(), e->stream);
  e->scalars.Reserve(std::max<size_t>(total, 64));
  SBNB_CUDA(cudaMemsetAsync(e->status.get(), 0, 2 * sizeof(int32_t), e->stream));
  GpQuartetParams qp{e->tips.get(),  rootward_count, sister_count, rotated_count, sorted_count, central,
                     e->node_probabilities.get(), e->inverted_prior.get()};
  GpQuartetKernel<<<static_cast<unsigned>(total), 256, 0, e->stream>>>(e->params, qp, e->scalars.get(),
                                                                      e->status.get());
  SBNB_CUDA(cudaGetLastError());
  e->launch_count++;
  int32_t status[2] = {0, 0};
  SBNB_CUDA(cudaMemcpyAsync(status, e->status.get(), sizeof(status), cudaMemcpyDeviceToHost, e->stream));
  CopyOut(e, out->data(), e->scalars.get(), total);
  if (status[0] != 0)
    Fail(SBNB_ERR_GP_ASSERT, "Rescaling not implemented in CalculateQuartetHybridLikelihoods.");
}

// Everything that depends on the number of rate categories: the launch shape (one thread per
// (pattern, category)), the shared-memory plan, the PLVs -- zeroed, tips re-initialised (one-hot /
// all-ones gaps, gp_engine.cpp:268-286, the same in every category) -- and the rescaling counts.
void SetCategories(sbnb_gp_engine* e, int categories, const double* rates, const double* proportions) {
  Bind(e);
  SBNB_CUDA(cudaStreamSynchronize(e->stream));
  const int64_t P = e->pattern_count, E = P * categories;
  const size_t gpcsps = std::max(e->gpcsp_count, 1);
  // One (pattern, category) per thread while the resident CTAs can hold them (an op is then a
  // short dependency chain per thread, and the CTAs share the fp64 work of the SMs they sit
  // on); strided beyond that.
  static const int forced_threads = EnvInt("SBNB_GP_THREADS", 0), forced_blocks = EnvInt("SBNB_GP_BLOCKS", 0);
  e->no_cluster = EnvInt("SBNB_GP_NO_CLUSTER", 0) != 0;
  const int max_blocks = std::min(kGpMaxGridBlocks, e->sm_count);
  e->threads = E <= static_cast<int64_t>(kGpBlockThreads) * max_blocks
                   ? static_cast<int>(std::min<int64_t>((E + 31) / 32 * 32, kGpBlockThreads))
                   : kGpGridBlockThreads;
  if (forced_threads > 0) e->threads = std::min(std::max(forced_threads / 32 * 32, 32), kGpMaxBlockThreads);
  // Shared-memory plan, in the order of what an op touches most: the transition matrices
  // (+ q), the per-warp rescaling counts, a scratch for UpdateSBNProbabilities; the op
  // program takes what is left, launch by launch.
  SBNB_CUDA(cudaFuncSetAttribute(GpInterpretKernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 static_cast<int>(kGpSmemBudget)));
  SBNB_CUDA(cudaFuncSetAttribute(GpInterpretKernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 static_cast<int>(kGpSmemBudget)));
  {
    GpSmemPlan plan{};
    size_t used = 0;
    const size_t matrix_bytes = gpcsps * (16 * categories + 1) * sizeof(double);
    plan.matrices = used + matrix_bytes <= kGpSmemBudget / 2;
    if (plan.matrices) used += matrix_bytes;
    plan.scratch = kGpScratchDoubles;
    used += plan.scratch * sizeof(double);
    const size_t count_bytes = static_cast<size_t>(e->threads / 32) * e->plv_count * sizeof(int32_t);
    plan.counts = used + count_bytes <= kGpSmemBudget * 3 / 4;
    if (plan.counts) used += count_bytes;
    plan.bytes = used;
    e->plan = plan;
  }
  {
    int per_sm = 0;
    SBNB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, GpInterpretKernel<false>, e->threads, kGpSmemBudget));
    const int64_t resident = std::min<int64_t>(static_cast<int64_t>(std::max(per_sm, 1)) * e->sm_count, max_blocks);
    e->blocks = static_cast<int>(std::min<int64_t>((E + e->threads - 1) / e->threads, resident));
    if (forced_blocks > 0) e->blocks = std::min(e->blocks, forced_blocks);
  }
  {
    const size_t plv_doubles = static_cast<size_t>(e->plv_count) * E * 4;
    e->plvs.Reserve(plv_doubles);
    SBNB_CUDA(cudaMemsetAsync(e->plvs.get(), 0, plv_doubles * sizeof(double), e->stream));
    std::vector<double> tips(static_cast<size_t>(e->taxon_count) * E * 4, 0.0);
    for (int taxon = 0; taxon < e->taxon_count; taxon++)
      for (int64_t k = 0; k < P; k++) {
        const uint8_t symbol = e->host_tips[static_cast<size_t>(taxon) * P + k];
        for (int c = 0; c < categories; c++) {
          double* x = tips.data() + (static_cast<size_t>(taxon) * E + k * categories + c) * 4;
          if (e->tip_masks) {
            for (int s = 0; s < 4; s++) x[s] = (symbol >> s) & 1 ? 1.0 : 0.0;  // 15: the all-ones gap
          } else if (symbol == 4) {
            x[0] = x[1] = x[2] = x[3] = 1.0;
          } else if (symbol < 4) {
            x[symbol] = 1.0;
          }  // symbols > 4 leave the column zero, as the reference does
        }
      }
    SBNB_CUDA(cudaMemcpyAsync(e->plvs.get(), tips.data(), tips.size() * sizeof(double), cudaMemcpyHostToDevice,
                              e->stream));
    SBNB_CUDA(cudaStreamSynchronize(e->stream));
  }
  const size_t count_copies = static_cast<size_t>(e->blocks) * (kGpMaxBlockThreads / 32);
  e->counts.Reserve(count_copies * e->plv_count);
  SBNB_CUDA(cudaMemsetAsync(e->counts.get(), 0, count_copies * e->plv_count * sizeof(int32_t), e->stream));
  e->exchange.Reserve(static_cast<size_t>(2) * e->blocks * 2 * kGpReduceValues);  // 8-byte words
  e->matrix_cache.Reserve(gpcsps * 16 * categories);
  SBNB_CUDA(cudaStreamSynchronize(e->stream));
  GpParams& p = e->params;
  p.pattern_count = P;
  p.plv_count = e->plv_count;
  p.gpcsp_count = e->gpcsp_count;
  p.categories = categories;
  p.log2_categories = 0;
  while ((1 << p.log2_categories) < categories) p.log2_categories++;
  for (int c = 0; c < kGpMaxCategories; c++) {
    p.rates[c] = c < categories ? rates[c] : 1.0;
    p.proportions[c] = c < categories ? proportions[c] : 0.0;
  }
  p.plvs = e->plvs.get();
  p.counts = e->counts.get();
  p.exchange = e->exchange.get();
  p.matrix_cache = e->matrix_cache.get();
}

void CompileProgram(int32_t plv_count, int32_t gpcsp_count, const int32_t* program, int64_t word_count,
                    CompiledProgram* out) {
  // ---- pass 1: the caller's records; runs of IncrementWithWeightedEvolvedPLV into one PLV
  // (the reference emits a node's increments side by side, gp_dag.cpp:264-290) become ONE
  // record -- SBNB_GP_INTERNAL_EVOLVE_SUM: dest, n, (gpcsp, src) x n, at most kGpChain sources --
  // that loads every source at once and adds them in the reference's order; and when the PLV
  // was last written by a ZeroPLV nobody has read since, the sum starts from 0 without
  // loading it ("fresh") and that ZeroPLV only clears the rescaling count: 0 + x = x exactly.
  struct Op {
    int32_t at;                 // word offset in the caller's program (of its first record)
    int32_t opcode, level = 0;
    std::vector<int32_t> words;  // the record as the device sees it (word 0 without its batch length)
  };
  static const bool fusing = EnvInt("SBNB_GP_FUSE", 1) != 0;
  std::vector<Op> ops;
  {
    std::vector<int32_t> zeroed_by(plv_count, -1);  // index in `ops` of an unread ZeroPLV of the PLV, or -1
    auto touch = [&](int32_t plv_index) { zeroed_by[plv_index] = -1; };
    int64_t pc = 0;
    while (pc < word_count) {
      const int32_t* w = program + pc;
      const int opcode = w[0];
      Op op;
      op.at = static_cast<int32_t>(pc);
      op.opcode = opcode;
      int32_t size = 0;
      switch (opcode) {
        case SBNB_GP_ZERO_PLV:
          size = 2;
          break;
        case SBNB_GP_SET_TO_STATIONARY:
          size = 3;
          touch(w[1]);
          break;
        case SBNB_GP_INCREMENT_WITH_EVOLVED: {
          size = 4;
          if (!fusing) {
            touch(w[1]), touch(w[3]);
            break;
          }
          const int32_t dest = w[1];
          std::vector<std::pair<int32_t, int32_t>> sources;  // (gpcsp, src)
          int64_t next = pc;
          while (next < word_count && program[next] == SBNB_GP_INCREMENT_WITH_EVOLVED && program[next + 1] == dest &&
                 program[next + 3] != dest && static_cast<int>(sources.size()) < kGpChain) {
            sources.emplace_back(program[next + 2], program[next + 3]);
            next += 4;
          }
          if (sources.empty()) {  // (dest == src: left as it is)
            touch(w[1]);
            break;
          }
          const bool fresh = zeroed_by[dest] >= 0;
          if (fresh) ops[zeroed_by[dest]].words[0] |= kGpFlag;  // that ZeroPLV: rescaling count only
          touch(dest);
          for (const auto& source : sources) touch(source.second);
          if (sources.size() == 1) {
            op.words = {SBNB_GP_INCREMENT_WITH_EVOLVED | (fresh ? kGpFlag : 0), dest, sources[0].first, sources[0].second};
          } else {
            op.opcode = SBNB_GP_INTERNAL_EVOLVE_SUM;
            op.words = {SBNB_GP_INTERNAL_EVOLVE_SUM | (fresh ? kGpFlag : 0), dest, static_cast<int32_t>(sources.size())};
            for (const auto& source : sources) op.words.insert(op.words.end(), {source.first, source.second});
          }
          size = static_cast<int32_t>(next - pc);
          break;
        }
        case SBNB_GP_MULTIPLY:
          size = 4;
          touch(w[1]), touch(w[2]), touch(w[3]);
          break;
        case SBNB_GP_LIKELIHOOD:
        case SBNB_GP_INCREMENT_MARGINAL:
          size = 4;
          touch(opcode == SBNB_GP_LIKELIHOOD ? w[2] : w[1]), touch(w[3]);
          break;
        case SBNB_GP_OPTIMIZE_BRANCH_LENGTH:
          size = 4;
          touch(w[1]), touch(w[2]);
          break;
        case SBNB_GP_UPDATE_SBN_PROBABILITIES:
          size = 3;
          break;
        case SBNB_GP_RESET_MARGINAL_LIKELIHOOD:
          size = 1;
          break;
        case SBNB_GP_PREP_FOR_MARGINALIZATION:
          size = 3 + w[2];
          break;
        default:
          Fail(SBNB_ERR_INVALID_ARGUMENT, "Unknown GP opcode " + std::to_string(opcode) + ".");
      }
      if (op.words.empty()) op.words.assign(w, w + size);
      ops.push_back(std::move(op));
      if (opcode == SBNB_GP_ZERO_PLV && fusing) zeroed_by[w[1]] = static_cast<int32_t>(ops.size()) - 1;
      if (opcode == SBNB_GP_ZERO_PLV && !fusing) touch(w[1]);
      pc += size;
    }
  }

  // ---- pass 2: dependency levels.  Last writer's level, and the highest level among the
  // readers since, per resource.
  struct Track {
    int32_t written = -1, read = -1;
  };
  const size_t gpcsps = std::max(gpcsp_count, 1);
  std::vector<Track> plv(plv_count), count(plv_count), prior(gpcsps), length(gpcsps), row(gpcsps);
  Track marginal;
  int32_t level = 0;
  auto reads = [&](Track& t) { level = std::max(level, t.written + 1); };
  auto writes = [&](Track& t) { level = std::max(level, std::max(t.written, t.read) + 1); };
  auto did_read = [&](Track& t) { t.read = std::max(t.read, level); };
  auto did_write = [&](Track& t) {
    t.written = level;
    t.read = -1;
  };
  for (Op& op : ops) {
    const int32_t* w = op.words.data();
    const bool flagged = (w[0] & kGpFlag) != 0;
    level = 0;
    // two passes over the op's resources: find its level, then record it
    for (int pass = 0; pass < 2; pass++) {
      auto R = [&](Track& t) { pass == 0 ? reads(t) : did_read(t); };
      auto W = [&](Track& t) { pass == 0 ? writes(t) : did_write(t); };
      switch (op.opcode) {
        case SBNB_GP_ZERO_PLV:
          if (!flagged) W(plv[w[1]]);
          W(count[w[1]]);
          break;
        case SBNB_GP_SET_TO_STATIONARY:
          R(prior[w[2]]), W(plv[w[1]]), W(count[w[1]]);
          break;
        case SBNB_GP_INCREMENT_WITH_EVOLVED:
          R(plv[w[3]]), R(count[w[3]]), R(count[w[1]]), R(prior[w[2]]), R(length[w[2]]);
          if (!flagged) R(plv[w[1]]);
          W(plv[w[1]]);
          break;
        case SBNB_GP_INTERNAL_EVOLVE_SUM:
          for (int i = 0; i < w[2]; i++) R(plv[w[4 + 2 * i]]), R(count[w[4 + 2 * i]]), R(prior[w[3 + 2 * i]]), R(length[w[3 + 2 * i]]);
          R(count[w[1]]);
          if (!flagged) R(plv[w[1]]);
          W(plv[w[1]]);
          break;
        case SBNB_GP_MULTIPLY:
          R(plv[w[2]]), R(plv[w[3]]), R(count[w[2]]), R(count[w[3]]), W(plv[w[1]]), W(count[w[1]]);
          break;
        case SBNB_GP_LIKELIHOOD:
          R(plv[w[2]]), R(plv[w[3]]), R(count[w[2]]), R(count[w[3]]), R(length[w[1]]), W(row[w[1]]);
          break;
        case SBNB_GP_OPTIMIZE_BRANCH_LENGTH:
          R(plv[w[1]]), R(plv[w[2]]), R(count[w[1]]), R(count[w[2]]), R(length[w[3]]), W(length[w[3]]);
          break;
        case SBNB_GP_UPDATE_SBN_PROBABILITIES:
          for (int g = w[1]; g < w[2]; g++) R(row[g]), R(prior[g]);
          for (int g = w[1]; g < w[2]; g++) W(prior[g]);
          break;
        case SBNB_GP_RESET_MARGINAL_LIKELIHOOD:
          W(marginal);
          break;
        case SBNB_GP_INCREMENT_MARGINAL:
          R(plv[w[1]]), R(plv[w[3]]), R(count[w[1]]), R(count[w[3]]), R(prior[w[2]]), R(marginal), W(marginal),
              W(row[w[2]]);
          break;
        case SBNB_GP_PREP_FOR_MARGINALIZATION:
          for (int i = 0; i < w[2]; i++) R(count[w[3 + i]]);
          W(count[w[1]]);
          break;
      }
    }
    op.level = level;
  }
  // by level, then kind (the scalar-only PrepForMarginalization first), then the reference's order
  static const bool reorder = EnvInt("SBNB_GP_LEVELS", 1) != 0;
  if (reorder)
    std::stable_sort(ops.begin(), ops.end(), [](const Op& a, const Op& b) {
      if (a.level != b.level) return a.level < b.level;
      const int ka = a.opcode == SBNB_GP_PREP_FOR_MARGINALIZATION ? -1 : a.opcode;
      const int kb = b.opcode == SBNB_GP_PREP_FOR_MARGINALIZATION ? -1 : b.opcode;
      return ka < kb;
    });
  auto batch_limit = [](int opcode) {
    switch (opcode) {
      case SBNB_GP_ZERO_PLV:
      case SBNB_GP_SET_TO_STATIONARY:
        return 255;
      case SBNB_GP_INCREMENT_WITH_EVOLVED:
      case SBNB_GP_MULTIPLY:
      case SBNB_GP_LIKELIHOOD:
        return kGpBatch;
      default:
        return 1;
    }
  };
  static const bool batching = EnvInt("SBNB_GP_BATCH", 1) != 0;
  out->source.assign(program, program + word_count);
  out->words.clear();
  out->words.reserve(word_count);
  out->origin.clear();
  out->origin.reserve(ops.size());
  for (size_t i = 0; i < ops.size();) {
    size_t run = 1;
    const int limit = batching ? batch_limit(ops[i].opcode) : 1;
    while (reorder && i + run < ops.size() && static_cast<int>(run) < limit && ops[i + run].opcode == ops[i].opcode &&
           ops[i + run].level == ops[i].level)
      run++;
    for (size_t r = 0; r < run; r++) {
      const Op& op = ops[i + r];
      out->origin.emplace_back(static_cast<int32_t>(out->words.size()), op.at);
      out->words.insert(out->words.end(), op.words.begin(), op.words.end());
      if (r == 0) out->words[out->words.size() - op.words.size()] |= static_cast<int32_t>(run) << 8;
    }
    i += run;
  }
}

}  // namespace

extern "C" {

int sbnb_gp_create(int32_t taxon_count, int64_t pattern_count, const uint8_t* tip_states,
                   const double* pattern_weights, int64_t site_count, int32_t plv_count, int32_t gpcsp_count,
                   double rescaling_threshold, const double* sbn_prior,
                   const double* unconditional_node_probabilities, int32_t node_count,
                   const double* inverted_sbn_prior, int32_t device, sbnb_gp_engine** out) {
  return sbnb_gp_create_encoded(taxon_count, pattern_count, tip_states, SBNB_TIPS_STATES, pattern_weights,
                                site_count, plv_count, gpcsp_count, rescaling_threshold, sbn_prior,
                                unconditional_node_probabilities, node_count, inverted_sbn_prior, device, out);
}

int sbnb_gp_create_encoded(int32_t taxon_count, int64_t pattern_count, const uint8_t* tip_states, int32_t tip_encoding,
                           const double* pattern_weights, int64_t site_count, int32_t plv_count,
                           int32_t gpcsp_count, double rescaling_threshold, const double* sbn_prior,
                           const double* unconditional_node_probabilities, int32_t node_count,
                           const double* inverted_sbn_prior, int32_t device, sbnb_gp_engine** out) {
  return Guard([&] {
    Require(out != nullptr, "NULL output handle.");
    *out = nullptr;
    Require(taxon_count >= 1 && pattern_count >= 1, "Need at least 1 taxon and 1 site pattern.");
    Require(tip_states && pattern_weights, "NULL tip_states / pattern_weights.");
    Require(tip_encoding == SBNB_TIPS_STATES || tip_encoding == SBNB_TIPS_NUCLEOTIDE_MASKS, "Unknown tip encoding.");
    if (tip_encoding == SBNB_TIPS_NUCLEOTIDE_MASKS)
      for (size_t i = 0; i < static_cast<size_t>(taxon_count) * pattern_count; i++)
        if (tip_states[i] == 0 || tip_states[i] > 15)
          Fail(SBNB_ERR_INVALID_ARGUMENT, "Invalid nucleotide mask " + std::to_string(tip_states[i]) + " at taxon " +
                                              std::to_string(i / pattern_count) + ", pattern " +
                                              std::to_string(i % pattern_count) + " (masks are 1..15).");
    Require(plv_count >= taxon_count, "plv_count must cover the taxa (6 PLVs per DAG node).");
    Require(gpcsp_count >= 0, "Negative GPCSP count.");
    Require(rescaling_threshold > 0.0 && rescaling_threshold < 1.0, "rescaling_threshold must be in (0, 1).");
    int device_count = 0;
    if (cudaGetDeviceCount(&device_count) != cudaSuccess || device_count < 1) {
      cudaGetLastError();
      Fail(SBNB_ERR_NO_DEVICE, "No CUDA device available: libsbn_b200 has no CPU fallback (cudaGetDeviceCount).");
    }
    Require(device >= 0 && device < device_count, "CUDA device ordinal out of range.");
    auto e = std::make_unique<sbnb_gp_engine>();
    e->device = device;
    Bind(e.get());
    cudaDeviceProp prop{};
    SBNB_CUDA(cudaGetDeviceProperties(&prop, device));
    e->sm_count = prop.multiProcessorCount;
    e->taxon_count = taxon_count;
    e->pattern_count = pattern_count;
    e->site_count = site_count;
    e->plv_count = plv_count;
    e->gpcsp_count = gpcsp_count;
    e->node_count = node_count;
    SBNB_CUDA(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
    SBNB_CUDA(cudaEventCreate(&e->begin));
    SBNB_CUDA(cudaEventCreate(&e->end));
    const int64_t P = pattern_count;
    const size_t gpcsps = std::max(gpcsp_count, 1);
    e->host_tips.assign(tip_states, tip_states + static_cast<size_t>(taxon_count) * P);
    e->tip_masks = tip_encoding == SBNB_TIPS_NUCLEOTIDE_MASKS;
    const double unit = 1.0;
    SetCategories(e.get(), 1, &unit, &unit);
    e->weights.Upload(pattern_weights, P, e->stream);
    std::vector<double> branch_lengths(gpcsps, 0.1);  // default_branch_length_, gp_engine.hpp:84
    e->branch_lengths.Upload(branch_lengths.data(), gpcsps, e->stream);
    std::vector<double> q(gpcsps, 0.0);
    if (sbn_prior) std::copy(sbn_prior, sbn_prior + gpcsp_count, q.begin());
    e->q.Upload(q.data(), gpcsps, e->stream);
    std::vector<double> minus_infinity(std::max<size_t>(gpcsps, P), -INFINITY);
    e->hybrid.Upload(minus_infinity.data(), gpcsps, e->stream);
    e->log_marginal.Upload(minus_infinity.data(), P, e->stream);
    e->log_likelihoods.Reserve(gpcsps * P);
    SBNB_CUDA(cudaMemsetAsync(e->log_likelihoods.get(), 0, gpcsps * P * sizeof(double), e->stream));
    e->status.Reserve(2);
    if (unconditional_node_probabilities && inverted_sbn_prior && node_count > 0) {
      e->node_probabilities.Upload(unconditional_node_probabilities, node_count, e->stream);
      e->inverted_prior.Upload(inverted_sbn_prior, gpcsps == static_cast<size_t>(gpcsp_count) ? gpcsp_count : 0,
                               e->stream);
      e->has_node_probabilities = true;
    }
    SBNB_CUDA(cudaStreamSynchronize(e->stream));

    GpParams& p = e->params;
    p.branch_lengths = e->branch_lengths.get();
    p.q = e->q.get();
    p.hybrid = e->hybrid.get();
    p.log_likelihoods = e->log_likelihoods.get();
    p.log_marginal = e->log_marginal.get();
    p.weights = e->weights.get();
    p.threshold = rescaling_threshold;
    p.log_threshold = std::log(rescaling_threshold);
    p.status = e->status.get();
    ModelTables tables;
    BuildModelTables(ModelSpec::Parse("JC69", "constant", "none"), nullptr, &tables);
    std::copy(tables.evec, tables.evec + 16, p.evec);
    std::copy(tables.ivec, tables.ivec + 16, p.ivec);
    std::copy(tables.eval, tables.eval + 4, p.eval);
    std::copy(tables.freqs, tables.freqs + 4, p.freqs);
    *out = e.release();
  });
}

void sbnb_gp_destroy(sbnb_gp_engine* engine) {
  if (!engine) return;
  FloatingPointEnvironmentKeeper keep_caller_environment;
  cudaSetDevice(engine->device);
  delete engine;
}

int sbnb_gp_process_operations(sbnb_gp_engine* e, const int32_t* program, int64_t word_count) {
  return Guard([&] {
    Require(e != nullptr, "NULL GP engine.");
    Require(word_count >= 0 && (program != nullptr || word_count == 0), "NULL program.");
    if (word_count == 0) return;
    Bind(e);
    // The compiled form of a program seen before is still on the device.
    CompiledProgram* compiled = nullptr;
    for (auto& candidate : e->compiled)
      if (candidate->source.size() == static_cast<size_t>(word_count) &&
          std::memcmp(candidate->source.data(), program, word_count * sizeof(int32_t)) == 0)
        compiled = candidate.get();
    if (compiled == nullptr) {
      ValidateProgram(GpShape{e->plv_count, e->gpcsp_count}, program, word_count);
      if (e->compiled.size() >= kGpProgramCacheSize) {
        auto oldest = std::min_element(e->compiled.begin(), e->compiled.end(),
                                       [](const auto& a, const auto& b) { return a->last_used < b->last_used; });
        SBNB_CUDA(cudaStreamSynchronize(e->stream));
        e->compiled.erase(oldest);
      }
      e->compiled.push_back(std::make_unique<CompiledProgram>());
      compiled = e->compiled.back().get();
      CompileProgram(e->plv_count, e->gpcsp_count, program, word_count, compiled);
      compiled->device.Upload(compiled->words.data(), compiled->words.size(), e->stream);
    }
    compiled->last_used = ++e->program_clock;
    SBNB_CUDA(cudaMemsetAsync(e->status.get(), 0, 2 * sizeof(int32_t), e->stream));
    if (e->blocks > 1)  // (epochs restart at 1 in every launch)
      SBNB_CUDA(cudaMemsetAsync(e->exchange.get(), 0,
                                static_cast<size_t>(2) * e->blocks * 2 * kGpReduceValues * sizeof(double), e->stream));
    GpParams p = e->params;
    p.program = compiled->device.get();
    p.word_count = static_cast<int64_t>(compiled->words.size());
    SBNB_CUDA(cudaEventRecord(e->begin, e->stream));
    GpSmemPlan plan = e->plan;
    if (plan.bytes + compiled->words.size() * sizeof(int32_t) <= kGpSmemBudget) {
      plan.program_words = static_cast<int32_t>(compiled->words.size());
      plan.bytes += compiled->words.size() * sizeof(int32_t);
    }
    // (multi-block launches were sized for the whole budget)
    const size_t smem_bytes = e->blocks == 1 ? plan.bytes : kGpSmemBudget;
    const bool single = static_cast<int64_t>(e->blocks) * e->threads >= e->pattern_count * e->params.categories;
    if (e->blocks == 1) {
      if (single) {
        GpInterpretKernel<true><<<1, e->threads, smem_bytes, e->stream>>>(p, plan);
      } else {
        GpInterpretKernel<false><<<1, e->threads, smem_bytes, e->stream>>>(p, plan);
      }
    } else if (e->blocks <= kGpClusterBlocks && !e->no_cluster) {
      // One thread-block cluster: co-scheduled by construction, reductions through distributed
      // shared memory (SBNB_GP_NO_CLUSTER=1 forces the L2 mailbox path below).
      p.cluster_exchange = 1;
      cudaLaunchConfig_t config{};
      config.gridDim = dim3(e->blocks);
      config.blockDim = dim3(e->threads);
      config.dynamicSmemBytes = smem_bytes;
      config.stream = e->stream;
      cudaLaunchAttribute attribute{};
      attribute.id = cudaLaunchAttributeClusterDimension;
      attribute.val.clusterDim.x = e->blocks;
      attribute.val.clusterDim.y = 1;
      attribute.val.clusterDim.z = 1;
      config.attrs = &attribute;
      config.numAttrs = 1;
      const cudaError_t launched = single ? cudaLaunchKernelEx(&config, GpInterpretKernel<true>, p, plan)
                                          : cudaLaunchKernelEx(&config, GpInterpretKernel<false>, p, plan);
      if (launched != cudaSuccess) {
        // (a cluster of this shape cannot be placed here: the mailbox path from now on)
        cudaGetLastError();
        e->no_cluster = true;
        p.cluster_exchange = 0;
      }
    }
    if (e->blocks > 1 && !p.cluster_exchange) {
      // (cooperative: every CTA resident at once, which the cross-CTA exchanges rely on)
      void* args[] = {&p, &plan};
      SBNB_CUDA(cudaLaunchCooperativeKernel(
          single ? reinterpret_cast<void*>(GpInterpretKernel<true>) : reinterpret_cast<void*>(GpInterpretKernel<false>),
          dim3(e->blocks), dim3(e->threads), args, smem_bytes, e->stream));
    }
    SBNB_CUDA(cudaGetLastError());
    SBNB_CUDA(cudaEventRecord(e->end, e->stream));
    e->launch_count++;
    int32_t status[2] = {0, 0};
    SBNB_CUDA(cudaMemcpyAsync(status, e->status.get(), sizeof(status), cudaMemcpyDeviceToHost, e->stream));
    SBNB_CUDA(cudaStreamSynchronize(e->stream));
    float ms = 0.f;
    SBNB_CUDA(cudaEventElapsedTime(&ms, e->begin, e->end));
    e->last_kernel_ms = ms;
    if (status[0] != kGpOk)
      Fail(status[0] == kGpFaultBadProgram ? SBNB_ERR_INVALID_ARGUMENT : SBNB_ERR_GP_ASSERT,
           std::string(FaultMessage(status[0])) + " (operation at word " + std::to_string(OriginalOffset(*compiled, status[1])) + ")");
  });
}

int sbnb_gp_set_substitution_model(sbnb_gp_engine* e, const char* substitution, const double* params,
                                   int32_t param_count) {
  return Guard([&] {
    Require(e != nullptr && substitution != nullptr, "NULL argument.");
    const ModelSpec spec = ModelSpec::Parse(substitution, "constant", "none");
    Require(param_count == spec.param_count,
            std::string("The ") + substitution + " substitution model takes " + std::to_string(spec.param_count) +
                " parameters.");
    Require(params != nullptr || param_count == 0, "NULL parameters.");
    ModelTables tables;
    BuildModelTables(spec, params, &tables);
    GpParams& p = e->params;
    std::copy(tables.evec, tables.evec + 16, p.evec);
    std::copy(tables.ivec, tables.ivec + 16, p.ivec);
    std::copy(tables.eval, tables.eval + 4, p.eval);
    std::copy(tables.freqs, tables.freqs + 4, p.freqs);
  });
}

int sbnb_gp_set_site_model(sbnb_gp_engine* e, const char* site, const double* params, int32_t param_count) {
  return Guard([&] {
    Require(e != nullptr && site != nullptr, "NULL argument.");
    const ModelSpec spec = ModelSpec::Parse("JC69", site, "none");
    Require(!spec.invariant, "The GP engine has no invariable-site (+I) model.");
    Require(param_count == spec.param_count,
            std::string("The ") + site + " site model takes " + std::to_string(spec.param_count) + " parameters.");
    Require(params != nullptr || param_count == 0, "NULL parameters.");
    const int C = spec.category_count;
    Require(C >= 1 && C <= kGpMaxCategories && (C & (C - 1)) == 0,
            "The GP engine takes 1, 2, 4 or 8 rate categories.");
    ModelTables tables;
    BuildSite(spec, params, &tables);
    SetCategories(e, C, tables.rates, tables.weights);
  });
}

int32_t sbnb_gp_category_count(const sbnb_gp_engine* e) { return e ? e->params.categories : 0; }

int sbnb_gp_schedule_program(int32_t plv_count, int32_t gpcsp_count, const int32_t* program, int64_t word_count,
                             int32_t* out, int64_t* out_word_count) {
  return Guard([&] {
    Require(plv_count >= 0 && gpcsp_count >= 0, "Negative PLV / GPCSP count.");
    Require(word_count >= 0 && (program != nullptr || word_count == 0), "NULL program.");
    Require(out != nullptr || word_count == 0, "NULL output.");
    ValidateProgram(GpShape{plv_count, gpcsp_count}, program, word_count);
    CompiledProgram compiled;
    CompileProgram(plv_count, gpcsp_count, program, word_count, &compiled);
    Require(static_cast<int64_t>(compiled.words.size()) <= word_count, "The schedule outgrew the program.");
    std::copy(compiled.words.begin(), compiled.words.end(), out);
    if (out_word_count) *out_word_count = static_cast<int64_t>(compiled.words.size());
  });
}

int sbnb_gp_set_branch_lengths(sbnb_gp_engine* e, const double* branch_lengths) {
  return Guard([&] {
    Require(e && branch_lengths, "NULL argument.");
    Bind(e);
    SBNB_CUDA(cudaMemcpyAsync(e->branch_lengths.get(), branch_lengths, e->gpcsp_count * sizeof(double),
                              cudaMemcpyHostToDevice, e->stream));
    SBNB_CUDA(cudaStreamSynchronize(e->stream));
  });
}

int sbnb_gp_set_branch_lengths_to_constant(sbnb_gp_engine* e, double branch_length) {
  return Guard([&] {
    Require(e != nullptr, "NULL GP engine.");
    std::vector<double> values(e->gpcsp_count, branch_length);
    Bind(e);
    SBNB_CUDA(cudaMemcpyAsync(e->branch_lengths.get(), values.data(), values.size() * sizeof(double),
                              cudaMemcpyHostToDevice, e->stream));
    SBNB_CUDA(cudaStreamSynchronize(e->stream));
  });
}

int sbnb_gp_get_branch_lengths(sbnb_gp_engine* e, double* out) {
  return Guard([&] {
    Require(e && out, "NULL argument.");
    Bind(e);
    CopyOut(e, out, e->branch_lengths.get(), e->gpcsp_count);
  });
}

int sbnb_gp_reset_log_marginal_likelihood(sbnb_gp_engine* e) {
  return Guard([&] {
    Require(e != nullptr, "NULL GP engine.");
    Bind(e);
    std::vector<double> values(e->pattern_count, -INFINITY);
    SBNB_CUDA(cudaMemcpyAsync(e->log_marginal.get(), values.data(), values.size() * sizeof(double),
                              cudaMemcpyHostToDevice, e->stream));
    SBNB_CUDA(cudaStreamSynchronize(e->stream));
  });
}

int sbnb_gp_get_log_marginal_likelihood(sbnb_gp_engine* e, double* out) {
  return Guard([&] {
    Require(e && out, "NULL argument.");
    Bind(e);
    WeightedRowSums(e, e->log_marginal.get(), 1, out);
  });
}

int sbnb_gp_get_per_gpcsp_log_likelihoods(sbnb_gp_engine* e, int32_t start, int32_t length, double* out) {
  return Guard([&] {
    Require(e && out, "NULL argument.");
    Require(start >= 0 && length >= 0 && start + length <= e->gpcsp_count, "GPCSP range out of bounds.");
    Bind(e);
    WeightedRowSums(e, e->log_likelihoods.get() + static_cast<size_t>(start) * e->pattern_count, length, out);
  });
}

int sbnb_gp_get_per_gpcsp_components_of_full_log_marginal(sbnb_gp_engine* e, double* out) {
  return Guard([&] {
    Require(e && out, "NULL argument.");
    Bind(e);
    WeightedRowSums(e, e->log_likelihoods.get(), e->gpcsp_count, out);
    std::vector<double> q(e->gpcsp_count);
    CopyOut(e, q.data(), e->q.get(), e->gpcsp_count);
    for (int g = 0; g < e->gpcsp_count; g++) out[g] += static_cast<double>(e->site_count) * std::log(q[g]);
  });
}

int sbnb_gp_get_log_likelihood_matrix(sbnb_gp_engine* e, double* out) {
  return Guard([&] {
    Require(e && out, "NULL argument.");
    Bind(e);
    CopyOut(e, out, e->log_likelihoods.get(), static_cast<size_t>(e->gpcsp_count) * e->pattern_count);
  });
}

int sbnb_gp_get_sbn_parameters(sbnb_gp_engine* e, double* out) {
  return Guard([&] {
    Require(e && out, "NULL argument.");
    Bind(e);
    CopyOut(e, out, e->q.get(), e->gpcsp_count);
  });
}

int sbnb_gp_set_sbn_parameters(sbnb_gp_engine* e, const double* q) {
  return Guard([&] {
    Require(e && q, "NULL argument.");
    Bind(e);
    SBNB_CUDA(cudaMemcpyAsync(e->q.get(), q, e->gpcsp_count * sizeof(double), cudaMemcpyHostToDevice, e->stream));
    SBNB_CUDA(cudaStreamSynchronize(e->stream));
  });
}

int sbnb_gp_get_hybrid_marginals(sbnb_gp_engine* e, double* out) {
  return Guard([&] {
    Require(e && out, "NULL argument.");
    Bind(e);
    CopyOut(e, out, e->hybrid.get(), e->gpcsp_count);
  });
}

int sbnb_gp_set_hybrid_marginals(sbnb_gp_engine* e, const double* values) {
  return Guard([&] {
    Require(e && values, "NULL argument.");
    Bind(e);
    SBNB_CUDA(cudaMemcpyAsync(e->hybrid.get(), values, e->gpcsp_count * sizeof(double), cudaMemcpyHostToDevice,
                              e->stream));
    SBNB_CUDA(cudaStreamSynchronize(e->stream));
  });
}

int sbnb_gp_log_likelihood_and_derivative(sbnb_gp_engine* e, int32_t leafward, int32_t rootward, int32_t gpcsp,
                                          double* out) {
  return Guard([&] {
    Require(e && out, "NULL argument.");
    CheckPlv(e, leafward);
    CheckPlv(e, rootward);
    CheckGpcsp(e, gpcsp);
    Bind(e);
    e->scalars.Reserve(64);
    GpLogLikelihoodAndDerivativeKernel<<<1, 512, 0, e->stream>>>(e->params, leafward, rootward, gpcsp,
                                                                  e->scalars.get());
    SBNB_CUDA(cudaGetLastError());
    e->launch_count++;
    CopyOut(e, out, e->scalars.get(), 2);
  });
}

int sbnb_gp_transition_matrix(sbnb_gp_engine* e, double branch_length, double* out) {
  return Guard([&] {
    Require(e && out, "NULL argument.");
    Bind(e);
    e->scalars.Reserve(64);
    GpTransitionMatrixKernel<<<1, 32, 0, e->stream>>>(e->params, branch_length, e->scalars.get());
    SBNB_CUDA(cudaGetLastError());
    e->launch_count++;
    CopyOut(e, out, e->scalars.get(), 16);
  });
}

int sbnb_gp_quartet_hybrid_likelihoods(sbnb_gp_engine* e, int32_t central_gpcsp, const int32_t* rootward_tips,
                                       int32_t rootward_count, const int32_t* sister_tips, int32_t sister_count,
                                       const int32_t* rotated_tips, int32_t rotated_count,
                                       const int32_t* sorted_tips, int32_t sorted_count, double* out) {
  return Guard([&] {
    Require(e != nullptr, "NULL GP engine.");
    std::vector<double> values;
    QuartetLikelihoods(e, central_gpcsp, rootward_tips, rootward_count, sister_tips, sister_count, rotated_tips,
                       rotated_count, sorted_tips, sorted_count, &values);
    Require(out != nullptr || values.empty(), "NULL output.");
    std::copy(values.begin(), values.end(), out);
  });
}

int sbnb_gp_process_quartet_hybrid_request(sbnb_gp_engine* e, int32_t central_gpcsp,
                                           const int32_t* rootward_tips, int32_t rootward_count,
                                           const int32_t* sister_tips, int32_t sister_count,
                                           const int32_t* rotated_tips, int32_t rotated_count,
                                           const int32_t* sorted_tips, int32_t sorted_count) {
  return Guard([&] {
    Require(e != nullptr, "NULL GP engine.");
    // IsFullyFormed (quartet_hybrid_request.cpp): every tip list non-empty.
    if (rootward_count <= 0 || sister_count <= 0 || rotated_count <= 0 || sorted_count <= 0) return;
    std::vector<double> values;
    QuartetLikelihoods(e, central_gpcsp, rootward_tips, rootward_count, sister_tips, sister_count, rotated_tips,
                       rotated_count, sorted_tips, sorted_count, &values);
    // NumericalUtils::LogSum = left fold with LogAdd (numerical_utils.cpp:8)
    auto log_add = [](double x, double y) {
      if (y > x) std::swap(x, y);
      if (x == -INFINITY) return x;
      const double neg_diff = y - x;
      if (neg_diff < std::log(2.220446049250313e-16)) return x;
      return x + std::log(1.0 + std::exp(neg_diff));
    };
    double total = values[0];
    for (size_t i = 1; i < values.size(); i++) total = log_add(total, values[i]);
    SBNB_CUDA(cudaMemcpyAsync(e->hybrid.get() + central_gpcsp, &total, sizeof(double), cudaMemcpyHostToDevice,
                              e->stream));
    SBNB_CUDA(cudaStreamSynchronize(e->stream));
  });
}

int sbnb_gp_get_plv(sbnb_gp_engine* e, int32_t plv_idx, double* out) {
  return Guard([&] {
    Require(e && out, "NULL argument.");
    CheckPlv(e, plv_idx);
    Bind(e);
    const size_t plv_doubles = static_cast<size_t>(e->pattern_count) * e->params.categories * 4;
    CopyOut(e, out, e->plvs.get() + plv_idx * plv_doubles, plv_doubles);
  });
}

int sbnb_gp_get_rescaling_counts(sbnb_gp_engine* e, int32_t* out) {
  return Guard([&] {
    Require(e && out, "NULL argument.");
    Bind(e);
    SBNB_CUDA(cudaMemcpyAsync(out, e->counts.get(), e->plv_count * sizeof(int32_t), cudaMemcpyDeviceToHost,
                              e->stream));
    SBNB_CUDA(cudaStreamSynchronize(e->stream));
  });
}

int64_t sbnb_gp_launch_count(const sbnb_gp_engine* e) { return e ? e->launch_count : -1; }
double sbnb_gp_last_kernel_ms(const sbnb_gp_engine* e) { return e ? e->last_kernel_ms : -1.0; }

}  // extern "C"
