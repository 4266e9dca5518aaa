// Device code of libsbn_b200 (sm_100a, fp64, no tensor cores -- 4x4 mat-vecs).
//
// Kernels:
//   TransitionMatrixKernel  per (tree, edge, category): P = V diag(exp(lambda r_c t)) V^-1, its
//                           transpose, and (Q P)^T, in the layout the tree walk stages
//                           [replaces beagleUpdateTransitionMatrices, fat_beagle.cpp:304-314, and
//                            beagleSetDifferentialMatrix, fat_beagle.cpp:128-131]
//   TreeWalkKernel          one pass over a tree for a tile of site patterns: the
//                           post-order partial updates, per-pattern power-of-two
//                           rescaling, the root log-likelihood, and (gradient mode)
//                           the pre-order pass fused with all edge derivatives
//                           [replaces beagleUpdatePartials, beagleUpdatePrePartials,
//                            beagleCalculateEdgeDerivatives, beagleCalculateRootLogLikelihoods,
//                            beagleResetScaleFactors, beagleSetPartials(root pre := pi);
//                            fat_beagle.cpp:50-70, 119-175]
//   ReducePartialsKernel    fixed-order sum of the per-(chunk, warp) partial sums
//
// Design (see DESIGN.md): site patterns are independent, so a thread owns K
// patterns -- all rate categories of them -- and walks the WHOLE tree for them.
// The walk order (host-generated, Strahler-ordered, tree_program.cpp) keeps the
// result of the previous op in registers ("cur"); only nodes with two internal
// children touch a small stack (global memory, L2 resident).  In gradient mode
// the evolved post-order partials P_x L_x are streamed to a per-CTA scratch
// arena (written once, read once by the pre-order pass).
//
// Everything an op needs besides partials -- the transition matrices of both
// child edges for every category and the tip states of the tile -- is brought
// into a shared-memory ring by TMA bulk copies (cp.async.bulk +
// mbarrier), issued two ops ahead by one elected thread; all lanes of a warp
// read the same matrix element, so matrix loads are shared-memory broadcasts.
#ifndef SBNB_KERNELS_CUH_
#define SBNB_KERNELS_CUH_

#include <cuda_runtime.h>
#include <stdint.h>

#include "model.hpp"
#include "tree_program.hpp"

namespace sbnb {

constexpr int kThreads = 128;  // 4 warps per CTA; warps only meet at the ring's mbarriers
constexpr int kWarps = kThreads / 32;

// Per (tree, edge) block written by TransitionMatrixKernel, in doubles, C = categories:
//   [0        .. 18C)  P_c            row-major (+ 2 doubles of padding), c = 0..C-1
//                                      (internal child: y = P L)
//   [18C      .. 38C)  per c: P_c^T (row s = column s of P) then 4 ones
//                                      (tip child: y = column of P; gap: y = 1)
//   [38C      .. 58C)  per c: (Q P_c)^T then 4 zeros
//                                      (tip child: Q y; gap: Q 1 = 0)
constexpr int kTipTableDoubles = 20;  // per category: 4 state rows + the gap row
// P_c blocks are 18 doubles apart (16 + 2 of padding): lanes that hold different
// categories then read the same element of their matrices from different banks.
constexpr int kPStride = 18;
constexpr int kEdgeDoublesPerCategory = kPStride + 2 * kTipTableDoubles;

// One op of the walk: 16 bytes.  Post-order op (first n-1 of a program) and
// pre-order op (last n-1) share the layout.
//   x = child 0 node id, y = child 1 node id,
//   z = node id | flags << 24
//   w = post: push_slot | a_slot << 8 | b_slot << 16
//       pre:  pop_slot  | a_push_slot << 8 | b_push_slot << 16      (0xff = none)
typedef int4 WalkOp;
// flags beyond kALeaf | kBLeaf | kRoot (tree_program.hpp)
enum : int32_t {
  kStackBefore = 8,  // post: push cur first; pre: pop cur first
  kACur = 16,        // post: child 0's partial is cur; pre: child 0's pre-order partial stays in cur
  kBCur = 32
};

struct WalkParams {
  // alignment (device)
  const uint8_t* tips;  // [taxon][tip_pitch], padded with gap states
  int64_t tip_pitch;
  const double* weights;  // [tip_pitch] padded with zeros
  int64_t pattern_begin, pattern_end;
  int32_t taxon_count;
  // programs (device): [program][2(n-1)] = post-order ops then pre-order ops
  const WalkOp* ops;
  // virtual trees: vtree v uses program vtree_program[v], model vtree_model[v]
  int32_t vtree_begin, vtree_count;
  const int32_t* vtree_program;
  const int32_t* vtree_model;
  const ModelTables* models;
  const double* matrices;  // [vtree][2n-2][56 C]
  // tiling
  int32_t tiles_total, tiles_per_chunk, chunks;
  int32_t slots;  // stack depth
  // per-CTA arenas + outputs
  double2* stack;         // [grid][slots][K][C][2][kThreads]
  int32_t* stack_exps;    // [grid][slots][K][kThreads]              (rescaling)
  double2* scratch;       // [grid][n-1][C][K][2][kThreads]          (gradient mode)
  double* logl_partial;   // [vtree][chunk][warp]
  double* grad_partial;   // [vtree][chunk][warp][2n-1]               (gradient mode)
  double* rgrad_partial;  // same, with d rate_c / d shape as the scalers (C > 1)
};

// Shared memory of one CTA (host and device agree through these).
// Per-item model constants of a walk over C (padded) categories: Q[16], then p_c, r_c and
// dr_c/dshape with ModelSmemCategories(C) entries each, pi[4].  Up to 16 categories the
// arrays keep 16 entries.
__host__ __device__ constexpr int ModelSmemCategories(int C) { return C > 16 ? C : 16; }
__host__ __device__ constexpr int ModelSmemDoubles(int C) { return 16 + 3 * ModelSmemCategories(C) + 4; }

// ---------------------------------------------------------------------------
// mbarrier / TMA bulk-copy helpers (PTX; see blackwell_cuda_programming.md)

__device__ __forceinline__ uint32_t SmemAddress(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void MbarInit(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(SmemAddress(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void MbarExpectTx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(SmemAddress(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void MbarArrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(SmemAddress(bar)) : "memory");
}
// A waiting warp may stay suspended this long before it has to re-issue the wait:
// a spinning warp takes issue slots from the warps it is waiting for.
constexpr uint32_t kMbarSuspendHintNs = 4000;
__device__ __forceinline__ void MbarWait(uint64_t* bar, uint32_t parity) {
  const uint32_t address = SmemAddress(bar);
  uint32_t done;
  do {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(done)
        : "r"(address), "r"(parity), "r"(kMbarSuspendHintNs)
        : "memory");
  } while (!done);
}
// global -> shared bulk copy (TMA, no tensor map); bytes and both addresses are
// multiples of 16; completion is signalled on `bar` as transaction bytes.
__device__ __forceinline__ void BulkCopy(void* smem_dst, const void* global_src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   SmemAddress(smem_dst)),
               "l"(global_src), "r"(bytes), "r"(SmemAddress(bar))
               : "memory");
}

// ---------------------------------------------------------------------------
// small helpers (everything is fully unrolled; partials live in registers)

__device__ __forceinline__ void Load4(const double* src, double (&x)[4]) {
  const double2 v0 = reinterpret_cast<const double2*>(src)[0];
  const double2 v1 = reinterpret_cast<const double2*>(src)[1];
  x[0] = v0.x, x[1] = v0.y, x[2] = v1.x, x[3] = v1.y;
}

// y = M^T x
template <int K>
__device__ __forceinline__ void MatTVecSharedK(const double* m, const double (&x)[K][4], double (&y)[K][4]) {
#pragma unroll
  for (int i = 0; i < 4; i++) {
    double row[4];
    Load4(m + 4 * i, row);
#pragma unroll
    for (int j = 0; j < K; j++)
#pragma unroll
      for (int s = 0; s < 4; s++) y[j][s] = (i == 0) ? row[s] * x[j][0] : fma(row[s], x[j][i], y[j][s]);
  }
}

__device__ __forceinline__ double Dot4(const double (&a)[4], const double (&b)[4]) {
  return fma(a[3], b[3], fma(a[2], b[2], fma(a[1], b[1], a[0] * b[0])));
}

__device__ __forceinline__ double WarpSum(double v) {
#pragma unroll
  for (int m = 16; m >= 1; m >>= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
  return v;
}

// Per-pattern power-of-two normalisation over all C x 4 entries: when the
// largest entry has dropped below 2^-kLazyBits, scales by 2^-e (e = its
// exponent) and returns e.  Exact (no rounding), so rescaled and unrescaled
// runs agree bit for bit until the final log.
constexpr int kLazyBits = 128;
template <int C>
__device__ __forceinline__ int Normalize(double (&v)[C][4]) {
  int hi = __double2hiint(v[0][0]);
#pragma unroll
  for (int c = 0; c < C; c++)
#pragma unroll
    for (int i = 0; i < 4; i++) hi = max(hi, __double2hiint(v[c][i]));
  const int biased = (hi >> 20) & 0x7ff;
  // zero / subnormal / inf / nan, or still large enough: leave as is
  if (biased == 0 || biased >= 1023 - kLazyBits) return 0;
  const double scale = __hiloint2double((2046 - biased) << 20, 0);
#pragma unroll
  for (int c = 0; c < C; c++)
#pragma unroll
    for (int i = 0; i < 4; i++) v[c][i] *= scale;
  return biased - 1023;
}

// ---------------------------------------------------------------------------

// One thread per (virtual tree, edge, category).
__global__ void TransitionMatrixKernel(const ModelTables* __restrict__ models,
                                       const int32_t* __restrict__ vtree_model,
                                       const int32_t* __restrict__ vtree_lengths,
                                       const double* __restrict__ branch_lengths,
                                       double* __restrict__ matrices, int32_t vtree_count,
                                       int32_t edge_count, int32_t node_count, int32_t C) {
  const int64_t idx = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int64_t total = static_cast<int64_t>(vtree_count) * edge_count * C;
  if (idx >= total) return;
  const int c = static_cast<int>(idx % C);
  const int e = static_cast<int>((idx / C) % edge_count);
  const int v = static_cast<int>(idx / (static_cast<int64_t>(C) * edge_count));
  const ModelTables& model = models[vtree_model[v]];
  const double t =
      branch_lengths[static_cast<int64_t>(vtree_lengths[v]) * node_count + e] * model.rates[c];
  double ex[4];
#pragma unroll
  for (int k = 0; k < 4; k++) ex[k] = exp(model.eval[k] * t);
  double P[16];
#pragma unroll
  for (int i = 0; i < 4; i++)
#pragma unroll
    for (int j = 0; j < 4; j++) {
      double sum = 0.0;
#pragma unroll
      for (int k = 0; k < 4; k++) sum += (model.evec[i * 4 + k] * ex[k]) * model.ivec[k * 4 + j];
      P[i * 4 + j] = sum > 0.0 ? sum : 0.0;  // BEAGLE clamps round-off negatives
    }
  double* edge = matrices + (static_cast<int64_t>(v) * edge_count + e) * kEdgeDoublesPerCategory * C;
  double2* out = reinterpret_cast<double2*>(edge + kPStride * c);
#pragma unroll
  for (int x = 0; x < 8; x++) out[x] = make_double2(P[2 * x], P[2 * x + 1]);
  out = reinterpret_cast<double2*>(edge + kPStride * C + kTipTableDoubles * c);
#pragma unroll
  for (int s = 0; s < 4; s++) {  // P^T: row s = column s of P
    out[2 * s] = make_double2(P[s], P[4 + s]);
    out[2 * s + 1] = make_double2(P[8 + s], P[12 + s]);
  }
  out[8] = make_double2(1.0, 1.0);
  out[9] = make_double2(1.0, 1.0);
  out = reinterpret_cast<double2*>(edge + (kPStride + kTipTableDoubles) * C + kTipTableDoubles * c);
#pragma unroll
  for (int s = 0; s < 4; s++) {  // (Q P)^T: row s = column s of Q P
    double col[4];
#pragma unroll
    for (int i = 0; i < 4; i++)
      col[i] = fma(model.q[i * 4 + 3], P[12 + s],
                   fma(model.q[i * 4 + 2], P[8 + s], fma(model.q[i * 4 + 1], P[4 + s], model.q[i * 4] * P[s])));
    out[2 * s] = make_double2(col[0], col[1]);
    out[2 * s + 1] = make_double2(col[2], col[3]);
  }
  out[8] = make_double2(0.0, 0.0);
  out[9] = make_double2(0.0, 0.0);
}

// out[v][e] = sum over the `parts` per-(chunk, warp) partial rows, in fixed order.
__global__ void ReducePartialsKernel(const double* __restrict__ partial, double* __restrict__ out,
                                     int32_t vtree_begin, int32_t vtree_count, int32_t parts,
                                     int32_t width) {
  const int64_t idx = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= static_cast<int64_t>(vtree_count) * width) return;
  const int64_t v = vtree_begin + idx / width;
  const int e = static_cast<int>(idx % width);
  const double* src = partial + v * parts * width + e;
  double sum = 0.0;
  for (int part = 0; part < parts; part++) sum += src[static_cast<int64_t>(part) * width];
  out[v * width + e] = sum;
}

}  // namespace sbnb

#endif  // SBNB_KERNELS_CUH_
