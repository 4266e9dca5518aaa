// beagle_shim.cu -> libsbn_b200/lib/libhmsbeagle_b200.so: the INNER drop-in boundary of
// libsbn_b200 (SURVEY.md 8b) -- the 17 entry points of the BEAGLE C API that phylovi/libsbn
// links against (include/libhmsbeagle/beagle.h; every call site is in the reference's
// src/fat_beagle.cpp), each one running on the B200.  Relink the UNMODIFIED reference
// (fat_beagle.cpp, engine.cpp, ... as they are) against this library instead of
// libhmsbeagle and its partial-likelihood arithmetic runs on the device; nothing else
// changes (integration/Makefile builds the reference's own doctest that way).
//
// This is the compatibility path: BEAGLE's op-at-a-time schedule with every partial
// materialised in HBM -- B_grad = (10n - 14) U bytes per logL + gradient evaluation
// (SURVEY.md 8d).  The performance path is the outer boundary (include/sbn_b200.h), whose
// fused tree walk moves a fifth of that.
//
// Layout in HBM, per instance (BEAGLE's own conventions, fat_beagle.cpp:207-256):
//   partials [buffer][category][pattern][state] fp64 (state fastest), one slab;
//   compact tips [tip][pattern] uint8 (state >= 4 = missing);
//   matrices [matrix][category][i][j]; scale buffers [scaler][pattern] (raw maxima; buffer
//   `cumulative` holds sums of logs).
// Kernels: a thread owns a site pattern.  One beagleUpdatePartials / UpdatePrePartials call
// is ONE launch: the ops of a call depend on each other only through buffers indexed by
// pattern, so a thread works through the whole op list for its pattern and every hazard is
// a same-thread hazard (no barrier, no launch per op).  Reads and writes are 32 bytes per
// (pattern, category), consecutive threads consecutive patterns: fully coalesced; the
// kernels are HBM-bound (3 U of traffic per op against 60 flop per 96 bytes).
// Reductions (root logL, edge derivatives) are per-block partial sums added in a fixed
// order by a second launch: deterministic.
//
// There is no CPU path in this file: without a CUDA device beagleCreateInstance returns
// BEAGLE_ERROR_NO_RESOURCE.

#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <vector>

#include "../../include/libhmsbeagle/beagle.h"

namespace {

constexpr int kStates = 4;
constexpr int kBlock = 128;
// the pipelined partial updates: threads per CTA (the op records and matrices a CTA stages are
// shared by more threads) and resident CTAs per SM (64 registers: 1024 threads)
#ifndef SBNB_SHIM_PIPE_BLOCK
#define SBNB_SHIM_PIPE_BLOCK 256
#endif
constexpr int kPipeBlock = SBNB_SHIM_PIPE_BLOCK;
constexpr int kPipeMinBlocks = 1024 / kPipeBlock;

struct alignas(16) DeviceOp {
  int32_t dest, scale_write, child1, matrix1, child2, matrix2;
  int32_t flags;  // what the host knows about the children (the pipelined kernel's cases)
  int32_t pad;
  // the same, as element offsets (the pipelined kernel adds its thread's offset: no 64-bit
  // multiplications per op): partials in doubles -- a compact child in bytes of the state
  // array --, the scale buffer in doubles (unused when scale_write < 0)
  int64_t dest_at, child1_at, child2_at, scale_at;
};
static_assert(sizeof(DeviceOp) == 64, "op records are four 16-byte words");
// child x is a compact tip / is the destination of the PREVIOUS op of the list (still in the
// thread's registers: no load)
enum : int32_t { kChild1Compact = 1, kChild2Compact = 2, kChild1Forward = 4, kChild2Forward = 8 };

struct InstanceView {
  int32_t tips, buffers, P, C, matrices, scalers;
  double* partials;          // [buffer][C][P][4]
  const uint8_t* compact;    // [tips][P]
  const uint8_t* is_compact; // [buffers]
  double* matrix;            // [matrix][C][16]
  double* scale;             // [scaler][P]
  const double* cat_weights; // [C]
  const double* freqs;       // [4]
  const double* pattern_weights;  // [P]
};

// The four states of one (pattern, category) in global memory: ONE 256-bit access (sm_100;
// LDG.E.256 / STG.E.256), so a warp's request covers whole 128-byte lines -- two 128-bit halves
// 32 bytes apart take twice the L1 wavefronts.  32-byte aligned: every partial and matrix row is.
__device__ __forceinline__ void Load4(const double* src, double (&x)[4]) {
  asm volatile("ld.global.v4.f64 {%0, %1, %2, %3}, [%4];" : "=d"(x[0]), "=d"(x[1]), "=d"(x[2]), "=d"(x[3]) : "l"(src));
}
__device__ __forceinline__ void Store4(double* dst, const double (&x)[4]) {
  asm volatile("st.global.v4.f64 [%0], {%1, %2, %3, %4};" ::"l"(dst), "d"(x[0]), "d"(x[1]), "d"(x[2]), "d"(x[3]) : "memory");
}
// ... and in shared memory (16-byte aligned rows)
__device__ __forceinline__ void LoadShared4(const double* src, double (&x)[4]) {
  const double2 a = reinterpret_cast<const double2*>(src)[0], b = reinterpret_cast<const double2*>(src)[1];
  x[0] = a.x, x[1] = a.y, x[2] = b.x, x[3] = b.y;
}
__device__ __forceinline__ double* Partial(const InstanceView& v, int buffer, int c, int64_t k) {
  return v.partials + ((static_cast<size_t>(buffer) * v.C + c) * v.P + k) * kStates;
}

// (P L)[i] for one child: a mat-vec for a full partial, column s of P for a compact state
// s < 4, all ones for a missing state (beagleUpdatePartials' tip cases).
__device__ __forceinline__ void ChildTerm(const InstanceView& v, int buffer, const double* m, int c, int64_t k,
                                          double (&out)[4]) {
  if (v.is_compact[buffer]) {
    const int s = v.compact[static_cast<size_t>(buffer) * v.P + k];
#pragma unroll
    for (int i = 0; i < 4; i++) out[i] = s < kStates ? __ldg(m + i * 4 + s) : 1.0;
  } else {
    double L[4];
    Load4(Partial(v, buffer, c, k), L);
#pragma unroll
    for (int i = 0; i < 4; i++) {
      double row[4];
      Load4(m + i * 4, row);
      out[i] = fma(row[3], L[3], fma(row[2], L[2], fma(row[1], L[1], row[0] * L[0])));
    }
  }
}

// beagleUpdatePartials (PRE = false; fat_beagle.cpp:60-63, 139-141):
//     dest = (P1 L1) o (P2 L2)
// beagleUpdatePrePartials (PRE = true; fat_beagle.cpp:143-151): child1 is the parent's
// pre-order partial, matrix1 the node's OWN matrix applied transposed, child2 the sister:
//     dest[j] = sum_i P1[i][j] (pre[i] (P2 L2)[i])
// With a scale buffer to write: per pattern divide by the maximum over (category, state)
// (0 -> 1), store the raw maximum, add its log to the cumulative buffer if one is given.
//
// One op for one (pattern, category); returns the largest entry.
template <bool PRE>
__device__ __forceinline__ double OpTerm(const InstanceView& v, const DeviceOp& op, int c, int64_t k, double (&d)[4]) {
  const double* m1 = v.matrix + (static_cast<size_t>(op.matrix1) * v.C + c) * 16;
  const double* m2 = v.matrix + (static_cast<size_t>(op.matrix2) * v.C + c) * 16;
  double b[4];
  ChildTerm(v, op.child2, m2, c, k, b);
  if (PRE) {
    double pre[4], t[4];
    Load4(Partial(v, op.child1, c, k), pre);
#pragma unroll
    for (int i = 0; i < 4; i++) t[i] = pre[i] * b[i];
#pragma unroll
    for (int j = 0; j < 4; j++)
      d[j] = fma(__ldg(m1 + 12 + j), t[3], fma(__ldg(m1 + 8 + j), t[2], fma(__ldg(m1 + 4 + j), t[1], __ldg(m1 + j) * t[0])));
  } else {
    double a[4];
    ChildTerm(v, op.child1, m1, c, k, a);
#pragma unroll
    for (int i = 0; i < 4; i++) d[i] = a[i] * b[i];
  }
  return fmax(fmax(d[0], d[1]), fmax(d[2], d[3]));
}

// Up to 16 rate categories on CT = 1, 2, 4, 8 or 16 lanes per pattern (the next power of two;
// spare lanes shadow category 0): a thread owns K adjacent patterns of one category --
// category-major inside the warp, so the 32 / CT lanes of a category read consecutive patterns
// (32 K bytes each: coalesced) -- for the whole op list of the call.  The walk is a chain of
// dependent global-memory round trips per thread (ncu of the first version: 66 % of the
// stalls on the long scoreboard at half of the HBM peak), so:
//   * a child that is the destination of the previous op is taken from registers (the host
//     flags it: in a post-order list that is one child of nearly every op);
//   * the other internal children of op o + 1 are requested right after the mat-vecs of op o
//     have consumed op o's operands -- the rest of op o (maximum, division, logarithm, stores)
//     and the other warps cover the latency;
//   * op records and the two matrices of each op are staged in shared memory a chunk of ops at
//     a time (a compact child's matrix transposed: column s is one 32-byte row), category
//     blocks 144 bytes apart (no bank conflicts between the categories of a warp);
//   * the cumulative scale buffer is read once, summed in a register in the op order and
//     written once (the host checks that no op of the list writes the same buffer);
//   * the per-pattern maximum of a rescaled op is taken over the pattern's CT lanes by
//     shuffles, and the logarithms of CT rescaled ops are taken at once, one per category lane
//     (a quarter of the instructions of the first version were the logarithm that one lane in
//     CT needed);
//   * a record carries its buffers as element offsets, and the four states of a (pattern,
//     category) move as one 256-bit access.
constexpr int kMatrixStride = 18;  // doubles between the category blocks of a staged matrix
#ifndef SBNB_SHIM_CHUNK
#define SBNB_SHIM_CHUNK 32
#endif
__host__ __device__ constexpr int ChunkOps(int CT) { return CT <= 4 ? SBNB_SHIM_CHUNK : (CT == 8 ? SBNB_SHIM_CHUNK / 2 : SBNB_SHIM_CHUNK / 4); }

template <bool PRE, int CT, int K, bool PADDED>
__global__ void __launch_bounds__(kPipeBlock, K == 1 ? kPipeMinBlocks : (kPipeMinBlocks + 1) / 2) UpdatePartialsPipelinedKernel(const InstanceView v,
                                                                       const DeviceOp* __restrict__ ops, int op_count,
                                                                       int cumulative, int cumulative_in_register) {
  constexpr int kPerWarp = 32 / CT;  // pattern groups of a warp
  constexpr int kChunk = ChunkOps(CT);
  constexpr int kPipeBlockPatterns = (kPipeBlock / 32) * kPerWarp * K;
  constexpr int kOpMatrixDoubles = 2 * CT * kMatrixStride;
  constexpr int kOpEntries = 2 * CT * 16;  // matrix entries staged per op
  constexpr unsigned kFull = 0xffffffffu;
  __shared__ __align__(16) DeviceOp s_ops[kChunk];
  __shared__ __align__(16) double s_matrix[kChunk * kOpMatrixDoubles];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // v.C <= CT categories on CT lanes per pattern: the lanes past the last category shadow
  // category 0 (same values: the maximum over the lanes does not change) and store nothing.
  // (PADDED = false: v.C == CT, and none of this costs anything -- with the run-time form the
  //  pre-order update of 4 categories measured 13 % slower)
  const int category_lane = lane / kPerWarp;
  const bool padding_lane = PADDED && category_lane >= v.C;
  const int c = padding_lane ? 0 : category_lane;
  const int categories = PADDED ? v.C : CT;
  // (the trip count is the same for every thread of a block: the chunk loop has barriers)
  for (int64_t base = static_cast<int64_t>(blockIdx.x) * kPipeBlockPatterns; base < v.P;
       base += static_cast<int64_t>(gridDim.x) * kPipeBlockPatterns) {
    const int64_t first = base + static_cast<int64_t>(warp * kPerWarp + lane % kPerWarp) * K;
    // This thread's place in a partial buffer (doubles), in a state / scale row, and whether it
    // stores: kept opaque to the compiler, which otherwise re-derives them from threadIdx at
    // every op of the list (a third of the instructions of an op, measured).
    int64_t elem[K];
    int pattern[K], live[K];
#pragma unroll
    for (int j = 0; j < K; j++) {
      pattern[j] = static_cast<int>(first + j < v.P ? first + j : v.P - 1);  // (idle slots shadow the last pattern)
      live[j] = first + j < v.P && !padding_lane;
      elem[j] = (static_cast<int64_t>(c) * v.P + pattern[j]) * kStates;
      asm volatile("" : "+l"(elem[j]), "+r"(pattern[j]), "+r"(live[j]));
    }
    // The logarithms of the cumulative scale buffer are taken CT at a time: the pattern's
    // lanes all hold the op's maximum, the lane of category (rescaled ops so far) % CT keeps
    // it, and after CT rescaled ops every lane takes ONE logarithm; the terms are then added
    // in op order (shuffles), each lane of the pattern keeping the same sum.
    double cum[K], held[K];
    int pending = 0;
#pragma unroll
    for (int j = 0; j < K; j++) {
      held[j] = 1.0;
      cum[j] = (cumulative >= 0 && cumulative_in_register)
                   ? v.scale[static_cast<int64_t>(cumulative) * v.P + pattern[j]]
                   : 0.0;
    }
    auto flush_logarithms = [&]() {
      double term[K];
#pragma unroll
      for (int j = 0; j < K; j++) term[j] = log(held[j]);
#pragma unroll
      for (int i = 0; i < CT; i++) {
        if (i < pending) {
#pragma unroll
          for (int j = 0; j < K; j++) cum[j] += __shfl_sync(kFull, term[j], lane % kPerWarp + i * kPerWarp);
        }
      }
      pending = 0;
    };
    double d[K][4];    // the result of the previous op
    double n1[K][4], n2[K][4];  // requested partials of the next op's children
    int s1[K], s2[K];  // ... or their compact states
#pragma unroll
    for (int j = 0; j < K; j++) {
      s1[j] = s2[j] = 0;
#pragma unroll
      for (int i = 0; i < 4; i++) d[j][i] = n1[j][i] = n2[j][i] = 0.0;
    }
    auto request = [&](const DeviceOp& op) {
      const int flags = op.flags;
      if (flags & kChild1Compact) {
#pragma unroll
        for (int j = 0; j < K; j++) s1[j] = v.compact[op.child1_at + pattern[j]];
      } else if (!(flags & kChild1Forward)) {
#pragma unroll
        for (int j = 0; j < K; j++) Load4(v.partials + (op.child1_at + elem[j]), n1[j]);
      }
      if (flags & kChild2Compact) {
#pragma unroll
        for (int j = 0; j < K; j++) s2[j] = v.compact[op.child2_at + pattern[j]];
      } else if (!(flags & kChild2Forward)) {
#pragma unroll
        for (int j = 0; j < K; j++) Load4(v.partials + (op.child2_at + elem[j]), n2[j]);
      }
    };
    // out[j] = M x[j] (a full partial; M row-major in shared memory)
    auto evolve = [&](const double* m, const double (&x)[K][4], double (&out)[K][4]) {
#pragma unroll
      for (int i = 0; i < 4; i++) {
        double row[4];
        LoadShared4(m + 4 * i, row);
#pragma unroll
        for (int j = 0; j < K; j++)
          out[j][i] = fma(row[3], x[j][3], fma(row[2], x[j][2], fma(row[1], x[j][1], row[0] * x[j][0])));
      }
    };
    // out[j] = column s of M (staged transposed: row s), all ones for a missing state
    auto column = [&](const double* mt, const int (&s)[K], double (&out)[K][4]) {
#pragma unroll
      for (int j = 0; j < K; j++) {
        LoadShared4(mt + 4 * (s[j] & 3), out[j]);
        if (s[j] >= kStates) out[j][0] = out[j][1] = out[j][2] = out[j][3] = 1.0;
      }
    };

    for (int chunk_begin = 0; chunk_begin < op_count; chunk_begin += kChunk) {
      const int chunk_ops = min(kChunk, op_count - chunk_begin);
      __syncthreads();  // every warp is done with the previous chunk
      for (int e = threadIdx.x; e < chunk_ops * 4; e += kPipeBlock)
        reinterpret_cast<int4*>(s_ops)[e] = reinterpret_cast<const int4*>(ops + chunk_begin)[e];
      // the two matrices of every op of the chunk (a thread's entry of an op does not change
      // from pass to pass when the block covers whole ops)
      if (kOpEntries <= kPipeBlock) {
        const int within = threadIdx.x % kOpEntries;
        const int entry = within & 15, cc = (within >> 4) % CT, which = within / (16 * CT);
        const int plain = (which * CT + cc) * kMatrixStride + entry;
        const int transposed = (which * CT + cc) * kMatrixStride + (entry & 3) * 4 + (entry >> 2);
        for (int o = threadIdx.x / kOpEntries; o < chunk_ops; o += kPipeBlock / kOpEntries) {
          const DeviceOp& op = ops[chunk_begin + o];
          const int flags = op.flags;
          const int matrix = which ? op.matrix2 : op.matrix1;
          if (cc < categories)
            s_matrix[o * kOpMatrixDoubles + ((flags & (which ? kChild2Compact : kChild1Compact)) ? transposed : plain)] =
                v.matrix[(static_cast<size_t>(matrix) * categories + cc) * 16 + entry];
        }
      } else {
        for (int e = threadIdx.x; e < chunk_ops * kOpEntries; e += kPipeBlock) {
          const int entry = e & 15, cc = (e >> 4) % CT, which = (e / (16 * CT)) & 1, o = e / kOpEntries;
          const DeviceOp& op = ops[chunk_begin + o];
          const bool transposed = op.flags & (which ? kChild2Compact : kChild1Compact);
          const int matrix = which ? op.matrix2 : op.matrix1;
          if (cc < categories)
            s_matrix[o * kOpMatrixDoubles + (which * CT + cc) * kMatrixStride +
                     (transposed ? (entry & 3) * 4 + (entry >> 2) : entry)] =
                v.matrix[(static_cast<size_t>(matrix) * categories + cc) * 16 + entry];
        }
      }
      __syncthreads();
      request(s_ops[0]);  // (the first op of a chunk waits for its operands)
      for (int o = 0; o < chunk_ops; o++) {
        const DeviceOp& op = s_ops[o];
        const int flags = op.flags;
        const double* const m1 = s_matrix + o * kOpMatrixDoubles + c * kMatrixStride;
        const double* const m2 = m1 + CT * kMatrixStride;
        double a[K][4], b[K][4];
        if (flags & kChild2Compact) {
          column(m2, s2, b);
        } else if (flags & kChild2Forward) {
          evolve(m2, d, b);
        } else {
          evolve(m2, n2, b);
        }
        if (PRE) {
          // a = pre o (P2 L2); child1 is the parent's pre-order partial (never compact)
          if (flags & kChild1Forward) {
#pragma unroll
            for (int j = 0; j < K; j++)
#pragma unroll
              for (int i = 0; i < 4; i++) a[j][i] = d[j][i] * b[j][i];
          } else {
#pragma unroll
            for (int j = 0; j < K; j++)
#pragma unroll
              for (int i = 0; i < 4; i++) a[j][i] = n1[j][i] * b[j][i];
          }
        } else if (flags & kChild1Compact) {
          column(m1, s1, a);
        } else if (flags & kChild1Forward) {
          evolve(m1, d, a);
        } else {
          evolve(m1, n1, a);
        }
        // this op's operands are consumed: ask for the next op's
        if (o + 1 < chunk_ops) request(s_ops[o + 1]);
        if (PRE) {
          // d[x] = sum_i P1[i][x] a[i]: rows of P1 scaled by a[i], added in the order i = 0..3
#pragma unroll
          for (int i = 0; i < 4; i++) {
            double row[4];
            LoadShared4(m1 + 4 * i, row);
#pragma unroll
            for (int j = 0; j < K; j++)
#pragma unroll
              for (int x = 0; x < 4; x++) d[j][x] = (i == 0) ? row[x] * a[j][0] : fma(row[x], a[j][i], d[j][x]);
          }
        } else {
#pragma unroll
          for (int j = 0; j < K; j++)
#pragma unroll
            for (int i = 0; i < 4; i++) d[j][i] = a[j][i] * b[j][i];
        }
        if (op.scale_write >= 0) {
          double largest[K];
#pragma unroll
          for (int j = 0; j < K; j++) {
            // the reference's maximum: starts at 0, takes v when v > max (so never a NaN)
            largest[j] = 0.0;
#pragma unroll
            for (int i = 0; i < 4; i++) largest[j] = d[j][i] > largest[j] ? d[j][i] : largest[j];
#pragma unroll
            for (int s = kPerWarp; s < 32; s <<= 1) {
              const double other = __shfl_xor_sync(kFull, largest[j], s);
              largest[j] = other > largest[j] ? other : largest[j];
            }
            if (largest[j] == 0.0) largest[j] = 1.0;
            const double inverse = 1.0 / largest[j];
#pragma unroll
            for (int i = 0; i < 4; i++) d[j][i] *= inverse;
          }
          if (category_lane == 0) {
#pragma unroll
            for (int j = 0; j < K; j++)
              if (live[j]) v.scale[op.scale_at + pattern[j]] = largest[j];
          }
          if (cumulative >= 0) {
            if (cumulative_in_register) {
#pragma unroll
              for (int j = 0; j < K; j++)
                if (category_lane == pending) held[j] = largest[j];
              if (++pending == CT) flush_logarithms();
            } else if (category_lane == 0) {
#pragma unroll
              for (int j = 0; j < K; j++)
                if (live[j]) v.scale[static_cast<int64_t>(cumulative) * v.P + pattern[j]] += log(largest[j]);
            }
          }
        }
#pragma unroll
        for (int j = 0; j < K; j++)
          if (live[j]) Store4(v.partials + (op.dest_at + elem[j]), d[j]);
      }
    }
    if (cumulative >= 0 && cumulative_in_register) {
      if (pending > 0) flush_logarithms();
      if (category_lane == 0) {
#pragma unroll
        for (int j = 0; j < K; j++)
          if (live[j]) v.scale[static_cast<int64_t>(cumulative) * v.P + pattern[j]] = cum[j];
      }
    }
  }
}

// Any category count: a thread owns a pattern and loops over its categories; a rescaled op
// re-reads what it wrote.
template <bool PRE>
__global__ void __launch_bounds__(kBlock) UpdatePartialsKernel(const InstanceView v, const DeviceOp* __restrict__ ops,
                                                              int op_count, int cumulative) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t k = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; k < v.P; k += stride) {
    for (int o = 0; o < op_count; o++) {
      const DeviceOp op = ops[o];
      double largest = 0.0;
      for (int c = 0; c < v.C; c++) {
        double d[4];
        largest = fmax(largest, OpTerm<PRE>(v, op, c, k, d));
        Store4(Partial(v, op.dest, c, k), d);
      }
      if (op.scale_write >= 0) {
        if (largest == 0.0) largest = 1.0;
        const double inverse = 1.0 / largest;
        for (int c = 0; c < v.C; c++) {
          double d[4];
          Load4(Partial(v, op.dest, c, k), d);
#pragma unroll
          for (int i = 0; i < 4; i++) d[i] *= inverse;
          Store4(Partial(v, op.dest, c, k), d);
        }
        v.scale[static_cast<size_t>(op.scale_write) * v.P + k] = largest;
        if (cumulative >= 0) v.scale[static_cast<size_t>(cumulative) * v.P + k] += log(largest);
      }
    }
  }
}

// P_c = V diag(exp(lambda r_c t)) V^-1, negative round-off clamped to 0
// (beagleUpdateTransitionMatrices, fat_beagle.cpp:304-314); one thread per (edge, category).
struct EigenSystem {
  double evec[16], ivec[16], eval[4];
};
__global__ void TransitionMatricesKernel(const EigenSystem eigen, const double* __restrict__ cat_rates, int C,
                                         const int32_t* __restrict__ indices, const double* __restrict__ lengths,
                                         int count, double* __restrict__ matrix) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= count * C) return;
  const int e = idx / C, c = idx % C;
  const double t = lengths[e] * cat_rates[c];
  double ex[4];
#pragma unroll
  for (int k = 0; k < 4; k++) ex[k] = exp(eigen.eval[k] * t);
  double* out = matrix + (static_cast<size_t>(indices[e]) * C + c) * 16;
#pragma unroll
  for (int i = 0; i < 4; i++)
#pragma unroll
    for (int j = 0; j < 4; j++) {
      double sum = 0.0;
#pragma unroll
      for (int k = 0; k < 4; k++) sum += (eigen.evec[i * 4 + k] * ex[k]) * eigen.ivec[k * 4 + j];
      out[i * 4 + j] = sum > 0.0 ? sum : 0.0;
    }
}

// Sum over a block, in a fixed order; valid in thread 0.
__device__ __forceinline__ double BlockSum(double value, double* smem) {
#pragma unroll
  for (int m = 16; m >= 1; m >>= 1) value += __shfl_xor_sync(0xffffffffu, value, m);
  if ((threadIdx.x & 31) == 0) smem[threadIdx.x >> 5] = value;
  __syncthreads();
  double total = 0.0;
  if (threadIdx.x == 0)
    for (int w = 0; w < kBlock / 32; w++) total += smem[w];
  __syncthreads();
  return total;
}

// beagleCalculateRootLogLikelihoods (fat_beagle.cpp:65-68, 170-173):
//   sum_k w_k (log sum_i pi_i sum_c p_c root[c,k,i] + cumulative_k)  -> per-block partial sums,
//   and every pattern's term before its weight -> site_logl (beagleGetSiteLogLikelihoods)
__global__ void __launch_bounds__(kBlock) RootLogLikelihoodKernel(const InstanceView v, int root, int cumulative,
                                                                 double* __restrict__ block_sums,
                                                                 double* __restrict__ site_logl) {
  __shared__ double smem[kBlock / 32];
  double local = 0.0;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t k = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; k < v.P; k += stride) {
    double over_categories[4] = {0.0, 0.0, 0.0, 0.0};
    for (int c = 0; c < v.C; c++) {
      double L[4];
      Load4(Partial(v, root, c, k), L);
#pragma unroll
      for (int i = 0; i < 4; i++) over_categories[i] += v.cat_weights[c] * L[i];
    }
    double site = 0.0;
#pragma unroll
    for (int i = 0; i < 4; i++) site += v.freqs[i] * over_categories[i];
    double log_site = log(site);
    if (cumulative >= 0) log_site += v.scale[static_cast<size_t>(cumulative) * v.P + k];
    site_logl[k] = log_site;
    local += v.pattern_weights[k] * log_site;
  }
  const double total = BlockSum(local, smem);
  if (threadIdx.x == 0) block_sums[blockIdx.x] = total;
}

// beagleCalculateEdgeDerivatives (fat_beagle.cpp:154-166), edge blockIdx.y:
//   per pattern [sum_c p_c pre^T dQ_c post] / [sum_c p_c pre^T post]; a compact tip acts as its
//   one-hot (or all-ones) partial.  Per-site values when asked, and per-block partial sums of
//   w_k x and w_k x^2.
//   G categories of a pattern are loaded together (2 G independent 256-bit loads in flight per
//   thread: the kernel is a pure stream, 82 % of its stalls were on the long scoreboard with one
//   category at a time); the differential matrices sit in shared memory.
constexpr int kMaxStagedCategories = 16;
template <int G>
__global__ void __launch_bounds__(kBlock) EdgeDerivativesKernel(const InstanceView v, const int32_t* __restrict__ post,
                                                               const int32_t* __restrict__ pre,
                                                               const int32_t* __restrict__ dmatrix,
                                                               double* __restrict__ per_site,
                                                               double* __restrict__ block_sums) {
  __shared__ double smem[kBlock / 32];
  __shared__ __align__(16) double s_dq[kMaxStagedCategories * 16];
  __shared__ double s_weights[kMaxStagedCategories];
  const int e = blockIdx.y;
  const int post_buffer = post[e], pre_buffer = pre[e];
  const double* dq_base = v.matrix + static_cast<size_t>(dmatrix[e]) * v.C * 16;
  const bool staged = v.C <= kMaxStagedCategories;
  if (staged) {
    for (int i = threadIdx.x; i < v.C * 16; i += kBlock) s_dq[i] = dq_base[i];
    for (int i = threadIdx.x; i < v.C; i += kBlock) s_weights[i] = v.cat_weights[i];
    __syncthreads();
  }
  const bool compact = v.is_compact[post_buffer];
  double sum = 0.0, sum_squares = 0.0;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t k = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; k < v.P; k += stride) {
    double numerator = 0.0, denominator = 0.0;
    const int s = compact ? v.compact[static_cast<size_t>(post_buffer) * v.P + k] : 0;
    for (int c0 = 0; c0 < v.C; c0 += G) {
      double x[G][4], p[G][4];
#pragma unroll
      for (int g = 0; g < G; g++) {
        if (compact) {
#pragma unroll
          for (int i = 0; i < 4; i++) x[g][i] = (s >= kStates || s == i) ? 1.0 : 0.0;
        } else {
          Load4(Partial(v, post_buffer, c0 + g, k), x[g]);
        }
        Load4(Partial(v, pre_buffer, c0 + g, k), p[g]);
      }
#pragma unroll
      for (int g = 0; g < G; g++) {
        const int c = c0 + g;
        double num_c = 0.0, den_c = 0.0;
#pragma unroll
        for (int i = 0; i < 4; i++) {
          double row[4];
          if (staged) {
            LoadShared4(s_dq + c * 16 + i * 4, row);
          } else {
            Load4(dq_base + c * 16 + i * 4, row);
          }
          const double dq_post = row[0] * x[g][0] + row[1] * x[g][1] + row[2] * x[g][2] + row[3] * x[g][3];
          num_c += p[g][i] * dq_post;
          den_c += p[g][i] * x[g][i];
        }
        const double weight = staged ? s_weights[c] : v.cat_weights[c];
        numerator += weight * num_c;
        denominator += weight * den_c;
      }
    }
    const double derivative = numerator / denominator;
    if (per_site != nullptr) per_site[static_cast<size_t>(e) * v.P + k] = derivative;
    sum += v.pattern_weights[k] * derivative;
    sum_squares += v.pattern_weights[k] * derivative * derivative;
  }
  const double total = BlockSum(sum, smem);
  const double total_squares = BlockSum(sum_squares, smem);
  if (threadIdx.x == 0) {
    block_sums[(static_cast<size_t>(e) * gridDim.x + blockIdx.x) * 2] = total;
    block_sums[(static_cast<size_t>(e) * gridDim.x + blockIdx.x) * 2 + 1] = total_squares;
  }
}

// out[r][x] = sum over the blocks of row r, in block order.
__global__ void SumBlocksKernel(const double* __restrict__ block_sums, int blocks, int width, int rows,
                                double* __restrict__ out) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * width) return;
  const int r = idx / width, x = idx % width;
  double total = 0.0;
  for (int b = 0; b < blocks; b++) total += block_sums[(static_cast<size_t>(r) * blocks + b) * width + x];
  out[idx] = total;
}

// beagleSetTipPartials: [pattern][state] replicated over the categories.
__global__ void ReplicateKernel(const double* __restrict__ in, int64_t block, int C, double* __restrict__ out) {
  const int64_t idx = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= block) return;
  const double value = in[idx];
  for (int c = 0; c < C; c++) out[c * block + idx] = value;
}

template <typename T>
struct DeviceBuffer {
  T* ptr = nullptr;
  size_t capacity = 0;
  ~DeviceBuffer() { cudaFree(ptr); }
  bool Reserve(size_t count) {
    if (count <= capacity) return true;
    cudaFree(ptr);
    ptr = nullptr;
    capacity = 0;
    if (cudaMalloc(&ptr, std::max<size_t>(count, 1) * sizeof(T)) != cudaSuccess) {
      cudaGetLastError();
      return false;
    }
    capacity = count;
    return true;
  }
};

struct Instance {
  int device = 0;
  int tips = 0, buffers = 0, P = 0, C = 0, matrices = 0, scalers = 0;
  int sm_count = 1;
  cudaStream_t stream = nullptr;
  cudaEvent_t begin = nullptr, end = nullptr;
  DeviceBuffer<double> partials, matrix, scale, cat_weights, cat_rates, freqs, pattern_weights, staging, sums, out;
  DeviceBuffer<double> site_logl;  // [P] of the last root call
  bool has_site_logl = false;
  DeviceBuffer<uint8_t> compact, is_compact;
  DeviceBuffer<int32_t> indices;
  DeviceBuffer<DeviceOp> ops;
  std::vector<uint8_t> is_compact_host;
  EigenSystem eigen{};
  double last_kernel_ms = 0.0;
  int64_t launches = 0;

  ~Instance() {
    if (begin) cudaEventDestroy(begin);
    if (end) cudaEventDestroy(end);
    if (stream) cudaStreamDestroy(stream);
  }
  InstanceView View() const {
    return InstanceView{tips,       buffers,        P,          C,           matrices,        scalers,
                        partials.ptr, compact.ptr, is_compact.ptr, matrix.ptr, scale.ptr, cat_weights.ptr,
                        freqs.ptr,  pattern_weights.ptr};
  }
  size_t PartialSize() const { return static_cast<size_t>(C) * P * kStates; }
  int PatternBlocks() const {
    const int64_t wanted = (static_cast<int64_t>(P) + kBlock - 1) / kBlock;
    return static_cast<int>(std::max<int64_t>(1, std::min<int64_t>(wanted, static_cast<int64_t>(sm_count) * 16)));
  }
};

std::mutex g_mutex;
std::vector<std::unique_ptr<Instance>> g_instances;

Instance* Get(int handle) {
  std::lock_guard<std::mutex> lock(g_mutex);
  if (handle < 0 || handle >= static_cast<int>(g_instances.size())) return nullptr;
  return g_instances[handle].get();
}

char g_resource_name[] = "NVIDIA B200 (libsbn_b200)";
char g_impl_name[] = "libhmsbeagle_b200: BEAGLE-compatible fp64 CUDA kernels for sm_100a";
char g_impl_desc[] = "op-at-a-time partial updates, partials materialised in HBM, one launch per call";

int Code(cudaError_t status) {
  if (status == cudaSuccess) return BEAGLE_SUCCESS;
  cudaGetLastError();
  return status == cudaErrorMemoryAllocation ? BEAGLE_ERROR_OUT_OF_MEMORY : BEAGLE_ERROR_GENERAL;
}
#define SHIM_CUDA(call)                                   \
  do {                                                    \
    const cudaError_t status_ = (call);                   \
    if (status_ != cudaSuccess) return Code(status_);     \
  } while (0)

// Host array -> device (the caller's memory is borrowed for the call only: the copy has
// left it when this returns).
template <typename T>
int Upload(Instance* inst, T* device, const T* host, size_t count) {
  SHIM_CUDA(cudaMemcpyAsync(device, host, count * sizeof(T), cudaMemcpyHostToDevice, inst->stream));
  SHIM_CUDA(cudaStreamSynchronize(inst->stream));
  return BEAGLE_SUCCESS;
}

int MarkCompact(Instance* inst, int buffer, bool compact) {
  if (inst->is_compact_host[buffer] == static_cast<uint8_t>(compact)) return BEAGLE_SUCCESS;
  inst->is_compact_host[buffer] = compact;
  return Upload(inst, inst->is_compact.ptr + buffer, inst->is_compact_host.data() + buffer, 1);
}

template <bool PRE>
int UpdatePartials(int instance, const BeagleOperation* operations, int count, int cumulative) {
  Instance* inst = Get(instance);
  if (!inst) return BEAGLE_ERROR_UNINITIALIZED_INSTANCE;
  if (count <= 0) return BEAGLE_SUCCESS;
  if (operations == nullptr) return BEAGLE_ERROR_OUT_OF_RANGE;
  if (cumulative != BEAGLE_OP_NONE && (cumulative < 0 || cumulative >= inst->scalers)) return BEAGLE_ERROR_OUT_OF_RANGE;
  SHIM_CUDA(cudaSetDevice(inst->device));
  std::vector<DeviceOp> ops(count);
  int previous_dest = -1;
  bool cumulative_in_register = true;  // unless an op of the list writes the cumulative buffer itself
  for (int o = 0; o < count; o++) {
    const BeagleOperation& op = operations[o];
    if (op.destinationPartials < 0 || op.destinationPartials >= inst->buffers || op.child1Partials < 0 ||
        op.child1Partials >= inst->buffers || op.child2Partials < 0 || op.child2Partials >= inst->buffers ||
        op.child1TransitionMatrix < 0 || op.child1TransitionMatrix >= inst->matrices ||
        op.child2TransitionMatrix < 0 || op.child2TransitionMatrix >= inst->matrices ||
        op.destinationScaleWrite >= inst->scalers)
      return BEAGLE_ERROR_OUT_OF_RANGE;
    // (a pre-order parent partial is never a compact tip)
    if (PRE && inst->is_compact_host[op.child1Partials]) return BEAGLE_ERROR_OUT_OF_RANGE;
    int32_t flags = 0;
    if (inst->is_compact_host[op.child1Partials]) {
      flags |= kChild1Compact;
    } else if (op.child1Partials == previous_dest) {
      flags |= kChild1Forward;
    }
    if (inst->is_compact_host[op.child2Partials]) {
      flags |= kChild2Compact;
    } else if (op.child2Partials == previous_dest) {
      flags |= kChild2Forward;
    }
    ops[o] = DeviceOp{op.destinationPartials, op.destinationScaleWrite < 0 ? -1 : op.destinationScaleWrite,
                      op.child1Partials,      op.child1TransitionMatrix,
                      op.child2Partials,      op.child2TransitionMatrix,
                      flags,                  0,
                      0,                      0,
                      0,                      0};
    const int64_t partial = static_cast<int64_t>(inst->PartialSize());
    ops[o].dest_at = op.destinationPartials * partial;
    ops[o].child1_at = (flags & kChild1Compact) ? static_cast<int64_t>(op.child1Partials) * inst->P : op.child1Partials * partial;
    ops[o].child2_at = (flags & kChild2Compact) ? static_cast<int64_t>(op.child2Partials) * inst->P : op.child2Partials * partial;
    ops[o].scale_at = static_cast<int64_t>(std::max(op.destinationScaleWrite, 0)) * inst->P;
    if (op.destinationScaleWrite >= 0 && op.destinationScaleWrite == cumulative) cumulative_in_register = false;
    const int status = MarkCompact(inst, op.destinationPartials, false);
    if (status != BEAGLE_SUCCESS) return status;
    previous_dest = op.destinationPartials;
  }
  if (!inst->ops.Reserve(count)) return BEAGLE_ERROR_OUT_OF_MEMORY;
  SHIM_CUDA(cudaMemcpyAsync(inst->ops.ptr, ops.data(), count * sizeof(DeviceOp), cudaMemcpyHostToDevice, inst->stream));
  const InstanceView view = inst->View();
  const int blocks = inst->PatternBlocks();
  const int cumulative_index = cumulative == BEAGLE_OP_NONE ? -1 : cumulative;
  SHIM_CUDA(cudaEventRecord(inst->begin, inst->stream));
  // K adjacent patterns per thread (SBNB_BEAGLE_PATTERNS_PER_THREAD = 2: twice the loads in flight
  // per thread, half the matrix reads, half the threads).
  int lanes = 1;  // lanes per pattern: the category count rounded up to a power of two (more than 16: the generic kernel)
  while (lanes < inst->C) lanes <<= 1;
  const int64_t lane_threads = static_cast<int64_t>(inst->P) * lanes;
  int K = 1;  // (two measured slower on the pre-order list and the same on the post-order one at 100k x 4)
  if (const char* forced = std::getenv("SBNB_BEAGLE_PATTERNS_PER_THREAD")) K = std::atoi(forced) >= 2 ? 2 : 1;
  if (lanes != inst->C) K = 1;  // (the padded form exists with one pattern per thread)
  const int lane_blocks =
      static_cast<int>(std::max<int64_t>(1, std::min<int64_t>((lane_threads + kPipeBlock * K - 1) / (kPipeBlock * K), 1 << 30)));
#define SHIM_LANES(CT)                                                                                        \
  case CT:                                                                                                    \
    if (inst->C != CT) {                                                                                      \
      UpdatePartialsPipelinedKernel<PRE, CT, 1, true><<<lane_blocks, kPipeBlock, 0, inst->stream>>>(          \
          view, inst->ops.ptr, count, cumulative_index, cumulative_in_register);                              \
    } else if (K == 2) {                                                                                      \
      UpdatePartialsPipelinedKernel<PRE, CT, 2, false><<<lane_blocks, kPipeBlock, 0, inst->stream>>>(         \
          view, inst->ops.ptr, count, cumulative_index, cumulative_in_register);                              \
    } else {                                                                                                  \
      UpdatePartialsPipelinedKernel<PRE, CT, 1, false><<<lane_blocks, kPipeBlock, 0, inst->stream>>>(         \
          view, inst->ops.ptr, count, cumulative_index, cumulative_in_register);                              \
    }                                                                                                         \
    break;
  switch (lanes) {
    SHIM_LANES(1)
    SHIM_LANES(2)
    SHIM_LANES(4)
    SHIM_LANES(8)
    SHIM_LANES(16)
    default:
      UpdatePartialsKernel<PRE><<<blocks, kBlock, 0, inst->stream>>>(view, inst->ops.ptr, count, cumulative_index);
  }
#undef SHIM_LANES
  SHIM_CUDA(cudaGetLastError());
  SHIM_CUDA(cudaEventRecord(inst->end, inst->stream));
  inst->launches++;
  // BEAGLE_FLAG_COMPUTATION_SYNCH: the call returns when the work is done (the ops vector above
  // is also borrowed by the copy until then).
  SHIM_CUDA(cudaStreamSynchronize(inst->stream));
  float ms = 0.f;
  SHIM_CUDA(cudaEventElapsedTime(&ms, inst->begin, inst->end));
  inst->last_kernel_ms = ms;
  return BEAGLE_SUCCESS;
}

}  // namespace

extern "C" {

int beagleCreateInstance(int tipCount, int partialsBufferCount, int compactBufferCount, int stateCount,
                         int patternCount, int eigenBufferCount, int matrixBufferCount, int categoryCount,
                         int scaleBufferCount, int* resourceList, int resourceCount, long preferenceFlags,
                         long requirementFlags, BeagleInstanceDetails* returnInfo) {
  if (tipCount < 1 || stateCount < 1 || patternCount < 0 || categoryCount < 1 || eigenBufferCount < 1 ||
      partialsBufferCount < 0 || compactBufferCount < 0 || matrixBufferCount < 0 || scaleBufferCount < 0)
    return BEAGLE_ERROR_OUT_OF_RANGE;
  if (stateCount != kStates) return BEAGLE_ERROR_NO_IMPLEMENTATION;  // nucleotides, as the reference uses it
  if (requirementFlags & BEAGLE_FLAG_PRECISION_SINGLE) return BEAGLE_ERROR_NO_IMPLEMENTATION;  // fp64 only
  (void)preferenceFlags;
  int device_count = 0;
  if (cudaGetDeviceCount(&device_count) != cudaSuccess || device_count < 1) {
    cudaGetLastError();
    return BEAGLE_ERROR_NO_RESOURCE;  // no CPU fallback
  }
  auto inst = std::make_unique<Instance>();
  // BEAGLE numbers resources from the CPU (0): resource r >= 1 is GPU r - 1.  Without a list,
  // SBNB_BEAGLE_DEVICE picks the GPU (default 0).
  inst->device = 0;
  if (resourceList != nullptr && resourceCount > 0 && resourceList[0] >= 1) inst->device = resourceList[0] - 1;
  if (const char* forced = std::getenv("SBNB_BEAGLE_DEVICE")) inst->device = std::atoi(forced);
  if (inst->device < 0 || inst->device >= device_count) return BEAGLE_ERROR_NO_RESOURCE;
  SHIM_CUDA(cudaSetDevice(inst->device));
  cudaDeviceProp prop{};
  SHIM_CUDA(cudaGetDeviceProperties(&prop, inst->device));
  inst->sm_count = prop.multiProcessorCount;
  inst->tips = tipCount;
  inst->buffers = partialsBufferCount + compactBufferCount;
  inst->P = patternCount;
  inst->C = categoryCount;
  inst->matrices = matrixBufferCount;
  inst->scalers = scaleBufferCount;
  SHIM_CUDA(cudaStreamCreateWithFlags(&inst->stream, cudaStreamNonBlocking));
  SHIM_CUDA(cudaEventCreate(&inst->begin));
  SHIM_CUDA(cudaEventCreate(&inst->end));
  const size_t P = std::max(patternCount, 1);
  bool ok = inst->partials.Reserve(static_cast<size_t>(inst->buffers) * inst->PartialSize()) &&
            inst->compact.Reserve(static_cast<size_t>(tipCount) * P) && inst->is_compact.Reserve(inst->buffers) &&
            inst->matrix.Reserve(static_cast<size_t>(matrixBufferCount) * categoryCount * 16) &&
            inst->scale.Reserve(static_cast<size_t>(scaleBufferCount) * P) && inst->cat_weights.Reserve(categoryCount) &&
            inst->cat_rates.Reserve(categoryCount) && inst->freqs.Reserve(kStates) && inst->pattern_weights.Reserve(P);
  if (!ok) return BEAGLE_ERROR_OUT_OF_MEMORY;
  SHIM_CUDA(cudaMemsetAsync(inst->partials.ptr, 0, static_cast<size_t>(inst->buffers) * inst->PartialSize() * sizeof(double),
                            inst->stream));
  SHIM_CUDA(cudaMemsetAsync(inst->matrix.ptr, 0, static_cast<size_t>(matrixBufferCount) * categoryCount * 16 * sizeof(double),
                            inst->stream));
  SHIM_CUDA(cudaMemsetAsync(inst->scale.ptr, 0, static_cast<size_t>(scaleBufferCount) * P * sizeof(double), inst->stream));
  SHIM_CUDA(cudaMemsetAsync(inst->is_compact.ptr, 0, inst->buffers, inst->stream));
  inst->is_compact_host.assign(inst->buffers, 0);
  // BEAGLE's defaults: unit rates, equal category weights and frequencies, unit pattern weights.
  const std::vector<double> ones(std::max<size_t>(P, categoryCount), 1.0);
  const std::vector<double> equal_categories(categoryCount, 1.0 / categoryCount), equal_states(kStates, 1.0 / kStates);
  int status = Upload(inst.get(), inst->cat_rates.ptr, ones.data(), categoryCount);
  if (status == BEAGLE_SUCCESS) status = Upload(inst.get(), inst->cat_weights.ptr, equal_categories.data(), categoryCount);
  if (status == BEAGLE_SUCCESS) status = Upload(inst.get(), inst->freqs.ptr, equal_states.data(), kStates);
  if (status == BEAGLE_SUCCESS) status = Upload(inst.get(), inst->pattern_weights.ptr, ones.data(), patternCount);
  if (status != BEAGLE_SUCCESS) return status;
  if (returnInfo != nullptr) {
    returnInfo->resourceNumber = inst->device + 1;
    returnInfo->resourceName = g_resource_name;
    returnInfo->implName = g_impl_name;
    returnInfo->implDescription = g_impl_desc;
    returnInfo->flags = BEAGLE_FLAG_PRECISION_DOUBLE | BEAGLE_FLAG_COMPUTATION_SYNCH | BEAGLE_FLAG_EIGEN_REAL |
                        BEAGLE_FLAG_SCALING_MANUAL | BEAGLE_FLAG_SCALERS_RAW | BEAGLE_FLAG_VECTOR_NONE |
                        BEAGLE_FLAG_THREADING_NONE | BEAGLE_FLAG_PROCESSOR_GPU | BEAGLE_FLAG_FRAMEWORK_CUDA |
                        BEAGLE_FLAG_INVEVEC_STANDARD | BEAGLE_FLAG_PARALLELOPS_GRID;
  }
  std::lock_guard<std::mutex> lock(g_mutex);
  for (size_t h = 0; h < g_instances.size(); h++) {
    if (!g_instances[h]) {
      g_instances[h] = std::move(inst);
      return static_cast<int>(h);
    }
  }
  g_instances.push_back(std::move(inst));
  return static_cast<int>(g_instances.size()) - 1;
}

int beagleFinalizeInstance(int instance) {
  std::unique_ptr<Instance> doomed;
  {
    std::lock_guard<std::mutex> lock(g_mutex);
    if (instance < 0 || instance >= static_cast<int>(g_instances.size()) || !g_instances[instance])
      return BEAGLE_ERROR_UNINITIALIZED_INSTANCE;
    doomed = std::move(g_instances[instance]);
  }
  cudaSetDevice(doomed->device);
  cudaStreamSynchronize(doomed->stream);
  return BEAGLE_SUCCESS;
}

int beagleSetTipStates(int instance, int tipIndex, const int* inStates) {
  Instance* inst = Get(instance);
  if (!inst) return BEAGLE_ERROR_UNINITIALIZED_INSTANCE;
  if (tipIndex < 0 || tipIndex >= inst->tips || inStates == nullptr) return BEAGLE_ERROR_OUT_OF_RANGE;
  SHIM_CUDA(cudaSetDevice(inst->device));
  std::vector<uint8_t> states(inst->P);
  for (int k = 0; k < inst->P; k++) states[k] = (inStates[k] < 0 || inStates[k] > kStates) ? kStates : inStates[k];
  const int status = Upload(inst, inst->compact.ptr + static_cast<size_t>(tipIndex) * inst->P, states.data(), inst->P);
  return status != BEAGLE_SUCCESS ? status : MarkCompact(inst, tipIndex, true);
}

int beagleSetTipPartials(int instance, int tipIndex, const double* inPartials) {
  Instance* inst = Get(instance);
  if (!inst) return BEAGLE_ERROR_UNINITIALIZED_INSTANCE;
  if (tipIndex < 0 || tipIndex >= inst->tips || inPartials == nullptr) return BEAGLE_ERROR_OUT_OF_RANGE;
  SHIM_CUDA(cudaSetDevice(inst->device));
  const int64_t block = static_cast<int64_t>(inst->P) * kStates;
  if (!inst->staging.Reserve(block)) return BEAGLE_ERROR_OUT_OF_MEMORY;
  SHIM_CUDA(cudaMemcpyAsync(inst->staging.ptr, inPartials, block * sizeof(double), cudaMemcpyHostToDevice, inst->stream));
  if (block > 0) {
    ReplicateKernel<<<static_cast<unsigned>((block + 255) / 256), 256, 0, inst->stream>>>(
        inst->staging.ptr, block, inst->C, inst->partials.ptr + static_cast<size_t>(tipIndex) * inst->PartialSize());
    SHIM_CUDA(cudaGetLastError());
    inst->launches++;
  }
  SHIM_CUDA(cudaStreamSynchronize(inst->stream));
  return MarkCompact(inst, tipIndex, false);
}

int beagleSetPartials(int instance, int bufferIndex, const double* inPartials) {
  Instance* inst = Get(instance);
  if (!inst) return BEAGLE_ERROR_UNINITIALIZED_INSTANCE;
  if (bufferIndex < 0 || bufferIndex >= inst->buffers || inPartials == nullptr) return BEAGLE_ERROR_OUT_OF_RANGE;
  SHIM_CUDA(cudaSetDevice(inst->device));
  const int status = Upload(inst, inst->partials.ptr + static_cast<size_t>(bufferIndex) * inst->PartialSize(), inPartials,
                            inst->PartialSize());
  return status != BEAGLE_SUCCESS ? status : MarkCompact(inst, bufferIndex, false);
}

int beagleSetPatternWeights(int instance, const double* inPatternWeights) {
  Instance* inst = Get(instance);
  if (!inst) return BEAGLE_ERROR_UNINITIALIZED_INSTANCE;
  if (inPatternWeights == nullptr) return BEAGLE_ERROR_OUT_OF_RANGE;
  SHIM_CUDA(cudaSetDevice(inst->device));
  return Upload(inst, inst->pattern_weights.ptr, inPatternWeights, inst->P);
}

int beagleSetCategoryWeights(int instance, int categoryWeightsIndex, const double* inCategoryWeights) {
  Instance* inst = Get(instance);
  if (!inst) return BEAGLE_ERROR_UNINITIALIZED_INSTANCE;
  if (categoryWeightsIndex != 0 || inCategoryWeights == nullptr) return BEAGLE_ERROR_OUT_OF_RANGE;
  SHIM_CUDA(cudaSetDevice(inst->device));
  return Upload(inst, inst->cat_weights.ptr, inCategoryWeights, inst->C);
}

int beagleSetCategoryRates(int instance, const double* inCategoryRates) {
  Instance* inst = Get(instance);
  if (!inst) return BEAGLE_ERROR_UNINITIALIZED_INSTANCE;
  if (inCategoryRates == nullptr) return BEAGLE_ERROR_OUT_OF_RANGE;
  SHIM_CUDA(cudaSetDevice(inst->device));
  return Upload(inst, inst->cat_rates.ptr, inCategoryRates, inst->C);
}

int beagleSetStateFrequencies(int instance, int stateFrequenciesIndex, const double* inStateFrequencies) {
  Instance* inst = Get(instance);
  if (!inst) return BEAGLE_ERROR_UNINITIALIZED_INSTANCE;
  if (stateFrequenciesIndex != 0 || inStateFrequencies == nullptr) return BEAGLE_ERROR_OUT_OF_RANGE;
  SHIM_CUDA(cudaSetDevice(inst->device));
  return Upload(inst, inst->freqs.ptr, inStateFrequencies, kStates);
}

int beagleSetEigenDecomposition(int instance, int eigenIndex, const double* inEigenVectors,
                                const double* inInverseEigenVectors, const double* inEigenValues) {
  Instance* inst = Get(instance);
  if (!inst) return BEAGLE_ERROR_UNINITIALIZED_INSTANCE;
  if (eigenIndex != 0 || !inEigenVectors || !inInverseEigenVectors || !inEigenValues) return BEAGLE_ERROR_OUT_OF_RANGE;
  std::copy(inEigenVectors, inEigenVectors + 16, inst->eigen.evec);
  std::copy(inInverseEigenVectors, inInverseEigenVectors + 16, inst->eigen.ivec);
  std::copy(inEigenValues, inEigenValues + 4, inst->eigen.eval);
  return BEAGLE_SUCCESS;
}

int beagleUpdateTransitionMatrices(int instance, int eigenIndex, const int* probabilityIndices,
                                   const int* firstDerivativeIndices, const int* secondDerivativeIndices,
                                   const double* edgeLengths, int count) {
  Instance* inst = Get(instance);
  if (!inst) return BEAGLE_ERROR_UNINITIALIZED_INSTANCE;
  if (eigenIndex != 0) return BEAGLE_ERROR_OUT_OF_RANGE;
  // The reference always passes NULL derivative index lists (fat_beagle.cpp:310-311).
  if (firstDerivativeIndices != nullptr || secondDerivativeIndices != nullptr) return BEAGLE_ERROR_NO_IMPLEMENTATION;
  if (count <= 0) return BEAGLE_SUCCESS;
  if (probabilityIndices == nullptr || edgeLengths == nullptr) return BEAGLE_ERROR_OUT_OF_RANGE;
  for (int e = 0; e < count; e++)
    if (probabilityIndices[e] < 0 || probabilityIndices[e] >= inst->matrices) return BEAGLE_ERROR_OUT_OF_RANGE;
  SHIM_CUDA(cudaSetDevice(inst->device));
  if (!inst->indices.Reserve(count) || !inst->staging.Reserve(count)) return BEAGLE_ERROR_OUT_OF_MEMORY;
  SHIM_CUDA(cudaMemcpyAsync(inst->indices.ptr, probabilityIndices, count * sizeof(int32_t), cudaMemcpyHostToDevice,
                            inst->stream));
  SHIM_CUDA(cudaMemcpyAsync(inst->staging.ptr, edgeLengths, count * sizeof(double), cudaMemcpyHostToDevice, inst->stream));
  const int jobs = count * inst->C;
  TransitionMatricesKernel<<<(jobs + 127) / 128, 128, 0, inst->stream>>>(inst->eigen, inst->cat_rates.ptr, inst->C,
                                                                         inst->indices.ptr, inst->staging.ptr, count,
                                                                         inst->matrix.ptr);
  SHIM_CUDA(cudaGetLastError());
  inst->launches++;
  SHIM_CUDA(cudaStreamSynchronize(inst->stream));
  return BEAGLE_SUCCESS;
}

int beagleSetDifferentialMatrix(int instance, int matrixIndex, const double* inMatrix) {
  Instance* inst = Get(instance);
  if (!inst) return BEAGLE_ERROR_UNINITIALIZED_INSTANCE;
  if (matrixIndex < 0 || matrixIndex >= inst->matrices || inMatrix == nullptr) return BEAGLE_ERROR_OUT_OF_RANGE;
  SHIM_CUDA(cudaSetDevice(inst->device));
  return Upload(inst, inst->matrix.ptr + static_cast<size_t>(matrixIndex) * inst->C * 16, inMatrix,
                static_cast<size_t>(inst->C) * 16);
}

int beagleResetScaleFactors(int instance, int cumulativeScaleIndex) {
  Instance* inst = Get(instance);
  if (!inst) return BEAGLE_ERROR_UNINITIALIZED_INSTANCE;
  if (cumulativeScaleIndex < 0 || cumulativeScaleIndex >= inst->scalers) return BEAGLE_ERROR_OUT_OF_RANGE;
  SHIM_CUDA(cudaSetDevice(inst->device));
  SHIM_CUDA(cudaMemsetAsync(inst->scale.ptr + static_cast<size_t>(cumulativeScaleIndex) * inst->P, 0,
                            static_cast<size_t>(inst->P) * sizeof(double), inst->stream));
  return BEAGLE_SUCCESS;
}

int beagleUpdatePartials(int instance, const BeagleOperation* operations, int operationCount,
                         int cumulativeScaleIndex) {
  return UpdatePartials<false>(instance, operations, operationCount, cumulativeScaleIndex);
}

int beagleUpdatePrePartials(int instance, const BeagleOperation* operations, int operationCount,
                            int cumulativeScaleIndex) {
  return UpdatePartials<true>(instance, operations, operationCount, cumulativeScaleIndex);
}

int beagleCalculateEdgeDerivatives(int instance, const int* postBufferIndices, const int* preBufferIndices,
                                   const int* derivativeMatrixIndices, const int* categoryWeightsIndices, int count,
                                   double* outDerivatives, double* outSumDerivatives,
                                   double* outSumSquaredDerivatives) {
  Instance* inst = Get(instance);
  if (!inst) return BEAGLE_ERROR_UNINITIALIZED_INSTANCE;
  if (count <= 0) return BEAGLE_SUCCESS;
  if (!postBufferIndices || !preBufferIndices || !derivativeMatrixIndices || !categoryWeightsIndices ||
      categoryWeightsIndices[0] != 0)
    return BEAGLE_ERROR_OUT_OF_RANGE;
  for (int e = 0; e < count; e++)
    if (postBufferIndices[e] < 0 || postBufferIndices[e] >= inst->buffers || preBufferIndices[e] < 0 ||
        preBufferIndices[e] >= inst->buffers || derivativeMatrixIndices[e] < 0 ||
        derivativeMatrixIndices[e] >= inst->matrices || inst->is_compact_host[preBufferIndices[e]])
      return BEAGLE_ERROR_OUT_OF_RANGE;
  SHIM_CUDA(cudaSetDevice(inst->device));
  const int blocks = std::min(inst->PatternBlocks(), 64);
  const size_t per_site_count = outDerivatives ? static_cast<size_t>(count) * inst->P : 0;
  if (!inst->indices.Reserve(3 * static_cast<size_t>(count)) ||
      !inst->sums.Reserve(static_cast<size_t>(count) * blocks * 2) ||
      !inst->out.Reserve(2 * static_cast<size_t>(count) + per_site_count))
    return BEAGLE_ERROR_OUT_OF_MEMORY;
  std::vector<int32_t> indices(3 * static_cast<size_t>(count));
  std::copy(postBufferIndices, postBufferIndices + count, indices.begin());
  std::copy(preBufferIndices, preBufferIndices + count, indices.begin() + count);
  std::copy(derivativeMatrixIndices, derivativeMatrixIndices + count, indices.begin() + 2 * count);
  SHIM_CUDA(cudaMemcpyAsync(inst->indices.ptr, indices.data(), indices.size() * sizeof(int32_t), cudaMemcpyHostToDevice,
                            inst->stream));
  double* per_site = outDerivatives ? inst->out.ptr + 2 * static_cast<size_t>(count) : nullptr;
  SHIM_CUDA(cudaEventRecord(inst->begin, inst->stream));
  const dim3 derivative_grid(blocks, count);
#ifndef SBNB_SHIM_DERIV_G
#define SBNB_SHIM_DERIV_G 1  // (categories loaded together: 2 and 4 measured 4 % and 27 % SLOWER at 100k x 4 -- more concurrent DRAM streams)
#endif
  if (inst->C % 4 == 0 && SBNB_SHIM_DERIV_G >= 4) {
    EdgeDerivativesKernel<4><<<derivative_grid, kBlock, 0, inst->stream>>>(inst->View(), inst->indices.ptr,
                                                                          inst->indices.ptr + count,
                                                                          inst->indices.ptr + 2 * count, per_site,
                                                                          inst->sums.ptr);
  } else if (inst->C % 2 == 0 && SBNB_SHIM_DERIV_G >= 2) {
    EdgeDerivativesKernel<2><<<derivative_grid, kBlock, 0, inst->stream>>>(inst->View(), inst->indices.ptr,
                                                                          inst->indices.ptr + count,
                                                                          inst->indices.ptr + 2 * count, per_site,
                                                                          inst->sums.ptr);
  } else {
    EdgeDerivativesKernel<1><<<derivative_grid, kBlock, 0, inst->stream>>>(inst->View(), inst->indices.ptr,
                                                                          inst->indices.ptr + count,
                                                                          inst->indices.ptr + 2 * count, per_site,
                                                                          inst->sums.ptr);
  }
  SHIM_CUDA(cudaGetLastError());
  SumBlocksKernel<<<(2 * count + 127) / 128, 128, 0, inst->stream>>>(inst->sums.ptr, blocks, 2, count, inst->out.ptr);
  SHIM_CUDA(cudaGetLastError());
  SHIM_CUDA(cudaEventRecord(inst->end, inst->stream));
  inst->launches += 2;
  std::vector<double> sums(2 * static_cast<size_t>(count));
  SHIM_CUDA(cudaMemcpyAsync(sums.data(), inst->out.ptr, sums.size() * sizeof(double), cudaMemcpyDeviceToHost, inst->stream));
  if (outDerivatives)
    SHIM_CUDA(cudaMemcpyAsync(outDerivatives, per_site, per_site_count * sizeof(double), cudaMemcpyDeviceToHost,
                              inst->stream));
  SHIM_CUDA(cudaStreamSynchronize(inst->stream));
  float ms = 0.f;
  SHIM_CUDA(cudaEventElapsedTime(&ms, inst->begin, inst->end));
  inst->last_kernel_ms = ms;
  for (int e = 0; e < count; e++) {
    if (outSumDerivatives) outSumDerivatives[e] = sums[2 * e];
    if (outSumSquaredDerivatives) outSumSquaredDerivatives[e] = sums[2 * e + 1];
  }
  return BEAGLE_SUCCESS;
}

int beagleCalculateRootLogLikelihoods(int instance, const int* bufferIndices, const int* categoryWeightsIndices,
                                      const int* stateFrequenciesIndices, const int* cumulativeScaleIndices, int count,
                                      double* outSumLogLikelihood) {
  Instance* inst = Get(instance);
  if (!inst) return BEAGLE_ERROR_UNINITIALIZED_INSTANCE;
  if (count != 1) return BEAGLE_ERROR_NO_IMPLEMENTATION;  // fat_beagle passes 1
  if (!bufferIndices || !categoryWeightsIndices || !stateFrequenciesIndices || !cumulativeScaleIndices ||
      !outSumLogLikelihood)
    return BEAGLE_ERROR_OUT_OF_RANGE;
  const int root = bufferIndices[0], cumulative = cumulativeScaleIndices[0];
  if (root < 0 || root >= inst->buffers || inst->is_compact_host[root] || categoryWeightsIndices[0] != 0 ||
      stateFrequenciesIndices[0] != 0)
    return BEAGLE_ERROR_OUT_OF_RANGE;
  if (cumulative != BEAGLE_OP_NONE && (cumulative < 0 || cumulative >= inst->scalers)) return BEAGLE_ERROR_OUT_OF_RANGE;
  SHIM_CUDA(cudaSetDevice(inst->device));
  const int blocks = std::min(inst->PatternBlocks(), 256);
  if (!inst->sums.Reserve(blocks) || !inst->out.Reserve(1) || !inst->site_logl.Reserve(std::max(inst->P, 1)))
    return BEAGLE_ERROR_OUT_OF_MEMORY;
  RootLogLikelihoodKernel<<<blocks, kBlock, 0, inst->stream>>>(
      inst->View(), root, cumulative == BEAGLE_OP_NONE ? -1 : cumulative, inst->sums.ptr, inst->site_logl.ptr);
  SHIM_CUDA(cudaGetLastError());
  SumBlocksKernel<<<1, 32, 0, inst->stream>>>(inst->sums.ptr, blocks, 1, 1, inst->out.ptr);
  SHIM_CUDA(cudaGetLastError());
  inst->launches += 2;
  double total = 0.0;
  SHIM_CUDA(cudaMemcpyAsync(&total, inst->out.ptr, sizeof(double), cudaMemcpyDeviceToHost, inst->stream));
  SHIM_CUDA(cudaStreamSynchronize(inst->stream));
  *outSumLogLikelihood = total;
  inst->has_site_logl = true;
  return std::isnan(total) ? BEAGLE_ERROR_FLOATING_POINT : BEAGLE_SUCCESS;
}

// The values the last root call stored (not recomputed: the root buffer may have changed since).
int beagleGetSiteLogLikelihoods(int instance, double* outLogLikelihoods) {
  Instance* inst = Get(instance);
  if (!inst) return BEAGLE_ERROR_UNINITIALIZED_INSTANCE;
  if (!outLogLikelihoods) return BEAGLE_ERROR_OUT_OF_RANGE;
  if (!inst->has_site_logl) return BEAGLE_ERROR_GENERAL;  // no beagleCalculateRootLogLikelihoods yet
  SHIM_CUDA(cudaSetDevice(inst->device));
  SHIM_CUDA(cudaMemcpyAsync(outLogLikelihoods, inst->site_logl.ptr, static_cast<size_t>(inst->P) * sizeof(double),
                            cudaMemcpyDeviceToHost, inst->stream));
  SHIM_CUDA(cudaStreamSynchronize(inst->stream));
  return BEAGLE_SUCCESS;
}

// Not BEAGLE: diagnostics of this implementation (device time, ms by CUDA events, of the last
// UpdatePartials / UpdatePrePartials / CalculateEdgeDerivatives call; kernels launched so far).
double sbnbBeagleLastKernelMs(int instance) {
  Instance* inst = Get(instance);
  return inst ? inst->last_kernel_ms : -1.0;
}
long sbnbBeagleLaunchCount(int instance) {
  Instance* inst = Get(instance);
  return inst ? static_cast<long>(inst->launches) : -1;
}

}  // extern "C"
