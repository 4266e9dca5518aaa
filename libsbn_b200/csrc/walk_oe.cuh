// TreeWalkOeKernel: the tree walk (v6), lanes = (site pattern, rate category), with
// the pre-order half in "own-edge" form.
//
// One pass over a tree for a tile of site patterns -- post-order partial updates,
// per-pattern power-of-two rescaling, the root log-likelihood and (gradient mode) the
// pre-order pass fused with all edge derivatives [replaces beagleUpdatePartials,
// beagleUpdatePrePartials, beagleCalculateEdgeDerivatives,
// beagleCalculateRootLogLikelihoods, beagleResetScaleFactors and
// beagleSetPartials(root pre := pi); fat_beagle.cpp:50-70, 119-175].
//
// Site patterns are independent, so a warp owns a tile of them and walks the WHOLE
// tree for it; the C lanes of a pattern each own one rate category and a thread holds
// K patterns x 1 category x 4 states.  The walk order (host-generated,
// Strahler-ordered, tree_program.cpp) keeps the result of the previous op in
// registers ("cur"); only nodes with two internal children touch a small
// thread-private stack.
//
// Post-order op of node v with children a, b:  cur = y_a o y_b,  y_x = P_x L_x
// (a mat-vec for an internal child, a table row for a tip).  In gradient mode the
// y of internal children go to the warp's arena block of v (written once).
//
// Pre-order op of node v.  cur = T_v, the partial at the TOP of v's edge (everything
// outside v's subtree, seen from v's parent; root: pi, no edge).
//     pp  = P_v^T T_v                       the pre-order partial at v
//     L   = y_a o y_b                       (y read back from the arena / tip tables)
//     den = pp . L                          the site likelihood (shared by all edges)
//     own edge:   num = T_v^T Q P_v L = pp . (Q L)         (Q and P commute)
//     tip child a: num = T_a . (Q P_a)[:, state],  T_a = pp o y_b
//     internal child a: T_a stays in cur or is pushed; its derivative is computed at
//     a's own op.
// So every op does at most ONE P mat-vec and ONE Q mat-vec (the previous kernel did up
// to two of each, with both children's pre-order partials live: 232 registers, 8
// warps per SM; this form fits 12 warps per SM, and the walk is bound by dependency
// latency per warp -- one resident CTA fewer costs ~40 % of the throughput).
//
// Everything an op needs besides partials arrives in a shared-memory ring by TMA
// bulk copies (cp.async.bulk + mbarrier full/empty pairs): ONE copy of the op's
// operand block -- laid out per op by TransitionMatrixOeKernel: a header with the
// op's own record and the record of the op kOePrefetchOps ahead, then exactly the
// matrices / tip tables the op reads -- plus the tile's tip states of tip children.
// The first warp to reach op g wins a shared-memory ticket and requests op
// g + kOePrefetchOps from the record it finds in op g's header (no global load on
// that path).  Evolved partials come back through ONE per-warp bulk copy per
// (op, sub-batch) that completes on the warp's own mbarrier: a warp only reads what
// it wrote itself, so no CTA-wide barrier is involved.
#ifndef SBNB_WALK_OE_CUH_
#define SBNB_WALK_OE_CUH_

#include "kernels.cuh"

namespace sbnb {

// One op of the walk: 32 bytes.  Post-order ops (first n-1 of a program) and
// pre-order ops (last n-1) share the layout.
struct alignas(16) OeOp {
  int32_t operand_unit;   // first 16-byte unit of the op's operand block inside a (virtual) tree's block
  int32_t operand_units;  // its size in 16-byte units (header included)
  int32_t tip_a, tip_b;   // node (= taxon) id of a tip child, else -1
  int32_t node_flags;     // node id | flags << 24
  int32_t slots;          // post: push_slot | b's pop slot << 16;  pre: pop_slot | b's push slot << 16   (0xff = none)
  int32_t arena_slot;     // first arena block of this op's internal children
  int32_t next_arena_slot;  // the same of the NEXT pre-order op (whose read-back this op starts)
};
static_assert(sizeof(OeOp) == 32, "op records are two 16-byte words");
// flags beyond kALeaf | kBLeaf | kRoot | kStackBefore: kArenaSwapped (pre-order op with two
// internal children whose arena blocks are in the other order) and the leaf flags of the next
// pre-order op (how many blocks its read-back fetches)
enum : int32_t { kArenaSwapped = 16, kNextALeaf = 64, kNextBLeaf = 128 };

// Operand block of one op, in doubles (C = padded category count):
//   [0, 8)    header: the op's own record, then the record of the op kOePrefetchOps ahead
//   post-order op:  child a part, child b part; a part is P_c row-major, 18 doubles
//                   apart (internal child) or per c: P_c^T + a row of ones (tip child)
//   pre-order op:   own P (18 C; an identity at the root), then per TIP child 40 C:
//                   per c P_c^T + ones, per c (Q P_c)^T + zeros
constexpr int kOeHeaderDoubles = 8;
// (with the analytic substitution gradient every edge's part of a pre-order block is
//  followed by Phi_c, 16 doubles per category: see OeMatrixParams::with_subst)
constexpr int kOePhiDoubles = 16;
__host__ __device__ constexpr int OeMaxOperandDoubles(int C, bool subst = false) {
  return kOeHeaderDoubles + (kPStride + 4 * kTipTableDoubles + (subst ? 3 * kOePhiDoubles : 0)) * C;
}

struct OeParams {
  const uint8_t* tips;  // [taxon][tip_pitch], padded with gap states
  int64_t tip_pitch;
  const double* weights;  // [tip_pitch] padded with zeros
  int64_t pattern_begin, pattern_end;
  int32_t taxon_count;
  const OeOp* ops;  // [program][2(n-1)]
  int32_t vtree_begin, vtree_count;
  const int32_t* vtree_program;
  const int32_t* vtree_model;
  const ModelTables* models;
  const double* operands;        // operand blocks of vtrees [operand_origin, ...)
  int32_t operand_origin;        // first vtree held in `operands`
  int64_t operand_stride;        // doubles per vtree
  int32_t tiles_total, tiles_per_chunk, chunks;
  int32_t slots;           // stack depth
  double2* stack;          // [grid][slots][K][2][kThreads]
  int32_t* stack_exps;     // [grid][slots][K][kThreads]              (rescaling)
  double2* arena;          // [grid][n-2 blocks][K][2][kThreads]      (gradient mode)
  double* logl_partial;    // [vtree][chunk][warp]
  double* grad_partial;    // [vtree][chunk][warp][2n-1]               (gradient mode)
  double* rgrad_partial;   // same, with d rate_c / d shape as the scalers (C > 1)
  double* subst_partial;   // [vtree][chunk][warp][kOeSubstSums]        (analytic substitution gradient)
  const uint8_t* invariant_masks;  // [tip_pitch] the states every tip allows, per pattern (+I; 0 = padding)
  double* inv_partial;     // [vtree][chunk][warp][kOeInvariantSums]    (+I gradient runs)
  double* site_logl;       // [vtree][pattern - pattern_begin] log site likelihoods (SITES walks)
};

// ---------------------------------------------------------------------------
// TransitionMatrixOeKernel: per (virtual tree, edge, category) P = V diag(exp(lambda r_c t)) V^-1,
// written where the ops that read it will find it [replaces
// beagleUpdateTransitionMatrices, fat_beagle.cpp:304-314, and
// beagleSetDifferentialMatrix, fat_beagle.cpp:128-131]: into the post-order operand
// block of the edge's parent (P, or for a tip P^T + a row of ones) and, when the run
// has a pre-order half, into the pre-order block of the edge's own node (P) or of its
// parent (tip: P^T + ones and (Q P)^T + zeros).  The threads past the matrix jobs copy
// the op records into the block headers.
struct OeMatrixParams {
  const ModelTables* models;
  const int32_t* vtree_model;
  const int32_t* vtree_lengths;
  const int32_t* vtree_program;
  const double* branch_lengths;  // [tree][2n-1]
  const int2* edge_offsets;      // [program][2n-2]: doubles from the block start to the edge's post / pre part
  const OeOp* ops;               // [program][2(n-1)]
  double* operands;              // blocks of vtrees [vtree_begin, vtree_begin + vtree_count)
  int64_t operand_stride;        // doubles per vtree
  int32_t vtree_begin, vtree_count;
  int32_t taxon_count;
  int32_t categories;   // padded
  int32_t with_pre;     // the run has a pre-order half
  int32_t with_subst;   // ... whose blocks also carry Phi for the analytic substitution gradient:
                        //     Phi_kl = (e^{l_k tau} - e^{l_l tau}) / (l_k - l_l), tau e^{l_k tau} on the
                        //     diagonal (tau = r_c t), after the edge's matrix / tip tables
  int32_t prefetch;     // OePrefetchOps(C)
};

__global__ void TransitionMatrixOeKernel(const OeMatrixParams p) {
  const int n = p.taxon_count, C = p.categories;
  const int edge_count = 2 * n - 2, node_count = 2 * n - 1;
  const int ops_used = p.with_pre ? 2 * (n - 1) : n - 1;
  const int64_t idx = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int64_t matrix_jobs = static_cast<int64_t>(p.vtree_count) * edge_count * C;
  if (idx >= matrix_jobs) {
    const int64_t h = idx - matrix_jobs;
    if (h >= static_cast<int64_t>(p.vtree_count) * ops_used) return;
    const int v = p.vtree_begin + static_cast<int>(h / ops_used);
    const int o = static_cast<int>(h % ops_used);
    const OeOp* program = p.ops + static_cast<size_t>(p.vtree_program[v]) * 2 * (n - 1);
    const int4* own = reinterpret_cast<const int4*>(program + o);
    const int4* ahead = reinterpret_cast<const int4*>(program + (o + p.prefetch) % ops_used);
    int4* header = reinterpret_cast<int4*>(p.operands + static_cast<int64_t>(v - p.vtree_begin) * p.operand_stride +
                                            static_cast<int64_t>(program[o].operand_unit) * 2);
    header[0] = own[0];
    header[1] = own[1];
    int4 request = ahead[0];
    // how many tiles further on the op kOePrefetchOps ahead is (bits 16.. of the size word)
    request.y |= ((o + p.prefetch) / ops_used) << 16;
    header[2] = request;
    header[3] = ahead[1];
    if ((static_cast<unsigned>(program[o].node_flags) >> 24) & kRoot && o >= n - 1) {
      // The root has no edge: its pre-order op multiplies by an identity "P", so that
      // the kernel needs no root case (pp = I^T pi).
      double* identity = reinterpret_cast<double*>(header) + kOeHeaderDoubles;
      for (int c = 0; c < C; c++)
        for (int k = 0; k < kPStride; k++) identity[c * kPStride + k] = (k < 16 && k % 5 == 0) ? 1.0 : 0.0;
      if (p.with_subst)  // (no edge: no d P / d theta term)
        for (int k = 0; k < kOePhiDoubles * C; k++) identity[kPStride * C + k] = 0.0;
    }
    return;
  }
  const int c = static_cast<int>(idx % C);
  const int e = static_cast<int>((idx / C) % edge_count);
  const int v = p.vtree_begin + static_cast<int>(idx / (static_cast<int64_t>(C) * edge_count));
  const ModelTables& model = p.models[p.vtree_model[v]];
  const double t = p.branch_lengths[static_cast<int64_t>(p.vtree_lengths[v]) * node_count + e] * model.rates[c];
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
  const int2 offsets = p.edge_offsets[static_cast<size_t>(p.vtree_program[v]) * edge_count + e];
  double* const block = p.operands + static_cast<int64_t>(v - p.vtree_begin) * p.operand_stride;
  const bool tip = e < n;
  auto write_matrix = [&](double* part) {  // P_c row-major, blocks 18 doubles apart
    double2* out = reinterpret_cast<double2*>(part + kPStride * c);
#pragma unroll
    for (int x = 0; x < 8; x++) out[x] = make_double2(P[2 * x], P[2 * x + 1]);
  };
  auto write_tip_table = [&](double* part) {  // P^T (row s = column s of P) + a row of ones (the gap state)
    double2* out = reinterpret_cast<double2*>(part + kTipTableDoubles * c);
#pragma unroll
    for (int s = 0; s < 4; s++) {
      out[2 * s] = make_double2(P[s], P[4 + s]);
      out[2 * s + 1] = make_double2(P[8 + s], P[12 + s]);
    }
    out[8] = make_double2(1.0, 1.0);
    out[9] = make_double2(1.0, 1.0);
  };
  if (tip) {
    write_tip_table(block + offsets.x);
  } else {
    write_matrix(block + offsets.x);
  }
  if (!p.with_pre || offsets.y < 0) return;
  if (p.with_subst) {
    double2* out = reinterpret_cast<double2*>(block + offsets.y + (tip ? 2 * kTipTableDoubles : kPStride) * C +
                                              kOePhiDoubles * c);
#pragma unroll
    for (int k = 0; k < 4; k++) {
      double row[4];
#pragma unroll
      for (int l = 0; l < 4; l++) {
        // int_0^tau e^{l_k s} e^{l_l (tau - s)} ds, x = (l_k - l_l) tau, from the larger
        // exponent: e^{l_k tau} tau (1 - e^-x) / x if x > 0, else e^{l_l tau} tau (e^x - 1) / x.
        // (e^x - 1 overflows for x > 709 and e^{l_l tau} underflows on long branches.)
        const double x = (model.eval[k] - model.eval[l]) * t;
        if (x > 0.0) {
          const double ratio = x < 1e-8 ? 1.0 - 0.5 * x : -expm1(-x) / x;
          row[l] = ex[k] * t * ratio;
        } else {
          const double ratio = x > -1e-8 ? 1.0 + 0.5 * x : expm1(x) / x;
          row[l] = ex[l] * t * ratio;
        }
      }
      out[2 * k] = make_double2(row[0], row[1]);
      out[2 * k + 1] = make_double2(row[2], row[3]);
    }
  }
  if (!tip) {
    write_matrix(block + offsets.y);
    return;
  }
  write_tip_table(block + offsets.y);
  // (Q P)^T: row s = column s of Q P, + a row of zeros (Q 1 = 0)
  double2* out = reinterpret_cast<double2*>(block + offsets.y + kTipTableDoubles * C + kTipTableDoubles * c);
#pragma unroll
  for (int s = 0; s < 4; s++) {
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

constexpr int kOeSubstSums = 20;  // W (16) and R (4) of the analytic substitution gradient
// +I: D = sum of w (I - L) / lik and E_s = sum over the patterns whose tips all allow s of w / lik
constexpr int kOeInvariantSums = 5;

// One launch for all result arrays: out = [logl (logl_count) | grad (rows x width) |
// rgrad (rows x width) | substitution sums (rows x kOeSubstSums) | +I sums (rows x
// kOeInvariantSums)], each entry the fixed-order sum of its `parts` per-(chunk, warp)
// partial rows (bitwise deterministic run to run).
__global__ void ReduceAllKernel(const double* __restrict__ logl_partial, const double* __restrict__ grad_partial,
                                const double* __restrict__ rgrad_partial, const double* __restrict__ subst_partial,
                                double* __restrict__ out, int32_t logl_begin, int32_t logl_count,
                                int32_t logl_total, int32_t grad_rows, int32_t width, int32_t parts,
                                const double* __restrict__ inv_partial = nullptr) {
  int64_t idx = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int64_t grad_count = static_cast<int64_t>(grad_rows) * width;
  const int64_t subst_count = static_cast<int64_t>(grad_rows) * kOeSubstSums;
  if (inv_partial != nullptr && idx >= logl_count + 2 * grad_count + subst_count) {
    // the +I sums: [tree][kOeInvariantSums] after the substitution sums
    idx -= logl_count + 2 * grad_count + subst_count;
    if (idx >= static_cast<int64_t>(grad_rows) * kOeInvariantSums) return;
    const int64_t row = idx / kOeInvariantSums;
    const int e = static_cast<int>(idx % kOeInvariantSums);
    const double* src = inv_partial + row * parts * kOeInvariantSums + e;
    double sum = 0.0;
    for (int part = 0; part < parts; part++) sum += src[static_cast<int64_t>(part) * kOeInvariantSums];
    out[logl_total + 2 * grad_count + subst_count + idx] = sum;
    return;
  }
  if (subst_partial != nullptr && idx >= logl_count + 2 * grad_count) {
    // the substitution-gradient sums: [tree][kOeSubstSums] after the three arrays
    idx -= logl_count + 2 * grad_count;
    if (idx >= subst_count) return;
    const int64_t row = idx / kOeSubstSums;
    const int e = static_cast<int>(idx % kOeSubstSums);
    const double* src = subst_partial + row * parts * kOeSubstSums + e;
    double sum = 0.0;
    for (int part = 0; part < parts; part++) sum += src[static_cast<int64_t>(part) * kOeSubstSums];
    out[logl_total + 2 * grad_count + idx] = sum;
    return;
  }
  if (idx < logl_count) {
    const int64_t v = logl_begin + idx;
    const double* src = logl_partial + v * parts;
    double sum = 0.0;
    for (int part = 0; part < parts; part++) sum += src[part];
    out[v] = sum;
    return;
  }
  int64_t k = idx - logl_count;
  if (k >= 2 * grad_count) return;  // (a substitution-sum index of a run without them)
  const double* partial = grad_partial;
  double* dst = out + logl_total;
  if (k >= grad_count) {
    if (rgrad_partial == nullptr) return;
    k -= grad_count;
    partial = rgrad_partial;
    dst += grad_count;
  }
  const int64_t row = k / width;
  const int e = static_cast<int>(k % width);
  const double* src = partial + row * parts * width + e;
  double sum = 0.0;
  for (int part = 0; part < parts; part++) sum += src[static_cast<int64_t>(part) * width];
  dst[k] = sum;
}

// Rooted time trees: the O(n) tail of FatBeagle::Gradient(RootedTree) (fat_beagle.cpp:505-545)
// behind the reduction, one thread per tree -- RatioGradientOfBranchGradient
// (rooted_gradient_transforms.cpp:17-170: height gradient, chain rule to the height ratios
// through the epoch structure, root height, gradient of the log-det-Jacobian), ClockGradient
// and DiscreteSiteModelGradient (fat_beagle.cpp:367-398) -- so a rooted gradient leaves the
// device finished.  Internal node ids ascend in post-order, so an ascending loop is a
// post-order pass and a descending loop a pre-order pass (the same arithmetic as
// csrc/rooted.cpp, which finishes sharded runs on the host).
struct RootedFinishParams {
  int32_t tree_count, taxon_count, rate_count;
  const int32_t* children;   // [tree][2][2n-1]: child0 then child1 per node id (-1 for leaves)
  const double* fields;      // [tree]: rates (2n-2), branch lengths (2n-1), heights (2n-1), bounds (2n-1), ratios (n-1)
  const double* scaled_lengths;  // [tree][2n-1] branch length x rate, what the walk used
  const double* grad;        // [tree][2n-1] edge derivatives
  const double* rgrad;       // [tree][2n-1] or NULL (one category)
  double* scratch;           // [tree][5][n-1]
  double* out;               // [tree][(n-1) + rate_count + site_width]: ratios / root height, clock, site model
  // +I: the reduced [tree][kOeInvariantSums] sums and each tree's pinv, else NULL; the site-model
  // row is then [shape (if any) | proportion invariant]
  const double* inv_sums;
  const ModelTables* models;
  const int32_t* vtree_model;
  int32_t site_width;
};

__global__ void RootedFinishKernel(const RootedFinishParams p) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= p.tree_count) return;
  const int n = p.taxon_count, N = 2 * n - 1, root = N - 1;
  const int32_t* child0 = p.children + static_cast<size_t>(t) * 2 * N;
  const int32_t* child1 = child0 + N;
  const double* rates = p.fields + static_cast<size_t>(t) * (4 * N + n - 2);
  const double* lengths = rates + (N - 1);
  const double* heights = lengths + N;
  const double* bounds = heights + N;
  const double* ratios = bounds + N;
  const double* g = p.grad + static_cast<size_t>(t) * N;
  double* height_gradient = p.scratch + static_cast<size_t>(t) * 5 * (n - 1);
  double* chain = height_gradient + (n - 1);
  double* log_time = chain + (n - 1);
  double* jacobian = log_time + (n - 1);
  double* multiplier = jacobian + (n - 1);
  const int site_width = p.inv_sums != nullptr ? p.site_width : 1;
  double* out = p.out + static_cast<size_t>(t) * (n - 1 + p.rate_count + site_width);

  auto node_partial = [&](int node) { return (heights[node] - bounds[node]) / ratios[node - n]; };
  auto epoch_addition = [&](int node, int child, const double* ratio_gradient) {
    if (child < n) return 0.0;
    if (bounds[node] == bounds[child]) return ratio_gradient[child - n] * ratios[child - n] / ratios[node - n];
    return ratio_gradient[child - n] * ratios[child - n] / (heights[node] - bounds[child]) * node_partial(node);
  };
  auto ratio_chain = [&](const double* height_terms, double* result) {
    for (int node = n; node < N; node++) {
      if (node == root) {
        result[node - n] = 0.0;
        continue;
      }
      double value = node_partial(node) * height_terms[node - n];
      result[node - n] = value;  // (the children's entries are complete: ids ascend in post-order)
      value += epoch_addition(node, child0[node], result);
      result[node - n] = value;
      value += epoch_addition(node, child1[node], result);
      result[node - n] = value;
    }
  };
  auto root_height_chain = [&](const double* terms) {
    for (int i = 0; i < n - 1; i++) multiplier[i] = 0.0;
    multiplier[root - n] = 1.0;
    for (int node = N - 1; node >= n; node--) {
      const int c0 = child0[node], c1 = child1[node];
      if (c0 >= n) multiplier[c0 - n] = ratios[c0 - n] * multiplier[node - n];
      if (c1 >= n) multiplier[c1 - n] = ratios[c1 - n] * multiplier[node - n];
    }
    double sum = 0.0;
    for (int i = 0; i < n - 1; i++) sum += terms[i] * multiplier[i];
    return sum;
  };

  for (int node = n; node < N; node++) {
    double value = 0.0;
    if (node != root) value = -g[node] * rates[node];
    value += g[child0[node]] * rates[child0[node]];
    value += g[child1[node]] * rates[child1[node]];
    height_gradient[node - n] = value;
  }
  ratio_chain(height_gradient, chain);
  chain[root - n] = root_height_chain(height_gradient);
  for (int i = 0; i < n - 1; i++) log_time[i] = (i < n - 2) ? 1.0 / (heights[n + i] - bounds[n + i]) : 0.0;
  ratio_chain(log_time, jacobian);
  jacobian[root - n] = root_height_chain(log_time);
  for (int i = 0; i < n - 2; i++) out[i] = chain[i] + (jacobian[i] - 1.0 / ratios[i]);
  out[root - n] = chain[root - n] + jacobian[root - n];

  double* clock = out + (n - 1);
  if (p.rate_count == 1) {
    double sum = 0.0;
    for (int i = 0; i < N - 1; i++) sum += g[i] * lengths[i];
    clock[0] = sum;
  } else {
    for (int i = 0; i < N - 1; i++) clock[i] = g[i] * lengths[i];
  }
  double site = 0.0;
  if (p.rgrad != nullptr) {
    const double* rg = p.rgrad + static_cast<size_t>(t) * N;
    const double* scaled = p.scaled_lengths + static_cast<size_t>(t) * N;
    for (int node = 0; node < N - 1; node++) site += rg[node] * scaled[node];
  }
  out[n - 1 + p.rate_count] = site;
  if (p.inv_sums != nullptr) {
    // d logL / d pinv = D + sum over edges of tau g / (1 - pinv): the rates are divided by 1 - pinv
    const double* scaled = p.scaled_lengths + static_cast<size_t>(t) * N;
    double normalisation = 0.0;
    for (int node = 0; node < N - 1; node++) normalisation += g[node] * scaled[node];
    const double pinv = p.models[p.vtree_model[t]].pinv;
    out[n - 1 + p.rate_count + site_width - 1] =
        p.inv_sums[static_cast<size_t>(t) * kOeInvariantSums] + normalisation / (1.0 - pinv);
  }
}

// Device groups sharded by site pattern (engine.cu): the raw per-tree sums of the other
// devices, read through peer pointers over NVLink, are added onto this device's array.
struct PeerPointers {
  const double* part[16];
};

// out[i] += part[1][i] + part[2][i] + ... in a fixed order (part[0] is out itself).
__global__ void PeerSumKernel(double* __restrict__ out, PeerPointers peers, int32_t count_of_peers, int64_t count) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= count) return;
  double sum = out[i];
  for (int g = 1; g < count_of_peers; g++) sum += peers.part[g][i];
  out[i] = sum;
}


#ifndef SBNB_OE_STAGES
#define SBNB_OE_STAGES 8
#endif
#ifndef SBNB_OE_PREFETCH
#define SBNB_OE_PREFETCH (SBNB_OE_STAGES / 2)
#endif
// At 32 categories one op's operands take ~25 KB (37 KB with the analytic substitution
// gradient), so the ring is shallow and requests run one op ahead.  An op's request waits
// until every warp has left the op kStages - kPrefetch places before it: with a margin of one
// op (2 stages) the first warp waits for the last at every op, which costs the gradient walk
// 3.6x (measured); the logL-only walk, with no pre-order half, loses less to that than it
// would to going from three resident CTAs per SM to two.
#ifndef SBNB_OE_STAGES_32
#define SBNB_OE_STAGES_32 3  // gradient walks at 32 categories
#endif
__host__ __device__ constexpr int OeStages(int C, bool grad) {  // operand ring depth
  return C >= 32 ? (grad ? SBNB_OE_STAGES_32 : 2) : C >= 8 ? 4 : SBNB_OE_STAGES;
}
__host__ __device__ constexpr int OePrefetchOps(int C) { return C >= 32 ? 1 : C >= 8 ? 2 : SBNB_OE_PREFETCH; }
__host__ __device__ constexpr int OeGroup(int C) { return kThreads / C; }  // patterns per j-slab
__host__ __device__ constexpr int OeTilePatterns(int C, int K) { return OeGroup(C) * K; }
__host__ __device__ constexpr int OeTipBytes(int C, int K) { return (OeTilePatterns(C, K) + 15) / 16 * 16; }
__host__ __device__ constexpr int OeStageBytes(int C, int K, bool subst = false) {
  return OeMaxOperandDoubles(C, subst) * 8 + 2 * OeTipBytes(C, K);
}
// The pre-order op works through its K patterns in sub-batches of at most 2.
__host__ __device__ constexpr int OePreBatch(int K) { return K > 2 ? 2 : K; }
// Read-back slots of one pre-order op: [warp][batch][child][j][half][lane] double2.
__host__ __device__ constexpr int OeReadbackBytes(int K) { return 2 * K * 2 * kThreads * 16; }
// Tip codes.  An alignment given as nucleotide masks (bit 0 = A .. bit 3 = T) is held as
// codes 0..3 (one state), 4 (all four: missing, also the padding) and 5..14 (the ten two-
// and three-state masks, in ascending order of the mask).  Nibble c of kTipCodeMasks is
// the mask of code c.  Codes 0..4 index the rows of a tip table directly; a walk
// instantiated for ambiguous tips sums the state rows of codes 5..14.
constexpr int kFirstAmbiguousCode = 5;
constexpr int kTipCodes = 15;
constexpr uint64_t kTipCodeMasks = 0xEDCBA97653F8421ull;
__host__ __device__ constexpr unsigned TipCodeMask(int code) {
  return static_cast<unsigned>(kTipCodeMasks >> (4 * code)) & 15u;
}
// +I: per site pattern the set of states every tip allows (the AND of the tips' masks; a gap
// allows all four), one byte per pattern beside the weights.  One thread per pattern of the
// padded range, reading the [taxon][pattern] codes coalesced; the padding gets the empty set.
__global__ void InvariantMaskKernel(const uint8_t* __restrict__ tips, int64_t tip_pitch, int32_t taxon_count,
                                    int64_t pattern_count, uint8_t* __restrict__ masks) {
  const int64_t k = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k >= tip_pitch) return;
  unsigned mask = 15u;
  for (int taxon = 0; taxon < taxon_count && mask != 0u; taxon++)
    mask &= TipCodeMask(tips[static_cast<int64_t>(taxon) * tip_pitch + k]);
  masks[k] = static_cast<uint8_t>(k < pattern_count ? mask : 0u);
}
// model constants of the analytic substitution gradient: V, V^-1, and V^-1 L per tip code
// (codes 0..4; all 15 codes in a walk over ambiguous tips)
__host__ __device__ constexpr int OeTipZDoubles(bool ambig) { return 4 * (ambig ? kTipCodes : kFirstAmbiguousCode); }
__host__ __device__ constexpr int OeSubstSmemDoubles(bool ambig) { return 16 + 16 + OeTipZDoubles(ambig); }
__host__ __device__ constexpr size_t OeSmemBytes(int C, int K, bool grad, bool subst = false, bool ambig = false) {
  return static_cast<size_t>(OeStages(C, grad)) * OeStageBytes(C, K, subst) + 2 * OeStages(C, grad) * 8 +
         (ModelSmemDoubles(C) + OeSubstSmemDoubles(ambig)) * 8 + 16 + 2 * kWarps * 8 +
         (grad ? OeReadbackBytes(K) : 0);
}
// Resident CTAs per SM the register allocation is held to.
__host__ __device__ constexpr int OeMinBlocks(int K, bool grad, bool subst = false) {
  if (subst) return 2;  // 16 + 4 more accumulators per thread
  return grad ? 3 : (K <= 2 ? 4 : 3);
}

// y[j] = M x[j], M row-major in shared memory (per-lane address: the lane's category)
template <int K>
__device__ __forceinline__ void MatVecOe(const double* m, const double (&x)[K][4], double (&y)[K][4]) {
#pragma unroll
  for (int i = 0; i < 4; i++) {
    double row[4];
    Load4(m + 4 * i, row);
#pragma unroll
    for (int j = 0; j < K; j++)
      y[j][i] = fma(row[3], x[j][3], fma(row[2], x[j][2], fma(row[1], x[j][1], row[0] * x[j][0])));
  }
}
// out[j] = t[j] . (M x[j])
template <int K>
__device__ __forceinline__ void MatVecDotOe(const double* m, const double (&x)[K][4], const double (&t)[K][4],
                                            double (&out)[K]) {
#pragma unroll
  for (int i = 0; i < 4; i++) {
    double row[4];
    Load4(m + 4 * i, row);
#pragma unroll
    for (int j = 0; j < K; j++) {
      const double d = fma(row[3], x[j][3], fma(row[2], x[j][2], fma(row[1], x[j][1], row[0] * x[j][0])));
      out[j] = (i == 0) ? t[j][0] * d : fma(t[j][i], d, out[j]);
    }
  }
}

// 1 / x for a normal, positive x: hardware seed + two Newton steps (relative error
// ~1e-16; x is a per-pattern likelihood kept in range by the rescaling).
__device__ __forceinline__ double FastReciprocalOe(double x) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  double e = fma(-x, r, 1.0);
  r = fma(r, e, r);
  e = fma(-x, r, 1.0);
  return fma(r, e, r);
}

// Per-pattern power-of-two normalisation when the C lanes of a pattern hold one
// category each: a pattern is rescaled when its largest entry over all categories has
// dropped below 2^-BAR.  Finding that maximum takes shuffles, so the warp first votes
// on a cheaper, per-lane test with a lower bar (2^-(BAR + kOeLaneSlackBits)): a lane
// whose own category lags the pattern's maximum by less than 2^64 does not send the
// warp down the slow path at every op.  Until some lane trips the vote a pattern may
// sit between the two bars unrescaled -- far from underflow.
//   Post-order partials are rescaled with BAR = kOeLazyBits = 32.  The pre-order partial
// pp at a node satisfies sum_c pp_c . L_c = the pattern's (scaled) root likelihood over
// the factors the node's ancestors' own rescalings applied: with every scaled L inside
// [2^-32, 1] it moves only when an ancestor was rescaled, so the pre-order pass tests the
// already reduced pp . L against 2^-kOePreBits -- one vote per sub-batch and a slow path
// that practically only deep trees take (with the 2^-128 bar of the previous kernels pp
// lost ~2^-100 per level and 96 % of the pre-order ops went down a shuffle-based slow path).
constexpr int kOeLazyBits = 32;
constexpr int kOePreBits = 384;
constexpr int kOeLaneSlackBits = 64;
template <int C, int K, int BAR>
__device__ __forceinline__ void NormalizeOe(double (&v)[K][4], int (&exps)[K]) {
  int hi[K];
  bool low = false;
#pragma unroll
  for (int j = 0; j < K; j++) {
    hi[j] = max(max(__double2hiint(v[j][0]), __double2hiint(v[j][1])),
                max(__double2hiint(v[j][2]), __double2hiint(v[j][3])));
    low = low || (hi[j] < ((1023 - BAR - kOeLaneSlackBits) << 20));
  }
  if (!__any_sync(0xffffffffu, low)) return;
#pragma unroll
  for (int j = 0; j < K; j++) {
    int m = hi[j];
#pragma unroll
    for (int s = 32 / C; s < 32; s <<= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, s));
    const int biased = (m >> 20) & 0x7ff;
    // zero / subnormal / inf / nan, or still large enough: leave as is
    if (biased == 0 || biased >= 1023 - BAR) continue;
    const double scale = __hiloint2double((2046 - biased) << 20, 0);
#pragma unroll
    for (int i = 0; i < 4; i++) v[j][i] *= scale;
    exps[j] += biased - 1023;
  }
}

// y = the tip-table row(s) of the tip code of pattern j in `packed`: one row for codes 0..4,
// the sum of the state rows of an ambiguous code (a tip's contribution M L_tip is linear in
// L_tip, the indicator vector of its states).  Every lane loads the row of its code or of
// the lowest state of its mask; lanes of ambiguous codes then add one or two more rows.
__device__ __forceinline__ void LoadAmbiguousTipRow(const double* table, uint32_t packed, int j, double (&y)[4]) {
  const int code = (packed >> (8 * j)) & 0xff;
  const unsigned mask = code >= kFirstAmbiguousCode ? TipCodeMask(code) : 0u;
  Load4(table + 4 * (mask != 0u ? __ffs(mask) - 1 : code), y);
  for (unsigned rest = mask & (mask - 1); rest != 0u; rest &= rest - 1) {
    double row[4];
    Load4(table + 4 * (__ffs(rest) - 1), row);
#pragma unroll
    for (int i = 0; i < 4; i++) y[i] += row[i];
  }
}

// A proportion pinv of invariable sites (+I): lik = (1 - pinv) L + pinv I, with L = site 2^exp
// the mixture over the rate categories and I the summed frequencies of the states every tip
// of the pattern allows.  Everything is a function of rho = I / L formed in the scaled
// domain, so that neither 0 x inf nor inf / inf arises when L is far below the fp64 range:
//   x = pinv rho / (1 - pinv),  f = (1 - pinv) L / lik = 1 / (1 + x),
//   L / lik = f / (1 - pinv),   I / lik = rho f / (1 - pinv) = 1 / (pinv (1 + 1 / x)).
// At pinv = 0 the log-likelihood and f are bitwise those of the model without +I.
struct InvariantSiteTerms {
  double log_lik, f, inv_over_lik, var_over_lik;
};
__device__ __forceinline__ InvariantSiteTerms InvariantSite(double log_l, double site, int exp, double pinv,
                                                            double invariant) {
  const double rho = invariant == 0.0 ? 0.0 : ldexp(invariant / site, -exp);
  const double x = pinv == 0.0 ? 0.0 : pinv * rho / (1.0 - pinv);
  InvariantSiteTerms t;
  t.f = 1.0 / (1.0 + x);
  t.var_over_lik = t.f / (1.0 - pinv);
  if (x <= 1.0) {
    t.log_lik = log_l + log1p(-pinv) + log1p(x);
    t.inv_over_lik = rho * t.var_over_lik;
  } else {  // (rho may be inf: the variable part is then below the fp64 range)
    t.log_lik = log(pinv * invariant) + log1p(1.0 / x);
    t.inv_over_lik = 1.0 / (pinv * (1.0 + 1.0 / x));
  }
  return t;
}

// SITES (logL-only walks): the root op also stores every pattern's log site likelihood -- the
// term it adds into logL with the pattern's weight -- into p.site_logl.
template <int C, int K, bool GRAD, bool RESCALE, bool SUBST = false, bool AMBIG = false, bool INVAR = false,
          bool SITES = false>
__global__ void __launch_bounds__(kThreads, OeMinBlocks(K, GRAD, SUBST)) TreeWalkOeKernel(const OeParams p) {
  static_assert(GRAD || !SUBST, "the substitution gradient rides on the pre-order pass");
  static_assert(!(GRAD && SITES), "site log-likelihoods come from log-likelihood runs");
  static_assert((C & (C - 1)) == 0 && C >= 1 && C <= 32, "lanes per pattern must be a power of two");
  static_assert(OeTilePatterns(C, K) % 16 == 0, "tiles must start on 16-byte boundaries of the tip rows");
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int tid = threadIdx.x;
  const int warp = tid >> 5;
  const int lane = tid & 31;
  // Category-major lanes: the 32 / C lanes of one category are adjacent, so the lanes
  // a shared-memory load serves together read the SAME category's tables.
  constexpr int kPerWarp = 32 / C;  // patterns of one j-slab held by a warp
  const int cat = lane / kPerWarp;
  const int pidx = warp * kPerWarp + lane % kPerWarp;
  const int n = p.taxon_count;
  const int internal_count = n - 1;
  const int node_count = 2 * n - 1;
  const int ops_total = GRAD ? 2 * internal_count : internal_count;
  constexpr int kStages = OeStages(C, GRAD);
  constexpr int kPrefetch = OePrefetchOps(C);
  constexpr int kTilePatterns = OeTilePatterns(C, K);
  constexpr int kTipBytes = OeTipBytes(C, K);
  constexpr int kStage = OeStageBytes(C, K, SUBST);
  constexpr int kOperandBytes = OeMaxOperandDoubles(C, SUBST) * 8;
  constexpr int kPhiPart = SUBST ? kOePhiDoubles * C : 0;  // doubles of Phi behind an edge's part
  constexpr int kRow = 2 * kThreads;  // double2 per pattern slab: [half][tid]
  constexpr int KP = OePreBatch(K);   // patterns per pre-order sub-batch ...
  constexpr int kBatches = K / KP;    // ... and sub-batches per op, each with its own barrier
  static_assert(K % KP == 0 && kBatches <= 2, "pre-order sub-batches must tile K");
  constexpr int kLeafPart = kTipTableDoubles * C;  // doubles of one tip table set
  constexpr int kInnerPart = kPStride * C;         // doubles of one P block

  // ---- shared memory carve-up ------------------------------------------------
  unsigned char* const ring = smem_raw;
  uint64_t* const full = reinterpret_cast<uint64_t*>(smem_raw + kStages * kStage);
  uint64_t* const empty = full + kStages;
  double* const q_smem = reinterpret_cast<double*>(empty + kStages);
  double* const cat_weight_smem = q_smem + 16;
  double* const rate_weight_smem = cat_weight_smem + ModelSmemCategories(C);
  double* const drate_weight_smem = rate_weight_smem + ModelSmemCategories(C);
  double* const freqs_smem = drate_weight_smem + ModelSmemCategories(C);
  double* const evec_smem = freqs_smem + 4;  // V, V^-1 and V^-1 L per tip code: analytic substitution gradient
  double* const ivec_smem = evec_smem + 16;
  double* const tip_z_smem = ivec_smem + 16;
  constexpr int kTipZ = OeTipZDoubles(AMBIG);
  // Sequence number of the next op whose operands have not been requested yet.
  uint32_t* const ticket = reinterpret_cast<uint32_t*>(tip_z_smem + kTipZ);
  uint64_t* const readback_bars = reinterpret_cast<uint64_t*>(tip_z_smem + kTipZ + 2);
  uint64_t* const readback_full = readback_bars + warp * 2;
  // Read-back slots, [warp][batch][child][j][half][lane] double2, filled per warp by
  // bulk copies that complete on the warp's own barriers.
  double2* const readback_base = reinterpret_cast<double2*>(readback_bars + 2 * kWarps);
  constexpr int kBatchSlot = 2 * KP * 64;  // double2 of one (warp, batch) slot
  double2* const my_readback = readback_base + warp * kBatches * kBatchSlot;
  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < kStages; s++) {
      MbarInit(full + s, 1);
      MbarInit(empty + s, kWarps);
    }
    for (int w = 0; w < 2 * kWarps; w++) MbarInit(readback_bars + w, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  // Per-CTA scratch: coalesced 16 B per lane.  Stack rows are [slot][j][half][tid].
  double2* const my_stack = p.stack + static_cast<size_t>(blockIdx.x) * p.slots * K * kRow + tid;
  int32_t* const my_stack_exps =
      RESCALE ? p.stack_exps + static_cast<size_t>(blockIdx.x) * p.slots * K * kThreads + tid : nullptr;
  // Arena: blocks of K * kRow double2, one per internal child, grouped by the op that
  // writes and reads them: [op][warp][batch][child][j][half][lane].
  double2* const my_arena =
      GRAD ? p.arena + static_cast<size_t>(blockIdx.x) * max(n - 2, 1) * K * kRow : nullptr;
  uint32_t readback_sequence = 0;  // pre-order ops this warp has consumed
  uint32_t sequence = 0;           // ops this CTA has consumed; stage = sequence % kStages

  const int64_t total_items = static_cast<int64_t>(p.vtree_count) * p.chunks;
  for (int64_t item = blockIdx.x; item < total_items; item += gridDim.x) {
    const int vt = p.vtree_begin + static_cast<int>(item / p.chunks);
    const int chunk = static_cast<int>(item % p.chunks);
    const ModelTables& model = p.models[p.vtree_model[vt]];
    const double* const block = p.operands + static_cast<int64_t>(vt - p.operand_origin) * p.operand_stride;
    const size_t out_row = (static_cast<size_t>(vt) * p.chunks + chunk) * kWarps + warp;
    double* const grad_row = GRAD ? p.grad_partial + out_row * node_count : nullptr;
    double* const rgrad_row = (GRAD && C > 1) ? p.rgrad_partial + out_row * node_count : nullptr;
    __syncthreads();  // every warp is done with the previous item's model constants
    if (tid < 16) {
      q_smem[tid] = model.q[tid];
      cat_weight_smem[tid] = model.weights[tid];
      rate_weight_smem[tid] = model.rates[tid];    // r_c  (p_c rides in the pre-order partials)
      drate_weight_smem[tid] = model.drates[tid];  // dr_c/dshape
      if (tid < 4) freqs_smem[tid] = model.freqs[tid];
      if (SUBST) {
        evec_smem[tid] = model.evec[tid];
        ivec_smem[tid] = model.ivec[tid];
      }
    }
    if (C > 16 && tid >= 16 && tid < C) {
      cat_weight_smem[tid] = model.weights[tid];
      rate_weight_smem[tid] = model.rates[tid];
      drate_weight_smem[tid] = model.drates[tid];
    }
    if (SUBST && tid >= 32 && tid < 32 + kTipZ) {
      // V^-1 L for a tip: column s of V^-1 for a resolved state, the row sums for a gap,
      // the sum of its states' columns for an ambiguous code
      const int state = (tid - 32) / 4, k = (tid - 32) % 4;
      if constexpr (AMBIG) {
        if (state >= kFirstAmbiguousCode) {
          double sum = 0.0;
          for (int s = 0; s < 4; s++)
            if (TipCodeMask(state) >> s & 1u) sum += model.ivec[k * 4 + s];
          tip_z_smem[tid - 32] = sum;
        }
      }
      if (!AMBIG || state < kFirstAmbiguousCode)
        tip_z_smem[tid - 32] = state < 4 ? model.ivec[k * 4 + state]
                                         : model.ivec[k * 4] + model.ivec[k * 4 + 1] + model.ivec[k * 4 + 2] +
                                               model.ivec[k * 4 + 3];
    }
    if (GRAD) {
      // This warp owns its rows of edge-derivative sums for the whole item: clear them
      // (the ops accumulate with reductions; no separate memset launch).
      for (int e = lane; e < node_count; e += 32) {
        grad_row[e] = 0.0;
        if (C > 1) rgrad_row[e] = 0.0;
      }
      if (INVAR && lane < kOeInvariantSums) p.inv_partial[out_row * kOeInvariantSums + lane] = 0.0;
    }
    const int tile_begin = chunk * p.tiles_per_chunk;
    const int tile_end = min(tile_begin + p.tiles_per_chunk, p.tiles_total);
    // The item's ops form one stream g = 0 .. item_ops - 1 (tile-major).
    const int item_ops = max(tile_end - tile_begin, 0) * ops_total;

    // Bulk copies of one op's operands into its ring stage (one thread).
    auto issue = [&](uint32_t seq, const int4 record, int64_t tile_pat0) {
      const int s = seq % kStages;
      if (seq >= kStages) MbarWait(empty + s, ((seq / kStages) - 1) & 1);
      unsigned char* stage = ring + s * kStage;
      const uint32_t operand_bytes = static_cast<uint32_t>(record.y & 0xffff) * 16;
      const uint32_t bytes = operand_bytes + (record.z >= 0 ? kTipBytes : 0) + (record.w >= 0 ? kTipBytes : 0);
      MbarExpectTx(full + s, bytes);
      BulkCopy(stage, block + static_cast<int64_t>(record.x) * 2, operand_bytes, full + s);
      if (record.z >= 0)
        BulkCopy(stage + kOperandBytes, p.tips + static_cast<int64_t>(record.z) * p.tip_pitch + tile_pat0,
                 kTipBytes, full + s);
      if (record.w >= 0)
        BulkCopy(stage + kOperandBytes + kTipBytes,
                 p.tips + static_cast<int64_t>(record.w) * p.tip_pitch + tile_pat0, kTipBytes, full + s);
    };

    // Lane 0 of every warp: start the bulk copy of one sub-batch of a pre-order op's
    // internal children's evolved partials (the warp's own arena blocks).
    auto fetch_readback = [&](int arena_slot, int children, int batch) {
      if (children == 0) {
        MbarArrive(readback_full + batch);
        return;
      }
      const uint32_t bytes = static_cast<uint32_t>(children) * (KP * 64 * 16);
      MbarExpectTx(readback_full + batch, bytes);
      BulkCopy(my_readback + batch * kBatchSlot,
               my_arena + static_cast<size_t>(arena_slot) * K * kRow +
                   static_cast<size_t>(warp * kBatches + batch) * children * (KP * 64),
               bytes, readback_full + batch);
    };

    // Operands are requested kPrefetch ops ahead of the FIRST warp to get to an op.
    if (tid == 0) {
      const int first = min(kPrefetch, item_ops);
      const OeOp* program = p.ops + static_cast<size_t>(p.vtree_program[vt]) * 2 * internal_count;
      for (int g = 0; g < first; g++) {
        const int o = g % ops_total;
        issue(sequence + g, __ldg(reinterpret_cast<const int4*>(program + o)),
              p.pattern_begin + static_cast<int64_t>(tile_begin + g / ops_total) * kTilePatterns);
      }
      *ticket = sequence + first;
    }
    __syncthreads();
    const double cat_weight = cat_weight_smem[cat];
    const double rate_w = rate_weight_smem[cat];
    const double drate_w = drate_weight_smem[cat];
    int g = 0;

    double logl_acc = 0.0;
    // analytic substitution gradient: W_kl = sum of w/lik (V^T T)_k (V^-1 L)_l Phi_kl over edges and
    // patterns, R_l = sum of w/lik p_c L_root,l -- per thread over the whole item
    double wsub[SUBST ? 16 : 1], rsub[SUBST ? 4 : 1];
    if (SUBST) {
#pragma unroll
      for (int e = 0; e < 16; e++) wsub[e] = 0.0;
#pragma unroll
      for (int e = 0; e < 4; e++) rsub[e] = 0.0;
    }
    // wsub += sum_j scale_j (V^T t_j) (z_j)^T o Phi, Phi row-major at `phi` (this lane's category)
    auto accumulate_subst = [&](const double (&t)[OePreBatch(K)][4], const double (&z)[OePreBatch(K)][4],
                                const double (&scale)[OePreBatch(K)], const double* phi) {
      double u[OePreBatch(K)][4];
      MatTVecSharedK<OePreBatch(K)>(evec_smem, t, u);
#pragma unroll
      for (int k = 0; k < 4; k++) {
        double row[4];
        Load4(phi + 4 * k, row);
#pragma unroll
        for (int j = 0; j < OePreBatch(K); j++) {
          const double su = scale[j] * u[j][k];
#pragma unroll
          for (int l = 0; l < 4; l++) wsub[SUBST ? k * 4 + l : 0] = fma(su * z[j][l], row[l], wsub[SUBST ? k * 4 + l : 0]);
        }
      }
    };
    for (int tile = tile_begin; tile < tile_end; tile++) {
      const int64_t pat0 = p.pattern_begin + static_cast<int64_t>(tile) * kTilePatterns;
      double w[K];
#pragma unroll
      for (int j = 0; j < K; j++) {
        const int64_t pattern = pat0 + pidx * K + j;  // a thread's K patterns are adjacent
        w[j] = (pattern < p.pattern_end) ? p.weights[pattern] : 0.0;
      }

      double cur[K][4];
      int cur_exp[K];
#pragma unroll
      for (int j = 0; j < K; j++) {
        cur_exp[j] = 0;
#pragma unroll
        for (int i = 0; i < 4; i++) cur[j][i] = 0.0;
      }

      for (int o = 0; o < ops_total; o++, sequence++, g++) {
        const int stage_index = sequence % kStages;
        MbarWait(full + stage_index, (sequence / kStages) & 1);
        const unsigned char* stage = ring + stage_index * kStage;
        // The op's own record (all lanes read the same words; the flag word is
        // broadcast so that the branches below are warp-uniform for the compiler).
        const int4 record = *reinterpret_cast<const int4*>(stage + 16);
        const int flags = __shfl_sync(0xffffffffu, static_cast<unsigned>(record.x) >> 24, 0);
        if (lane == 0 && g + kPrefetch < item_ops) {
          const uint32_t target = sequence + kPrefetch;
          // (plain read first: only a warp that can win goes through the atomic)
          if (*reinterpret_cast<volatile uint32_t*>(ticket) == target &&
              atomicCAS(ticket, target, target + 1) == target)
          {
            // the record of op g + kPrefetch, and how many tiles further on it is
            const int4 request = *reinterpret_cast<const int4*>(stage + 32);
            issue(target, request, pat0 + static_cast<int64_t>(request.y >> 16) * kTilePatterns);
          }
        }
        __syncwarp();
        const double* const operand = reinterpret_cast<const double*>(stage) + kOeHeaderDoubles;
        // the tip states of this thread's K adjacent patterns: one load per tip child
        const unsigned char* const tips_at = stage + kOperandBytes + pidx * K;
        auto tip_states = [&](const unsigned char* at) -> uint32_t {
          if (K == 4) return *reinterpret_cast<const uint32_t*>(at);
          if (K == 2) return *reinterpret_cast<const uint16_t*>(at);
          return *at;
        };
        // doubles from the start of a category's tip table to the row of pattern j's state
        // (AMBIG: LoadAmbiguousTipRow sums the state rows of an ambiguous code)
        auto tip_row = [](uint32_t packed, int j) -> int { return ((packed >> (8 * j)) & 0xff) * 4; };
        // The host orders the children of every op so that an internal child whose
        // partial is (post-order) or stays (pre-order) in cur is child a, and a child
        // that goes through the stack is child b: a leaf => b leaf.
        const bool a_leaf = flags & kALeaf, b_leaf = flags & kBLeaf;
        const int children = (a_leaf ? 0 : 1) + (b_leaf ? 0 : 1);

        if (!GRAD || o < internal_count) {
          // ======================= post-order op ===========================
          // cur = (P_a L_a) o (P_b L_b), L_a = cur, L_b from the stack
          if (flags & kStackBefore) {
            const int s0 = record.y & 0xff;
#pragma unroll
            for (int j = 0; j < K; j++) {
              double2* dst = my_stack + (static_cast<size_t>(s0) * K + j) * kRow;
              dst[0] = make_double2(cur[j][0], cur[j][1]);
              dst[kThreads] = make_double2(cur[j][2], cur[j][3]);
              if (RESCALE) my_stack_exps[(s0 * K + j) * kThreads] = cur_exp[j];
            }
          }
          // arena rows of this op: [warp][batch][child][j][half][lane]
          double2* const region =
              GRAD ? my_arena + static_cast<size_t>(record.z) * K * kRow +
                         static_cast<size_t>(warp * kBatches) * children * (KP * 64) + lane
                   : nullptr;
          auto keep = [&](int child_index, const double (&y)[K][4]) {
#pragma unroll
            for (int j = 0; j < K; j++) {
              double2* dst = region + ((j / KP) * children + child_index) * (KP * 64) + (j % KP) * 64;
              dst[0] = make_double2(y[j][0], y[j][1]);
              dst[32] = make_double2(y[j][2], y[j][3]);
            }
          };
          double ya[K][4], yb[K][4];
          const double* const part_b = operand + (a_leaf ? kLeafPart : kInnerPart);
          // ---- child a
          if (a_leaf) {
            const uint32_t states_a = tip_states(tips_at);
#pragma unroll
            for (int j = 0; j < K; j++)
              if constexpr (AMBIG) LoadAmbiguousTipRow(operand + cat * kTipTableDoubles, states_a, j, ya[j]);
              else Load4(operand + cat * kTipTableDoubles + tip_row(states_a, j), ya[j]);
            if (RESCALE) {
#pragma unroll
              for (int j = 0; j < K; j++) cur_exp[j] = 0;
            }
          } else {
            MatVecOe<K>(operand + cat * kPStride, cur, ya);
            if (GRAD) keep(0, ya);
          }
          // ---- child b
          if (b_leaf) {
            const uint32_t states_b = tip_states(tips_at + kTipBytes);
#pragma unroll
            for (int j = 0; j < K; j++)
              if constexpr (AMBIG) LoadAmbiguousTipRow(part_b + cat * kTipTableDoubles, states_b, j, yb[j]);
              else Load4(part_b + cat * kTipTableDoubles + tip_row(states_b, j), yb[j]);
          } else {
            const int s2 = (record.y >> 16) & 0xff;
            double x[K][4];
#pragma unroll
            for (int j = 0; j < K; j++) {
              const double2* src = my_stack + (static_cast<size_t>(s2) * K + j) * kRow;
              const double2 v0 = src[0], v1 = src[kThreads];
              x[j][0] = v0.x, x[j][1] = v0.y, x[j][2] = v1.x, x[j][3] = v1.y;
              if (RESCALE) cur_exp[j] += my_stack_exps[(s2 * K + j) * kThreads];
            }
            MatVecOe<K>(part_b + cat * kPStride, x, yb);
            if (GRAD) keep(1, yb);
          }
#pragma unroll
          for (int j = 0; j < K; j++)
#pragma unroll
            for (int i = 0; i < 4; i++) cur[j][i] = ya[j][i] * yb[j][i];
          if (RESCALE) NormalizeOe<C, K, kOeLazyBits>(cur, cur_exp);
          if (flags & kRoot) {
            // beagleCalculateRootLogLikelihoods: log sum_c p_c sum_i pi_i L[c,k,i] (+ scale)
            double freqs[4];
            Load4(freqs_smem, freqs);
            uint32_t masks = 0;  // +I: the states all tips allow, one byte per pattern
            double pinv = 0.0;
            // +I gradient runs: this tile's D and E_s (E only for the analytic substitution gradient)
            double dinv = 0.0, einv[SUBST ? 4 : 1] = {};
            if constexpr (INVAR) {
              const uint8_t* const at = p.invariant_masks + pat0 + pidx * K;
              masks = K == 4 ? *reinterpret_cast<const uint32_t*>(at)
                             : (K == 2 ? *reinterpret_cast<const uint16_t*>(at) : *at);
              pinv = model.pinv;
            }
#pragma unroll
            for (int j = 0; j < K; j++) {
              double site = cat_weight * Dot4(freqs, cur[j]);
#pragma unroll
              for (int s = kPerWarp; s < 32; s <<= 1) site += __shfl_xor_sync(0xffffffffu, site, s);
              double log_site = log(site);
              if (RESCALE) log_site = fma(static_cast<double>(cur_exp[j]), 0.6931471805599453094, log_site);
              InvariantSiteTerms inv{};
              double invariant = 0.0;
              if constexpr (INVAR) {
                const unsigned mask = (masks >> (8 * j)) & 15u;
#pragma unroll
                for (int s = 0; s < 4; s++)
                  if (mask >> s & 1u) invariant += freqs[s];
                inv = InvariantSite(log_site, site, RESCALE ? cur_exp[j] : 0, pinv, invariant);
                log_site = inv.log_lik;
              }
              if constexpr (SITES) {
                // the same lane stores it, whatever the weight; the padding is never written
                const int64_t pattern = pat0 + pidx * K + j;
                if (cat == 0 && pattern < p.pattern_end)
                  p.site_logl[static_cast<int64_t>(vt) * (p.pattern_end - p.pattern_begin) + (pattern - p.pattern_begin)] =
                      log_site;
              }
              // one lane per pattern carries the term
              logl_acc = fma(w[j], (w[j] != 0.0 && cat == 0) ? log_site : 0.0, logl_acc);
              if constexpr (INVAR && GRAD) {
                if (w[j] != 0.0 && cat == 0) {
                  dinv += w[j] * (inv.inv_over_lik - inv.var_over_lik);
                  if constexpr (SUBST) {
                    const unsigned mask = (masks >> (8 * j)) & 15u;
                    const double share = invariant > 0.0 ? w[j] * inv.inv_over_lik / invariant : 0.0;
#pragma unroll
                    for (int s = 0; s < 4; s++)
                      if (mask >> s & 1u) einv[SUBST ? s : 0] += share;
                  }
                }
                // every derivative of the variable part is weighted by f = (1 - pinv) L / lik:
                // the pre-order pass below forms all of them from w
                w[j] *= inv.f;
              }
            }
            if constexpr (INVAR && GRAD) {
              // added to the warp's row at once (single writer, in tile order), so that no
              // accumulator stays live through the pre-order pass
              double* const sums = p.inv_partial + out_row * kOeInvariantSums;
              const double d_total = WarpSum(dinv);
              if (lane == 0) sums[0] += d_total;
              if constexpr (SUBST) {
#pragma unroll
                for (int s = 0; s < 4; s++) {
                  const double e_total = WarpSum(einv[s]);
                  if (lane == 0) sums[1 + s] += e_total;
                }
              }
            }
            if (GRAD) {
              // The pre-order pass starts at the root with T = p_c pi (its operand block
              // holds an identity in the place of the root's P).  Carrying the category
              // proportion in the pre-order partials makes pp . L the category's share of
              // the site likelihood and every numerator already weighted by p_c.
#pragma unroll
              for (int j = 0; j < K; j++)
#pragma unroll
                for (int i = 0; i < 4; i++) cur[j][i] = cat_weight * freqs[i];
              // It reads the arena back through bulk copies (the async proxy), which was
              // written with ordinary stores: the root's own blocks first.
              asm volatile("fence.proxy.async;" ::: "memory");
              __syncwarp();
              if (lane == 0) {
#pragma unroll
                for (int batch = 0; batch < kBatches; batch++) fetch_readback(record.z, children, batch);
              }
            }
          }
        } else {
          // ================ pre-order op + edge derivatives ================
          // operand layout: own P (an identity at the root), tip tables of a, tip tables of b
          const double* const table_a = operand + kInnerPart + kPhiPart;
          const double* const table_b = table_a + (a_leaf ? 2 * kLeafPart + kPhiPart : 0);
          const int next_children = ((flags & kNextALeaf) ? 0 : 1) + ((flags & kNextBLeaf) ? 0 : 1);
          // read-back order of two internal children: the post-order op's child order
          const bool swapped = flags & kArenaSwapped;
          const uint32_t states_a = a_leaf ? tip_states(tips_at) : 0;
          const uint32_t states_b = b_leaf ? tip_states(tips_at + kTipBytes) : 0;
          double g_own = 0.0, g_a = 0.0, g_b = 0.0;
#pragma unroll
          for (int batch = 0; batch < kBatches; batch++) {
            const int j0 = batch * KP;  // this sub-batch: patterns j0 .. j0 + KP - 1
            double(&top)[KP][4] = *reinterpret_cast<double(*)[KP][4]>(&cur[j0]);
            // ---- pre-order partial at this node: pp = P^T T
            double pp[KP][4];
            double tv[SUBST ? KP : 1][4];  // T_v itself, for the substitution gradient of v's edge
            if (flags & kStackBefore) {
              const int s0 = record.y & 0xff;
              double x[KP][4];
#pragma unroll
              for (int j = 0; j < KP; j++) {
                const double2* src = my_stack + (static_cast<size_t>(s0) * K + j0 + j) * kRow;
                const double2 v0 = src[0], v1 = src[kThreads];
                x[j][0] = v0.x, x[j][1] = v0.y, x[j][2] = v1.x, x[j][3] = v1.y;
              }
              MatTVecSharedK<KP>(operand + cat * kPStride, x, pp);
              if (SUBST) {
#pragma unroll
                for (int j = 0; j < KP; j++)
#pragma unroll
                  for (int i = 0; i < 4; i++) tv[j][i] = x[j][i];
              }
            } else {
              MatTVecSharedK<KP>(operand + cat * kPStride, top, pp);
              if (SUBST) {
#pragma unroll
                for (int j = 0; j < KP; j++)
#pragma unroll
                  for (int i = 0; i < 4; i++) tv[j][i] = top[j][i];
              }
            }
            // ---- evolved partials of both children
            double ya[KP][4], yb[KP][4];
            const double2* const slot = my_readback + batch * kBatchSlot + lane;
            MbarWait(readback_full + batch, readback_sequence & 1);
            if (a_leaf) {
#pragma unroll
              for (int j = 0; j < KP; j++)
                if constexpr (AMBIG) LoadAmbiguousTipRow(table_a + cat * kTipTableDoubles, states_a, j0 + j, ya[j]);
                else Load4(table_a + cat * kTipTableDoubles + tip_row(states_a, j0 + j), ya[j]);
            } else {
              const double2* const slot_a = slot + ((swapped && !b_leaf) ? KP * 64 : 0);
#pragma unroll
              for (int j = 0; j < KP; j++) {
                const double2 v0 = slot_a[j * 64], v1 = slot_a[j * 64 + 32];
                ya[j][0] = v0.x, ya[j][1] = v0.y, ya[j][2] = v1.x, ya[j][3] = v1.y;
              }
            }
            if (b_leaf) {
#pragma unroll
              for (int j = 0; j < KP; j++)
                if constexpr (AMBIG) LoadAmbiguousTipRow(table_b + cat * kTipTableDoubles, states_b, j0 + j, yb[j]);
                else Load4(table_b + cat * kTipTableDoubles + tip_row(states_b, j0 + j), yb[j]);
            } else {
              const double2* const slot_b = slot + (swapped ? 0 : KP * 64);
#pragma unroll
              for (int j = 0; j < KP; j++) {
                const double2 v0 = slot_b[j * 64], v1 = slot_b[j * 64 + 32];
                yb[j][0] = v0.x, yb[j][1] = v0.y, yb[j][2] = v1.x, yb[j][3] = v1.y;
              }
            }
            // ---- site likelihood, reduced over the pattern's categories
            double site[KP][4], scale[KP];
#pragma unroll
            for (int j = 0; j < KP; j++) {
#pragma unroll
              for (int i = 0; i < 4; i++) site[j][i] = ya[j][i] * yb[j][i];
              double d = Dot4(pp[j], site[j]);
#pragma unroll
              for (int s = kPerWarp; s < 32; s <<= 1) d += __shfl_xor_sync(0xffffffffu, d, s);
              // padding patterns contribute nothing (and may be 0/0)
              scale[j] = (w[j0 + j] != 0.0) ? w[j0 + j] * FastReciprocalOe(d) : 0.0;
              // (one category: no reduction above; this exchange is the dependency the
              //  copy below is issued behind -- 0 x a finite likelihood changes nothing)
              if (C == 1) scale[j] = fma(0.0, __shfl_xor_sync(0xffffffffu, d, 16), scale[j]);
            }
            // This sub-batch's read-back slot is free again: start the next op's copy.  The
            // slot was read through the generic proxy and the copy writes it through the
            // async proxy, and nothing but a proxy fence orders the two (measured without
            // one: run-to-run differences of 1e-5 in single edge derivatives when the
            // warps run fast; a fence.proxy.async here costs 10 % of the kernel).  The
            // shuffles above consumed values computed from every lane's loads, so by now
            // the loads have been performed: the copy is issued behind that dependency.
            if (lane == 0 && o + 1 < ops_total) fetch_readback(record.w, next_children, batch);

            // ---- own edge: T^T Q P L = pp . (Q L)   (computed and dropped at the root)
            {
              double num[KP];
              MatVecDotOe<KP>(q_smem, site, pp, num);
#pragma unroll
              for (int j = 0; j < KP; j++) g_own = fma(scale[j], num[j], g_own);
            }
            if (SUBST) {
              // v's own edge: T_v and L_v = site (Phi is zero in the root's block)
              double z[KP][4];
              MatVecOe<KP>(ivec_smem, site, z);
              accumulate_subst(*reinterpret_cast<const double(*)[KP][4]>(&tv[0]), z, scale,
                               operand + kInnerPart + cat * kOePhiDoubles);
              if (flags & kRoot) {
#pragma unroll
                for (int j = 0; j < KP; j++)
#pragma unroll
                  for (int l = 0; l < 4; l++)
                    rsub[SUBST ? l : 0] = fma(scale[j] * cat_weight, site[j][l], rsub[SUBST ? l : 0]);
              }
            }
            // ---- the partials at the top of the children's edges: T_a (kept in cur), T_b
#pragma unroll
            for (int j = 0; j < KP; j++)
#pragma unroll
              for (int i = 0; i < 4; i++) {
                top[j][i] = pp[j][i] * yb[j][i];
                yb[j][i] = pp[j][i] * ya[j][i];
              }
            if (a_leaf) {
#pragma unroll
              for (int j = 0; j < KP; j++) {
                double d[4];
                if constexpr (AMBIG) LoadAmbiguousTipRow(table_a + (C + cat) * kTipTableDoubles, states_a, j0 + j, d);
                else Load4(table_a + (C + cat) * kTipTableDoubles + tip_row(states_a, j0 + j), d);
                g_a = fma(scale[j], Dot4(top[j], d), g_a);
              }
              if (SUBST) {
                double z[KP][4];
#pragma unroll
                for (int j = 0; j < KP; j++) Load4(tip_z_smem + tip_row(states_a, j0 + j), z[j]);
                accumulate_subst(top, z, scale, table_a + 2 * kLeafPart + cat * kOePhiDoubles);
              }
            }
            if (RESCALE) {
              // pp . L is the pattern's root likelihood divided by the scale factors its
              // ancestors' own rescalings applied, so down a deep tree it shrinks (a
              // 1000-taxon ladder underflows without this).  All lanes of a pattern hold
              // the same reduced value: when it has dropped below 2^-kOePreBits the
              // partials handed down are scaled by its inverse power of two -- the scale
              // cancels in every numerator / denominator below.  Rare: one vote per batch.
              // (tested on scale = weight / (pp . L), whose power of two serves as the factor)
              bool low = false;
#pragma unroll
              for (int j = 0; j < KP; j++) low = low || (__double2hiint(scale[j]) > ((1023 + kOePreBits) << 20));
              if (__any_sync(0xffffffffu, low)) {
#pragma unroll
                for (int j = 0; j < KP; j++) {
                  const int biased = (__double2hiint(scale[j]) >> 20) & 0x7ff;
                  if (biased <= 1023 + kOePreBits || biased == 0x7ff) continue;
                  const double boost = __hiloint2double(biased << 20, 0);
#pragma unroll
                  for (int i = 0; i < 4; i++) {
                    top[j][i] *= boost;               // T_a (dead if a is a tip: its term is in g_a already)
                    if (!b_leaf) yb[j][i] *= boost;   // T_b, pushed below (a tip's term uses it as is)
                  }
                }
              }
            }
            if (b_leaf) {
#pragma unroll
              for (int j = 0; j < KP; j++) {
                double d[4];
                if constexpr (AMBIG) LoadAmbiguousTipRow(table_b + (C + cat) * kTipTableDoubles, states_b, j0 + j, d);
                else Load4(table_b + (C + cat) * kTipTableDoubles + tip_row(states_b, j0 + j), d);
                g_b = fma(scale[j], Dot4(yb[j], d), g_b);
              }
              if (SUBST) {
                double z[KP][4];
#pragma unroll
                for (int j = 0; j < KP; j++) Load4(tip_z_smem + tip_row(states_b, j0 + j), z[j]);
                accumulate_subst(yb, z, scale, table_b + 2 * kLeafPart + cat * kOePhiDoubles);
              }
            } else {
              const int s2 = (record.y >> 16) & 0xff;
#pragma unroll
              for (int j = 0; j < KP; j++) {
                double2* dst = my_stack + (static_cast<size_t>(s2) * K + j0 + j) * kRow;
                dst[0] = make_double2(yb[j][0], yb[j][1]);
                dst[kThreads] = make_double2(yb[j][2], yb[j][3]);
              }
            }
          }
          readback_sequence++;
          // ---- one transposed warp reduction per op: 8 slots
          //   slot 0..2 = rate_w x (own, a, b), slot 4..6 = drate_w x (own, a, b); after the
          //   exchange over lane bits 16, 8 and 4 the lane with bits (h, m, l) holds slot
          //   4h + 2m + l, summed over the warp by the last two steps.
          {
            const bool up16 = lane & 16, up8 = lane & 8, up4 = lane & 4;
            double r0, r1, r2;
            if (C > 1) {
              const double a0 = rate_w * g_own, a1 = rate_w * g_a, a2 = rate_w * g_b;
              const double b0 = drate_w * g_own, b1 = drate_w * g_a, b2 = drate_w * g_b;
              r0 = (up16 ? b0 : a0) + __shfl_xor_sync(0xffffffffu, up16 ? a0 : b0, 16);
              r1 = (up16 ? b1 : a1) + __shfl_xor_sync(0xffffffffu, up16 ? a1 : b1, 16);
              r2 = (up16 ? b2 : a2) + __shfl_xor_sync(0xffffffffu, up16 ? a2 : b2, 16);
            } else {
              // one category: no rate-gradient rows; both halves of the warp sum slots 0..2
              r0 = rate_w * g_own, r1 = rate_w * g_a, r2 = rate_w * g_b;
              r0 += __shfl_xor_sync(0xffffffffu, r0, 16);
              r1 += __shfl_xor_sync(0xffffffffu, r1, 16);
              r2 += __shfl_xor_sync(0xffffffffu, r2, 16);
            }
            const double q0 = (up8 ? r2 : r0) + __shfl_xor_sync(0xffffffffu, up8 ? r0 : r2, 8);
            const double q1 = (up8 ? 0.0 : r1) + __shfl_xor_sync(0xffffffffu, up8 ? r1 : 0.0, 8);
            double r = (up4 ? q1 : q0) + __shfl_xor_sync(0xffffffffu, up4 ? q0 : q1, 4);
            r += __shfl_xor_sync(0xffffffffu, r, 2);
            r += __shfl_xor_sync(0xffffffffu, r, 1);
            // Single writer per (row, edge), in program order, so the sums are
            // deterministic; a reduction (no return value) keeps the round trip to
            // L2 off the warp's critical path.
            if ((lane & 3) == 0) {
              const int which = (lane >> 2) & 3;  // 0 own edge, 1 tip child a, 2 tip child b
              const int2 tip_ids = *reinterpret_cast<const int2*>(stage + 8);
              int edge = -1;
              if (which == 0) edge = (flags & kRoot) ? -1 : (record.x & 0xffffff);
              if (which == 1) edge = a_leaf ? tip_ids.x : -1;
              if (which == 2) edge = b_leaf ? tip_ids.y : -1;
              if (edge >= 0) {
                if (!up16) {
                  atomicAdd(grad_row + edge, r);
                } else if (C > 1) {
                  atomicAdd(rgrad_row + edge, r);
                }
              }
            }
          }
        }
        __syncwarp();  // every lane is done reading this stage
        if (lane == 0) MbarArrive(empty + stage_index);
      }
    }
    // one partial per warp, in lane order
    logl_acc = WarpSum(logl_acc);
    if (lane == 0) p.logl_partial[out_row] = logl_acc;
    if (SUBST) {
      double* const sums = p.subst_partial + out_row * kOeSubstSums;
#pragma unroll
      for (int e = 0; e < 16; e++) {
        const double total = WarpSum(wsub[SUBST ? e : 0]);
        if (lane == 0) sums[e] = total;
      }
#pragma unroll
      for (int e = 0; e < 4; e++) {
        const double total = WarpSum(rsub[SUBST ? e : 0]);
        if (lane == 0) sums[16 + e] = total;
      }
    }
  }
}

}  // namespace sbnb

#endif  // SBNB_WALK_OE_CUH_
