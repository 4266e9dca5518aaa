// libsbn_b200 engine: device buffers, staging, kernel launches and the C ABI of
// include/sbn_b200.h.  Replaces the reference's Engine / FatBeagle pair
// (src/engine.cpp, src/fat_beagle.cpp) and the BEAGLE instance they drive.
//
// There is deliberately no CPU path in this file: without a CUDA device every
// entry point fails.

#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <exception>
#include <mutex>
#include <thread>
#include <unordered_map>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "common.hpp"
#include "device_common.cuh"
#include "kernels.cuh"
#include "walk_oe.cuh"
#include "model.hpp"
#include "rooted.hpp"
#include "tree_program.hpp"

namespace sbnb {

namespace {

thread_local std::string g_last_error;

// Category counts the tree walk is instantiated for (the lanes of a pattern hold
// one category each, so powers of two); other counts run padded
// with zero-weight categories.
int PadCategories(int c) {
  for (int supported : {1, 2, 4, 8, 16, 32})
    if (c <= supported) return supported;
  return 0;
}

}  // namespace

void SetLastError(const std::string& message) { g_last_error = message; }

}  // namespace sbnb

using namespace sbnb;

struct sbnb_engine {
  ModelSpec spec;
  int device = 0;
  int sm_count = 0;
  int taxon_count = 0;
  int64_t pattern_count = 0;
  int64_t tip_pitch = 0;
  int64_t range_begin = 0, range_end = 0;
  int categories = 1;         // C
  int padded_categories = 1;  // instantiated count >= C (extra categories have weight 0)
  // host copy of the alignment (shared by the children of a device group)
  std::shared_ptr<const std::vector<uint8_t>> host_tips;    // [taxon][pattern], tip codes 0..14 (walk_oe.cuh)
  bool ambiguous = false;  // some tip code is >= kFirstAmbiguousCode: the walks sum tip-table rows
  std::shared_ptr<const std::vector<double>> host_weights;  // [pattern]
  cudaStream_t stream = nullptr;
  // CUDA-event pairs bracketing the base tree-walk launch of the last
  // kWalkRing runs; harvested into (walk_total_ms, walk_samples).
  static constexpr int kWalkRing = 32;
  cudaEvent_t walk_begin[kWalkRing] = {}, walk_end[kWalkRing] = {};
  bool walk_pending[kWalkRing] = {};
  int64_t walk_runs = 0;
  double walk_total_ms = 0.0, walk_last_ms = 0.0;
  int64_t walk_samples = 0;
  int64_t launch_count = 0;
  int64_t h2d_bytes = 0, d2h_bytes = 0;
  // Page-locked staging: `staging` carries one batch to the device in one copy
  // (staging_free is recorded behind that copy: the arena is rewritten by the next
  // Stage, which waits for it instead of synchronising the stream); `landing`
  // receives one batch's results in one copy.
  PinnedArena staging, landing;
  cudaEvent_t staging_free = nullptr;
  bool staging_in_flight = false;
  DeviceArray<uint8_t> tips;
  DeviceArray<double> weights;
  DeviceArray<uint8_t> invariant_masks;  // +I: [tip_pitch] states every tip allows (InvariantMaskKernel)
  DeviceArray<double2> arena;  // evolved post-order partial arena, reused by every gradient run
  DeviceArray<double2> stack;  // per-CTA partial stacks
  DeviceArray<int32_t> stack_exps;
  DeviceArray<double> fd_operands;  // operand blocks of one slice of finite-difference evaluations

  // A destroyed batch parks here so that the next Stage() of the one-call entry
  // points (which stage per call) neither cudaMallocs nor cudaFrees, and finds the
  // traversal programs of an unchanged topology set already on the device.
  sbnb_batch* spare = nullptr;
  // resident CTAs per SM of every walk kernel this engine has launched: kernel -> (smem, CTAs)
  std::unordered_map<const void*, std::pair<size_t, int>> occupancy;

  // Multi-GPU group (sbnb_engine_create_multi): this object is then only a front
  // for one child engine per device; see the "device groups" section below.
  std::vector<sbnb_engine*> children;
  int shard_axis = 0;
  // How "substitution_model" gradients are computed: analytically in the gradient sweep
  // (default), or by the reference's 16 central-difference log-likelihood sweeps.
  int substitution_mode = SBNB_SUBSTITUTION_ANALYTIC;

  ~sbnb_engine();
};

struct sbnb_batch {
  int tree_count = 0;
  int taxon_count = 0;
  int node_count = 0;  // 2n-1
  bool rooted = false;
  bool slide_root = false;
  int fd_coords = 0;  // stick-breaking coordinates perturbed (0 if no FD staged)
  bool with_subst = false;  // staged for the analytic substitution gradient (Phi in the pre-order blocks)
  bool rooted_finish = false;  // time-tree fields staged: gradient runs end with RootedFinishKernel
  bool invariant = false;      // +I: gradient runs also reduce the kOeInvariantSums sums per tree
  int site_width = 1;          // entries of a tree's site-model gradient (ModelSpec::SiteGradientSize)
  int rate_count = 0;
  size_t children_at = 0, rooted_fields_at = 0;
  DeviceArray<double> rooted_scratch;
  int vtree_count = 0;
  int slots = 1;
  int last_mode = -1;
  int64_t patterns = 0;  // pattern range of the engine when staged
  int categories = 1;
  // host side, kept for the O(n) finishing steps
  std::vector<TreeProgram> programs;
  std::vector<double> lengths;  // [T][2n-1] after detrifurcation / rate scaling / root slide
  // The topology set whose programs are on the device (variational inference
  // re-evaluates the same trees with new branch lengths, vip/burrito.py:84-117).
  std::vector<int32_t> cached_parent_ids;
  int cached_input_nodes = 0, cached_padded_categories = 0;
  bool cached_with_subst = false, cached_rooted_finish = false;
  // device side: one packed input buffer
  //   [lengths | models | vtree_program | vtree_model | vtree_lengths]   every call
  //   [ops | edge_offsets]                                              per topology set
  DeviceArray<unsigned char> input;
  size_t lengths_at = 0, models_at = 0, vtree_program_at = 0, vtree_model_at = 0, vtree_lengths_at = 0,
         ops_at = 0, edge_offsets_at = 0;
  int64_t post_doubles = 0, full_doubles = 0;  // operand block of a logL-only / a gradient evaluation
  int64_t operand_stride = 0;                  // of the base trees' blocks in `operands` (last run)
  DeviceArray<double> operands;                // operand blocks of the base trees
  DeviceArray<double> logl_partial, grad_partial, rgrad_partial, subst_partial, inv_partial;
  // [logl (vtree_count) | grad (T x N) | rgrad (T x N) | subst sums (T x 20) | +I sums (T x 5) | rooted finish]
  DeviceArray<double> results;
  // tiling of the last run
  int chunks = 1;
  // One-call entry points on an unchanged topology set replay the launch sequence
  // [matrices, walk(s), reduce, results -> host] as a CUDA graph (one per mode and
  // rescaling flag), re-captured whenever a buffer it names has moved.
  struct Graph {
    cudaGraphExec_t exec = nullptr;
    std::vector<uintptr_t> signature;
    int kernels = 0;
    bool warm = false;  // this very sequence has run eagerly since the programs were staged: buffers sized
  };
  Graph graphs[2][2];
  int cache_hits = 0;  // consecutive Stage() calls that found the programs on the device
  ~sbnb_batch() {
    for (auto& row : graphs)
      for (auto& graph : row)
        if (graph.exec) cudaGraphExecDestroy(graph.exec);
  }

  template <typename T>
  T* At(size_t offset) const {
    return reinterpret_cast<T*>(input.get() + offset);
  }
  double* ResultLogl() const { return results.get(); }
  double* ResultGrad() const { return results.get() + vtree_count; }
  double* ResultRateGrad() const { return ResultGrad() + static_cast<size_t>(tree_count) * node_count; }
  double* ResultSubst() const { return ResultRateGrad() + static_cast<size_t>(tree_count) * node_count; }
  double* ResultInvariant() const { return ResultSubst() + static_cast<size_t>(tree_count) * kOeSubstSums; }
  double* ResultRooted() const { return ResultInvariant() + static_cast<size_t>(tree_count) * kOeInvariantSums; }
  // per tree: n-1 ratio / root-height entries, the clock gradient, the site-model gradient
  size_t RootedWidth() const { return static_cast<size_t>(taxon_count - 1) + rate_count + site_width; }
};

sbnb_engine::~sbnb_engine() {
  for (sbnb_engine* child : children) {
    cudaSetDevice(child->device);
    delete child;
  }
  delete spare;
  for (int i = 0; i < kWalkRing; i++) {
    if (walk_begin[i]) cudaEventDestroy(walk_begin[i]);
    if (walk_end[i]) cudaEventDestroy(walk_end[i]);
  }
  if (staging_free) cudaEventDestroy(staging_free);
  if (stream) cudaStreamDestroy(stream);
}

namespace {

// Parks a finished batch in its engine for reuse (see sbnb_engine::spare).
void Recycle(sbnb_engine* e, sbnb_batch* batch) {
  if (!batch) return;
  if (e && !e->spare) {
    batch->last_mode = -1;
    e->spare = batch;
  } else {
    delete batch;
  }
}
struct BatchRecycler {
  sbnb_engine* engine;
  void operator()(sbnb_batch* batch) const { Recycle(engine, batch); }
};
using BatchPtr = std::unique_ptr<sbnb_batch, BatchRecycler>;

struct LaunchPlan {
  int tiles_total, tiles_per_chunk, chunks, grid;
  size_t smem_bytes;
};

// Plans (and launches) TreeWalkOeKernel, whose tiles are kThreads / C * K patterns.
template <int C, int K, bool GRAD, bool RESCALE, bool SUBST, bool AMBIG, bool INVAR>
LaunchPlan PlanAndLaunchOe(sbnb_engine* e, OeParams p, bool launch, int chunks_override) {
  auto kernel = TreeWalkOeKernel<C, K, GRAD, RESCALE, SUBST, AMBIG, INVAR>;
  // (SBNB_EXTRA_SMEM: development aid -- pads the request to lower the resident CTA count)
  const size_t smem =
      OeSmemBytes(C, K, GRAD, SUBST, AMBIG) + static_cast<size_t>(std::max(0, EnvInt("SBNB_EXTRA_SMEM", 0)));
  // (attributes and occupancy of a kernel are asked for once per engine)
  auto known = e->occupancy.find(reinterpret_cast<const void*>(kernel));
  if (known == e->occupancy.end() || known->second.first != smem) {
    int per_sm_now = 0;
    SBNB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    SBNB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                   cudaSharedmemCarveoutMaxShared));
    SBNB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_now, kernel, kThreads, smem));
    known = e->occupancy.insert_or_assign(reinterpret_cast<const void*>(kernel), std::make_pair(smem, per_sm_now)).first;
  }
  const int cached_per_sm = known->second.second;
  const int per_sm = cached_per_sm;
  if (per_sm < 1) Fail(SBNB_ERR_CUDA, "TreeWalkOeKernel does not fit on an SM.");
  const int resident = per_sm * e->sm_count;
  constexpr int kTilePatterns = OeTilePatterns(C, K);
  LaunchPlan plan;
  const int64_t patterns = p.pattern_end - p.pattern_begin;
  plan.tiles_total = static_cast<int>((patterns + kTilePatterns - 1) / kTilePatterns);
  if (chunks_override > 0) {
    plan.chunks = chunks_override;
    plan.tiles_per_chunk = (plan.tiles_total + plan.chunks - 1) / plan.chunks;
  } else {
    // Enough (tree, chunk) work items to give every resident CTA ~4 of them, and
    // enough chunks per tree that the CTAs resident at any moment work on few
    // distinct trees: consecutive items are the chunks of one tree, and every tree
    // in flight keeps its ~0.3 MB of operand blocks in L2 next to the arena
    // stream (1024 trees at 2 chunks each had 222 trees -- 81 MB -- in flight).
    int64_t want = (4LL * resident + p.vtree_count - 1) / std::max(p.vtree_count, 1);
    const int in_flight = std::max(1, EnvInt("SBNB_TREES_IN_FLIGHT", 16));
    want = std::max<int64_t>(want, (resident + in_flight - 1) / in_flight);
    want = std::max<int64_t>(1, std::min<int64_t>(want, plan.tiles_total));
    plan.tiles_per_chunk = static_cast<int>((plan.tiles_total + want - 1) / want);
    plan.chunks = (plan.tiles_total + plan.tiles_per_chunk - 1) / plan.tiles_per_chunk;
  }
  const int64_t items = static_cast<int64_t>(p.vtree_count) * plan.chunks;
  plan.grid = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>(items, resident)));
  plan.smem_bytes = smem;
  if (launch) {
    p.tiles_total = plan.tiles_total;
    p.tiles_per_chunk = plan.tiles_per_chunk;
    p.chunks = plan.chunks;
    const size_t block = static_cast<size_t>(K) * 2 * kThreads;  // double2 per partial block
    const size_t slots = static_cast<size_t>(std::max(p.slots, 1));
    e->stack.Reserve(static_cast<size_t>(plan.grid) * slots * block);
    p.stack = e->stack.get();
    if (RESCALE) {
      e->stack_exps.Reserve(static_cast<size_t>(plan.grid) * slots * K * kThreads);
      p.stack_exps = e->stack_exps.get();
    }
    if (GRAD) {
      e->arena.Reserve(static_cast<size_t>(plan.grid) * std::max(p.taxon_count - 2, 1) * block);
      p.arena = e->arena.get();
    }
    kernel<<<plan.grid, kThreads, smem, e->stream>>>(p);
    SBNB_CUDA(cudaGetLastError());
    e->launch_count++;
  }
  return plan;
}

template <int C, int K, bool GRAD, bool SUBST, bool AMBIG, bool INVAR>
LaunchPlan DispatchRescale(sbnb_engine* e, const OeParams& p, bool rescale, bool launch, int chunks_override) {
  return rescale ? PlanAndLaunchOe<C, K, GRAD, true, SUBST, AMBIG, INVAR>(e, p, launch, chunks_override)
                 : PlanAndLaunchOe<C, K, GRAD, false, SUBST, AMBIG, INVAR>(e, p, launch, chunks_override);
}

// K_GRAD / K_LOGL patterns per thread for the gradient / logL-only walk; a gradient walk
// with p.subst_partial set also accumulates the analytic substitution-gradient sums.
template <int C, int K_GRAD, int K_LOGL, bool AMBIG, bool INVAR>
LaunchPlan DispatchModesOe(sbnb_engine* e, const OeParams& p, bool grad, bool rescale, bool launch,
                           int chunks_override) {
  if (grad && p.subst_partial != nullptr)
    return DispatchRescale<C, K_GRAD, true, true, AMBIG, INVAR>(e, p, rescale, launch, chunks_override);
  return grad ? DispatchRescale<C, K_GRAD, true, false, AMBIG, INVAR>(e, p, rescale, launch, chunks_override)
              : DispatchRescale<C, K_LOGL, false, false, AMBIG, INVAR>(e, p, rescale, launch, chunks_override);
}

// A site model with invariable sites (+I) runs the walks with the invariant class at the root
// op; every other model the walks without it (a compile-time variant: their code is unchanged).
template <int C, int K_GRAD, int K_LOGL, bool AMBIG>
LaunchPlan DispatchInvariantOe(sbnb_engine* e, const OeParams& p, bool grad, bool rescale, bool launch,
                               int chunks_override) {
  return e->spec.invariant
             ? DispatchModesOe<C, K_GRAD, K_LOGL, AMBIG, true>(e, p, grad, rescale, launch, chunks_override)
             : DispatchModesOe<C, K_GRAD, K_LOGL, AMBIG, false>(e, p, grad, rescale, launch, chunks_override);
}

// An alignment with ambiguous tip codes runs the walks that sum tip-table rows; any other
// runs the walks that read one row per tip.
template <int C, int K_GRAD, int K_LOGL>
LaunchPlan DispatchTipsOe(sbnb_engine* e, const OeParams& p, bool grad, bool rescale, bool launch,
                          int chunks_override) {
  return e->ambiguous ? DispatchInvariantOe<C, K_GRAD, K_LOGL, true>(e, p, grad, rescale, launch, chunks_override)
                      : DispatchInvariantOe<C, K_GRAD, K_LOGL, false>(e, p, grad, rescale, launch, chunks_override);
}

// Patterns per thread K: more of them amortise the per-op overhead (operand requests,
// barrier waits, reductions) but cost registers; the pre-order half of a gradient walk
// works through them two at a time (OePreBatch).  Tiles are kThreads / C * K patterns
// and must stay a multiple of 16.
LaunchPlan Dispatch(sbnb_engine* e, const OeParams& p, bool grad, bool rescale, bool launch,
                    int chunks_override) {
  switch (e->padded_categories) {
    case 1:
      return DispatchTipsOe<1, 2, 4>(e, p, grad, rescale, launch, chunks_override);
    case 2:
      return DispatchTipsOe<2, 2, 4>(e, p, grad, rescale, launch, chunks_override);
    case 4:
      // (measured: 4 patterns per thread at 12 warps/SM beat 2 at 16 warps/SM by 8 %)
      return DispatchTipsOe<4, 4, 4>(e, p, grad, rescale, launch, chunks_override);
    case 8:
      return DispatchTipsOe<8, 2, 2>(e, p, grad, rescale, launch, chunks_override);
    case 16:
      return DispatchTipsOe<16, 2, 2>(e, p, grad, rescale, launch, chunks_override);
    case 32:
      // (one pattern column per warp: tiles of 4 warps x 4 patterns)
      return DispatchTipsOe<32, 4, 4>(e, p, grad, rescale, launch, chunks_override);
  }
  Fail(SBNB_ERR_INVALID_ARGUMENT, "Unsupported category count.");
}

// (Re)builds the device copy of the alignment for patterns [begin, end): the
// range starts at column 0 of the device arrays (TMA bulk copies need 16-byte
// aligned rows), padded with gap states / zero weights so that the last tile
// needs no bounds checks (a tile is at most kThreads * 4 patterns).
void UploadPatternRange(sbnb_engine* e, int64_t begin, int64_t end) {
  const int64_t count = end - begin;
  e->tip_pitch = ((count + 511) / 512) * 512 + 512;
  std::vector<uint8_t> tips(static_cast<size_t>(e->taxon_count) * e->tip_pitch, 4);
  for (int taxon = 0; taxon < e->taxon_count; taxon++)
    std::copy(e->host_tips->begin() + static_cast<size_t>(taxon) * e->pattern_count + begin,
              e->host_tips->begin() + static_cast<size_t>(taxon) * e->pattern_count + end,
              tips.begin() + static_cast<size_t>(taxon) * e->tip_pitch);
  std::vector<double> weights(e->tip_pitch, 0.0);
  std::copy(e->host_weights->begin() + begin, e->host_weights->begin() + end, weights.begin());
  SBNB_CUDA(cudaStreamSynchronize(e->stream));  // nothing in flight reads the old arrays
  e->h2d_bytes += e->tips.Upload(tips.data(), tips.size(), e->stream);
  e->h2d_bytes += e->weights.Upload(weights.data(), weights.size(), e->stream);
  if (e->spec.invariant) {
    e->invariant_masks.Reserve(e->tip_pitch);
    const int block = 256;
    InvariantMaskKernel<<<static_cast<int>((e->tip_pitch + block - 1) / block), block, 0, e->stream>>>(
        e->tips.get(), e->tip_pitch, e->taxon_count, count, e->invariant_masks.get());
    SBNB_CUDA(cudaGetLastError());
    e->launch_count++;
  }
  SBNB_CUDA(cudaStreamSynchronize(e->stream));
  e->range_begin = begin;
  e->range_end = end;
}

void CheckTrees(const sbnb_engine* e, const sbnb_tree_batch* trees, bool rooted) {
  Require(trees != nullptr, "NULL tree batch.");
  Require(trees->tree_count >= 0, "Negative tree count.");
  if (trees->tree_count == 0) return;  // an empty collection evaluates to an empty result
  Require(trees->parent_ids && trees->branch_lengths, "NULL parent_ids / branch_lengths.");
  const int n = e->taxon_count;
  if (rooted) {
    Require(trees->node_count == 2 * n - 1,
            "Rooted trees must be bifurcating: node_count must be 2n-1.");
    Require(trees->rates != nullptr, "Rooted evaluation needs per-branch rates (RootedTree::rates_).");
  } else {
    Require(trees->node_count == 2 * n - 1 || trees->node_count == 2 * n - 2,
            "node_count must be 2n-2 (unrooted) or 2n-1 (bifurcating).");
  }
}

// Perturbed parameter rows of the finite-difference substitution gradient,
// in output order: GTR -> coordinates 0..4 = rates, 5..7 = frequencies
// (fat_beagle.cpp:455-464), each as (plus, minus).
void FiniteDifferenceRows(const ModelSpec& spec, const double* row, double delta,
                          std::vector<std::vector<double>>* rows) {
  rows->clear();
  auto perturb_simplex = [&](const std::string& key) {
    const auto [start, length] = spec.Block(key);
    std::vector<double> y(length - 1), x(length);
    StickBreakingInverse(row + start, length, y.data());
    for (int idx = 0; idx < length - 1; idx++) {
      for (int sign = +1; sign >= -1; sign -= 2) {
        std::vector<double> yy = y;
        yy[idx] += sign * delta;
        StickBreaking(yy.data(), length, x.data());
        std::vector<double> perturbed(row, row + spec.param_count);
        std::copy(x.begin(), x.end(), perturbed.begin() + start);
        rows->push_back(std::move(perturbed));
      }
    }
  };
  if (spec.substitution == SubstitutionKind::kGTR) {
    perturb_simplex("GTR rates");
    perturb_simplex("frequencies");
  } else if (spec.substitution == SubstitutionKind::kHKY) {
    const int kappa = spec.Block("kappa").first;
    for (int sign = +1; sign >= -1; sign -= 2) {
      std::vector<double> perturbed(row, row + spec.param_count);
      perturbed[kappa] += sign * delta;
      rows->push_back(std::move(perturbed));
    }
    perturb_simplex("frequencies");
  }
}

constexpr double kFiniteDifferenceDelta = 1.e-6;  // fat_beagle.cpp:454

// Host-side data parallelism over the trees of a batch (what the reference's
// TaskProcessor thread pool does, task_processor.hpp:43-112): contiguous chunks,
// one std::thread each; the first exception is rethrown on the calling thread.
template <typename F>
void ParallelOverTrees(int count, F&& body) {
  const int workers = std::max(1, std::min<int>({static_cast<int>(std::thread::hardware_concurrency()), 16,
                                                 count / 32}));
  if (workers <= 1) {
    for (int t = 0; t < count; t++) body(t);
    return;
  }
  std::vector<std::thread> threads;
  std::exception_ptr failure;
  std::mutex failure_mutex;
  for (int w = 0; w < workers; w++) {
    threads.emplace_back([&, w] {
      try {
        const int begin = static_cast<int>(static_cast<int64_t>(count) * w / workers);
        const int end = static_cast<int>(static_cast<int64_t>(count) * (w + 1) / workers);
        for (int t = begin; t < end; t++) body(t);
      } catch (...) {
        std::lock_guard<std::mutex> lock(failure_mutex);
        if (!failure) failure = std::current_exception();
      }
    });
  }
  for (auto& thread : threads) thread.join();
  if (failure) std::rethrow_exception(failure);
}

// The branch lengths one evaluation of tree t uses, indexed by node id of the
// bifurcating (2n-1 node) tree.
void EffectiveBranchLengths(const TreeProgram& program, const sbnb_tree_batch* trees, int t, bool rooted,
                            bool slide_root, int N, double* out) {
  const double* in = trees->branch_lengths + static_cast<size_t>(t) * trees->node_count;
  std::copy(in, in + trees->node_count, out);
  if (program.was_trifurcating) {
    // Detrifurcate (unrooted_tree.cpp:31-35): the node that takes the old
    // root's id and the new root both get length 0.
    out[N - 2] = 0.0;
    out[N - 1] = 0.0;
  }
  if (rooted) {
    // fat_beagle.cpp:96-101, 507-511
    const double* rates = trees->rates + static_cast<size_t>(t) * (N - 1);
    for (int i = 0; i < N - 1; i++) out[i] *= rates[i];
  } else if (slide_root) {
    // Tree::SlideRootPosition (tree.cpp:72-78), which the reference's unrooted Gradient
    // applies after Detrifurcate (fat_beagle.cpp:470-472): the root's second child gets
    // length 0, its first child the sum.  A no-op for a detrifurcated tree.
    const int fixed = program.child1[program.root], root_child = program.child0[program.root];
    out[root_child] += out[fixed];
    out[fixed] = 0.0;
  }
}

// Packs the two programs of one topology into the 32-byte records the kernel reads
// from its operand-block headers, assigns every op its operand block and every edge
// the places its matrices go, and returns the operand-block sizes (in doubles) of a
// logL-only and of a gradient evaluation.
//
// The children of every op are ordered for the kernel: child a is the internal child
// whose partial is in cur (post-order) or stays in cur (pre-order), child b the one
// that goes through the stack -- so a tip child a implies a tip child b, and the
// kernel has no "which child uses cur" cases.
void PackProgram(const TreeProgram& program, int n, int C, bool with_subst, OeOp* ops, int2* edge_offsets,
                 int64_t* post_doubles, int64_t* full_doubles) {
  const int phi_part = with_subst ? kOePhiDoubles * C : 0;  // behind every edge's part of a pre-order block
  Require(program.post_slots < 255 && program.pre_slots < 255 && 2 * n - 1 < (1 << 24), "Tree too large.");
  auto slot_byte = [](int32_t slot) { return slot < 0 ? 0xff : (slot & 0xff); };
  const int inner_part = kPStride * C, leaf_part = kTipTableDoubles * C;
  for (int e = 0; e < 2 * n - 2; e++) edge_offsets[e] = make_int2(-1, -1);
  std::vector<int32_t> arena_slot_of(2 * n - 1, 0), first_kept_child(2 * n - 1, -1);
  int64_t at = 0;  // doubles from the block start
  int arena_blocks = 0;
  for (int o = 0; o < n - 1; o++) {
    const PostOp& op = program.post[o];
    int a = op.a, b = op.b, a_src = op.a_src, b_src = op.b_src;
    if (b_src == kFromCur) std::swap(a, b), std::swap(a_src, b_src);
    const bool a_leaf = a < n, b_leaf = b < n;
    Require((a_leaf || a_src == kFromCur) && (b_leaf || b_src >= 0) && (!a_leaf || b_leaf),
            "internal error: unexpected operand sources in a post-order op");
    const int part_a = a_leaf ? leaf_part : inner_part, part_b = b_leaf ? leaf_part : inner_part;
    const int flags = (a_leaf ? kALeaf : 0) | (b_leaf ? kBLeaf : 0) | (op.flags & kRoot) |
                      (op.push_slot >= 0 ? kStackBefore : 0);
    OeOp& out = ops[o];
    out.operand_unit = static_cast<int32_t>(at / 2);
    out.operand_units = (kOeHeaderDoubles + part_a + part_b) / 2;
    out.tip_a = a_leaf ? a : -1;
    out.tip_b = b_leaf ? b : -1;
    out.node_flags = op.node | (flags << 24);
    out.slots = slot_byte(op.push_slot) | (0xff << 8) | (slot_byte(b_leaf ? -1 : b_src) << 16);
    out.arena_slot = arena_blocks;
    out.next_arena_slot = arena_blocks;  // the root's post-order op starts its own read-back
    arena_slot_of[op.node] = arena_blocks;
    first_kept_child[op.node] = a;
    arena_blocks += (a_leaf ? 0 : 1) + (b_leaf ? 0 : 1);
    edge_offsets[a].x = static_cast<int32_t>(at + kOeHeaderDoubles);
    edge_offsets[b].x = static_cast<int32_t>(at + kOeHeaderDoubles + part_a);
    at += kOeHeaderDoubles + part_a + part_b;
  }
  *post_doubles = at;
  auto ordered_pre = [&](const PreOp& op, int* a, int* b, int* b_dst) {
    *a = op.a, *b = op.b;
    int a_dst = op.a_dst;
    *b_dst = op.b_dst;
    if (*b_dst == kFromCur) std::swap(*a, *b), std::swap(a_dst, *b_dst);
    const bool a_leaf = *a < n, b_leaf = *b < n;
    Require((a_leaf || a_dst == kFromCur) && (b_leaf || *b_dst >= 0) && (!a_leaf || b_leaf),
            "internal error: unexpected destinations in a pre-order op");
  };
  for (int o = 0; o < n - 1; o++) {
    const PreOp& op = program.pre[o];
    int a, b, b_dst;
    ordered_pre(op, &a, &b, &b_dst);
    const bool a_leaf = a < n, b_leaf = b < n, root = op.flags & kRoot;
    int flags = (a_leaf ? kALeaf : 0) | (b_leaf ? kBLeaf : 0) | (op.flags & kRoot) |
                (op.pop_slot >= 0 ? kStackBefore : 0);
    // two internal children: their arena blocks are in the post-order op's order
    if (!a_leaf && !b_leaf && first_kept_child[op.node] != a) flags |= kArenaSwapped;
    OeOp& out = ops[n - 1 + o];
    int64_t part = kOeHeaderDoubles;
    if (!root) edge_offsets[op.node].y = static_cast<int32_t>(at + part);
    part += inner_part + phi_part;  // (the root's op gets an identity there)
    if (a_leaf) {
      edge_offsets[a].y = static_cast<int32_t>(at + part);
      part += 2 * leaf_part + phi_part;
    }
    if (b_leaf) {
      edge_offsets[b].y = static_cast<int32_t>(at + part);
      part += 2 * leaf_part + phi_part;
    }
    out.operand_unit = static_cast<int32_t>(at / 2);
    out.operand_units = static_cast<int32_t>(part / 2);
    out.tip_a = a_leaf ? a : -1;
    out.tip_b = b_leaf ? b : -1;
    out.slots = slot_byte(op.pop_slot) | (0xff << 8) | (slot_byte(b_leaf ? -1 : b_dst) << 16);
    out.arena_slot = arena_slot_of[op.node];
    out.next_arena_slot = 0;
    if (o + 1 < n - 1) {
      const PreOp& next = program.pre[o + 1];
      out.next_arena_slot = arena_slot_of[next.node];
      flags |= (next.a < n ? kNextALeaf : 0) | (next.b < n ? kNextBLeaf : 0);
    }
    out.node_flags = op.node | (flags << 24);
    at += part;
  }
  *full_doubles = at;
  Require(at / 2 < (int64_t{1} << 31), "Tree too large.");
}

RootedView ViewOf(const sbnb_tree_batch* trees, int t, int n);

// Waits until the copy out of the staging arena that the previous Stage queued has
// been done (normally long ago: every fetch synchronises the stream).
void WaitForStaging(sbnb_engine* e) {
  if (!e->staging_in_flight) return;
  SBNB_CUDA(cudaEventSynchronize(e->staging_free));
  e->staging_in_flight = false;
}

BatchPtr Stage(sbnb_engine* e, const sbnb_tree_batch* trees, const double* params, bool rooted,
               bool with_fd, bool slide_root, bool with_subst = false) {
  NvtxRange range("sbnb stage");
  CheckTrees(e, trees, rooted);
  const ModelSpec& spec = e->spec;
  Require(spec.param_count == 0 || params != nullptr || trees->tree_count == 0,
          "NULL phylo model parameter matrix.");
  SBNB_CUDA(cudaSetDevice(e->device));
  BatchPtr batch(e->spare ? e->spare : new sbnb_batch(), BatchRecycler{e});
  e->spare = nullptr;
  const int T = trees->tree_count, n = e->taxon_count, N = 2 * n - 1, C = e->padded_categories;
  const bool same_shape = batch->tree_count == T && batch->taxon_count == n;
  batch->tree_count = T;
  batch->taxon_count = n;
  batch->node_count = N;
  batch->rooted = rooted;
  batch->slide_root = slide_root && !rooted;
  batch->patterns = e->range_end - e->range_begin;
  batch->categories = e->categories;
  const int fd_evals = with_fd ? 2 * spec.SubstitutionGradientSize() : 0;
  batch->fd_coords = fd_evals / 2;
  batch->with_subst = with_subst;
  batch->invariant = spec.invariant;
  batch->site_width = spec.SiteGradientSize();
  batch->vtree_count = T * (1 + fd_evals);
  if (T == 0) return batch;

  // Layout of the packed input buffer (identical on the host and on the device): the
  // per-topology part first, so that its place does not depend on the model count.
  const size_t op_count = static_cast<size_t>(T) * 2 * (n - 1);
  const size_t edge_count = static_cast<size_t>(T) * (2 * n - 2);
  const size_t max_models = static_cast<size_t>(T) * (1 + fd_evals);
  size_t at = 0;
  auto place = [&at](size_t bytes) {
    const size_t here = at;
    at = (at + bytes + 255) / 256 * 256;
    return here;
  };
  batch->ops_at = place(op_count * sizeof(OeOp));
  batch->edge_offsets_at = place(edge_count * sizeof(int2));
  // Rooted time trees with all their fields: the O(n) gradient finishing runs on the device.
  batch->rooted_finish = rooted && trees->node_heights && trees->node_bounds && trees->height_ratios &&
                         (trees->rate_count == 1 || trees->rate_count == N - 1);
  batch->rate_count = batch->rooted_finish ? trees->rate_count : 0;
  batch->children_at = place(batch->rooted_finish ? static_cast<size_t>(T) * 2 * N * sizeof(int32_t) : 0);
  const size_t per_call_begin = at;
  const size_t rooted_stride = 4 * static_cast<size_t>(N) + n - 2;  // doubles per tree
  batch->rooted_fields_at = place(batch->rooted_finish ? static_cast<size_t>(T) * rooted_stride * sizeof(double) : 0);
  batch->lengths_at = place(static_cast<size_t>(T) * N * sizeof(double));
  batch->models_at = place(max_models * sizeof(ModelTables));
  batch->vtree_program_at = place(batch->vtree_count * sizeof(int32_t));
  batch->vtree_model_at = place(batch->vtree_count * sizeof(int32_t));
  batch->vtree_lengths_at = place(batch->vtree_count * sizeof(int32_t));
  const size_t total_bytes = at;

  // Is this the topology set whose programs are already on the device?
  const size_t id_count = static_cast<size_t>(T) * (trees->node_count - 1);
  const bool cached = same_shape && batch->cached_input_nodes == trees->node_count &&
                      batch->cached_padded_categories == C && batch->cached_with_subst == with_subst &&
                      batch->cached_rooted_finish == batch->rooted_finish &&
                      batch->cached_parent_ids.size() == id_count &&
                      batch->input.capacity() >= total_bytes &&
                      std::memcmp(batch->cached_parent_ids.data(), trees->parent_ids, id_count * sizeof(int32_t)) == 0;

  // Everything that goes to the device is assembled in page-locked memory.
  WaitForStaging(e);
  e->staging.Reset(total_bytes);
  unsigned char* host = e->staging.Take<unsigned char>(total_bytes);
  double* lengths = reinterpret_cast<double*>(host + batch->lengths_at);
  ModelTables* models = reinterpret_cast<ModelTables*>(host + batch->models_at);
  int32_t* vtree_program = reinterpret_cast<int32_t*>(host + batch->vtree_program_at);
  int32_t* vtree_model = reinterpret_cast<int32_t*>(host + batch->vtree_model_at);
  int32_t* vtree_lengths = reinterpret_cast<int32_t*>(host + batch->vtree_lengths_at);

  batch->cache_hits = cached ? batch->cache_hits + 1 : 0;
  if (!cached)
    for (auto& row : batch->graphs)
      for (auto& graph : row) graph.warm = false;
  if (!cached) {
    // Programs: host schedule generation, then the records the kernels read.
    OeOp* ops = reinterpret_cast<OeOp*>(host + batch->ops_at);
    int2* edge_offsets = reinterpret_cast<int2*>(host + batch->edge_offsets_at);
    batch->programs.assign(T, TreeProgram());
    std::vector<int> tree_slots(T, 1);
    std::vector<int64_t> post_doubles(T), full_doubles(T);
    ParallelOverTrees(T, [&](int t) {
      TreeProgram program = BuildTreeProgram(
          trees->parent_ids + static_cast<size_t>(t) * (trees->node_count - 1), trees->node_count, n);
      PackProgram(program, n, C, with_subst, ops + static_cast<size_t>(t) * 2 * (n - 1),
                  edge_offsets + static_cast<size_t>(t) * (2 * n - 2), &post_doubles[t], &full_doubles[t]);
      tree_slots[t] = std::max(program.post_slots, program.pre_slots);
      program.post.clear();
      program.post.shrink_to_fit();
      program.pre.clear();
      program.pre.shrink_to_fit();
      batch->programs[t] = std::move(program);
    });
    batch->slots = std::max(1, *std::max_element(tree_slots.begin(), tree_slots.end()));
    // (every bifurcating tree of n taxa has n-2 internal and n tip edges: one size)
    batch->post_doubles = post_doubles[0];
    batch->full_doubles = full_doubles[0];
    batch->cached_parent_ids.assign(trees->parent_ids, trees->parent_ids + id_count);
    batch->cached_input_nodes = trees->node_count;
    batch->cached_padded_categories = C;
    batch->cached_with_subst = with_subst;
    batch->cached_rooted_finish = batch->rooted_finish;
    if (batch->rooted_finish) {
      int32_t* children = reinterpret_cast<int32_t*>(host + batch->children_at);
      for (int t = 0; t < T; t++) {
        std::copy(batch->programs[t].child0.begin(), batch->programs[t].child0.end(), children + static_cast<size_t>(t) * 2 * N);
        std::copy(batch->programs[t].child1.begin(), batch->programs[t].child1.end(),
                  children + static_cast<size_t>(t) * 2 * N + N);
      }
    }
  }
  if (batch->rooted_finish) {
    double* fields = reinterpret_cast<double*>(host + batch->rooted_fields_at);
    for (int t = 0; t < T; t++) {
      double* row = fields + static_cast<size_t>(t) * rooted_stride;
      const RootedView view = ViewOf(trees, t, n);
      row = std::copy(view.rates, view.rates + (N - 1), row);
      row = std::copy(view.branch_lengths, view.branch_lengths + N, row);
      row = std::copy(view.node_heights, view.node_heights + N, row);
      row = std::copy(view.node_bounds, view.node_bounds + N, row);
      std::copy(view.height_ratios, view.height_ratios + (n - 1), row);
    }
  }
  for (int t = 0; t < T; t++)
    EffectiveBranchLengths(batch->programs[t], trees, t, rooted, batch->slide_root, N,
                           lengths + static_cast<size_t>(t) * N);
  batch->lengths.assign(lengths, lengths + static_cast<size_t>(T) * N);

  // Models: one table per distinct consecutive parameter row (+ its FD rows).
  size_t model_count = 0;
  const int K = spec.param_count;
  int previous_base_model = -1;
  std::vector<std::vector<double>> fd_rows;
  for (int t = 0; t < T; t++) {
    const double* row = params + static_cast<size_t>(t) * K;
    const bool same_as_previous =
        t > 0 && (K == 0 || std::memcmp(row, row - K, sizeof(double) * K) == 0);
    if (!same_as_previous) {
      previous_base_model = static_cast<int>(model_count);
      BuildModelTables(spec, row, &models[model_count++]);
      if (fd_evals) {
        FiniteDifferenceRows(spec, row, kFiniteDifferenceDelta, &fd_rows);
        for (const auto& fd_row : fd_rows) BuildModelTables(spec, fd_row.data(), &models[model_count++]);
      }
    }
    vtree_program[t] = t;
    vtree_model[t] = previous_base_model;
    vtree_lengths[t] = t;
    for (int f = 0; f < fd_evals; f++) {
      const int v = T + t * fd_evals + f;
      vtree_program[v] = t;
      vtree_model[v] = previous_base_model + 1 + f;
      vtree_lengths[v] = t;
    }
  }

  // One copy: the per-call part alone when the programs are already there.
  cudaStream_t s = e->stream;
  batch->input.Reserve(total_bytes);
  const size_t copy_from = cached ? per_call_begin : 0;
  SBNB_CUDA(cudaMemcpyAsync(batch->input.get() + copy_from, host + copy_from, total_bytes - copy_from,
                            cudaMemcpyHostToDevice, s));
  const size_t copy_bytes = total_bytes - copy_from;
  SBNB_CUDA(cudaEventRecord(e->staging_free, s));
  e->staging_in_flight = true;
  e->h2d_bytes += copy_bytes;
  batch->results.Reserve(batch->vtree_count + 2 * static_cast<size_t>(T) * N +
                         static_cast<size_t>(T) * (kOeSubstSums + kOeInvariantSums) + (batch->rooted_finish ? static_cast<size_t>(T) * batch->RootedWidth() : 0));
  if (batch->rooted_finish) batch->rooted_scratch.Reserve(static_cast<size_t>(T) * 5 * (n - 1));
  return batch;
}

// Folds one finished event pair into the running totals (waits for it).
void HarvestWalkTiming(sbnb_engine* e, int ring) {
  if (!e->walk_pending[ring]) return;
  SBNB_CUDA(cudaEventSynchronize(e->walk_end[ring]));
  float ms = 0.f;
  SBNB_CUDA(cudaEventElapsedTime(&ms, e->walk_begin[ring], e->walk_end[ring]));
  e->walk_total_ms += ms;
  e->walk_last_ms = ms;
  e->walk_samples++;
  e->walk_pending[ring] = false;
}

OeParams BaseParams(sbnb_engine* e, sbnb_batch* b) {
  OeParams p{};
  p.tips = e->tips.get();
  p.tip_pitch = e->tip_pitch;
  p.weights = e->weights.get();
  p.invariant_masks = e->spec.invariant ? e->invariant_masks.get() : nullptr;
  p.pattern_begin = 0;  // the device arrays start at the engine's pattern range
  p.pattern_end = e->range_end - e->range_begin;
  p.taxon_count = e->taxon_count;
  p.ops = b->At<OeOp>(b->ops_at);
  p.vtree_program = b->At<int32_t>(b->vtree_program_at);
  p.vtree_model = b->At<int32_t>(b->vtree_model_at);
  p.models = b->At<ModelTables>(b->models_at);
  p.slots = b->slots;
  return p;
}

// Transition matrices of virtual trees [begin, begin + count), written into the
// operand blocks of the ops that read them, and the block headers.
void LaunchMatrices(sbnb_engine* e, sbnb_batch* b, double* operands, int64_t stride, int begin, int count,
                    bool with_pre, bool with_subst = false) {
  const int n = e->taxon_count, C = e->padded_categories;
  OeMatrixParams m{};
  m.models = b->At<ModelTables>(b->models_at);
  m.vtree_model = b->At<int32_t>(b->vtree_model_at);
  m.vtree_lengths = b->At<int32_t>(b->vtree_lengths_at);
  m.vtree_program = b->At<int32_t>(b->vtree_program_at);
  m.branch_lengths = b->At<double>(b->lengths_at);
  m.edge_offsets = b->At<int2>(b->edge_offsets_at);
  m.ops = b->At<OeOp>(b->ops_at);
  m.operands = operands;
  m.operand_stride = stride;
  m.vtree_begin = begin;
  m.vtree_count = count;
  m.taxon_count = n;
  m.categories = C;
  m.with_pre = with_pre ? 1 : 0;
  m.with_subst = (with_pre && with_subst) ? 1 : 0;
  m.prefetch = OePrefetchOps(C);
  const int64_t jobs = static_cast<int64_t>(count) * (2 * n - 2) * C +
                       static_cast<int64_t>(count) * (with_pre ? 2 * (n - 1) : n - 1);
  const int block = 128;
  TransitionMatrixOeKernel<<<static_cast<int>((jobs + block - 1) / block), block, 0, e->stream>>>(m);
  SBNB_CUDA(cudaGetLastError());
  e->launch_count++;
}

void Run(sbnb_engine* e, sbnb_batch* b, int mode, bool rescaling, bool timed = true) {
  NvtxRange range("sbnb run");
  Require(mode == SBNB_MODE_LOG_LIKELIHOOD || mode == SBNB_MODE_BRANCH_GRADIENT, "Unknown mode.");
  SBNB_CUDA(cudaSetDevice(e->device));
  b->last_mode = mode;
  if (b->tree_count == 0) return;
  const bool grad = (mode == SBNB_MODE_BRANCH_GRADIENT);
  const int T = b->tree_count, N = b->node_count, C = e->padded_categories;
  cudaStream_t s = e->stream;
  const int vtrees = grad ? b->vtree_count : T;
  const int fd_vtrees = vtrees - T;

  // The finite-difference evaluations run in slices that share one operand buffer, so
  // that memory does not grow with 1 + 2 x coordinates (17 for GTR) times the batch.
  const int64_t slice_doubles = std::max<int64_t>(EnvInt("SBNB_FD_SLICE_MB", 1024), 1) * (1 << 20) / 8;
  const int slice = fd_vtrees > 0
                        ? static_cast<int>(std::max<int64_t>(1, std::min<int64_t>(fd_vtrees, slice_doubles / b->post_doubles)))
                        : 0;

  OeParams p = BaseParams(e, b);
  p.vtree_begin = 0;
  p.vtree_count = T;
  // (which walk is planned: the one with the substitution-gradient sums has its own occupancy)
  if (grad && b->with_subst) p.subst_partial = reinterpret_cast<double*>(1);
  LaunchPlan plan = Dispatch(e, p, grad, rescaling, /*launch=*/false, 0);
  LaunchPlan fd_plan{};
  if (fd_vtrees > 0) {
    OeParams q = p;
    q.vtree_begin = T;
    q.vtree_count = slice;
    q.subst_partial = nullptr;
    fd_plan = Dispatch(e, q, false, rescaling, false, 0);
  }
  // Partial-sum rows: [vtree][chunk][warp]; all launches share one chunk count so
  // that a single row stride addresses the buffers.  Every row is written by the warp
  // that owns it (no memset).
  const int chunks = std::max(plan.chunks, fd_vtrees > 0 ? fd_plan.chunks : 1);
  b->chunks = chunks;
  const size_t rows = static_cast<size_t>(vtrees) * chunks * kWarps;
  b->logl_partial.Reserve(rows);
  const bool subst = grad && b->with_subst;
  if (grad) {
    const size_t grad_rows = static_cast<size_t>(T) * chunks * kWarps * N;
    b->grad_partial.Reserve(grad_rows);
    if (C > 1) b->rgrad_partial.Reserve(grad_rows);
    if (subst) b->subst_partial.Reserve(static_cast<size_t>(T) * chunks * kWarps * kOeSubstSums);
    if (b->invariant) b->inv_partial.Reserve(static_cast<size_t>(T) * chunks * kWarps * kOeInvariantSums);
  }
  p.logl_partial = b->logl_partial.get();
  p.grad_partial = b->grad_partial.get();
  p.rgrad_partial = b->rgrad_partial.get();
  p.subst_partial = subst ? b->subst_partial.get() : nullptr;
  const bool inv = grad && b->invariant;
  p.inv_partial = inv ? b->inv_partial.get() : nullptr;

  // Base trees: matrices, then the logL or gradient sweep.
  b->operand_stride = grad ? b->full_doubles : b->post_doubles;
  b->operands.Reserve(static_cast<size_t>(T) * b->operand_stride);
  LaunchMatrices(e, b, b->operands.get(), b->operand_stride, 0, T, grad, b->with_subst);
  p.operands = b->operands.get();
  p.operand_origin = 0;
  p.operand_stride = b->operand_stride;
  if (timed) {
    const int ring = static_cast<int>(e->walk_runs++ % sbnb_engine::kWalkRing);
    HarvestWalkTiming(e, ring);  // the slot about to be reused
    SBNB_CUDA(cudaEventRecord(e->walk_begin[ring], s));
    Dispatch(e, p, grad, rescaling, /*launch=*/true, chunks);
    SBNB_CUDA(cudaEventRecord(e->walk_end[ring], s));
    e->walk_pending[ring] = true;
  } else {
    Dispatch(e, p, grad, rescaling, /*launch=*/true, chunks);
  }

  if (fd_vtrees > 0) {
    e->fd_operands.Reserve(static_cast<size_t>(slice) * b->post_doubles);
    for (int begin = T; begin < vtrees; begin += slice) {
      const int count = std::min(slice, vtrees - begin);
      LaunchMatrices(e, b, e->fd_operands.get(), b->post_doubles, begin, count, false);
      OeParams q = p;
      q.vtree_begin = begin;
      q.vtree_count = count;
      q.operands = e->fd_operands.get();
      q.operand_origin = begin;
      q.operand_stride = b->post_doubles;
      Dispatch(e, q, false, rescaling, true, chunks);
    }
  }

  // Fixed-order reduction of the per-(chunk, warp) partial sums, all arrays at once.
  {
    const int64_t total = vtrees + (grad ? 2 * static_cast<int64_t>(T) * N : 0) +
                          ((subst || inv) ? static_cast<int64_t>(T) * kOeSubstSums : 0) +
                          (inv ? static_cast<int64_t>(T) * kOeInvariantSums : 0);
    const int block = 128;
    ReduceAllKernel<<<static_cast<int>((total + block - 1) / block), block, 0, s>>>(
        b->logl_partial.get(), b->grad_partial.get(), (grad && C > 1) ? b->rgrad_partial.get() : nullptr,
        subst ? b->subst_partial.get() : nullptr, b->results.get(), 0, vtrees, b->vtree_count, grad ? T : 0, N,
        chunks * kWarps, inv ? b->inv_partial.get() : nullptr);
    SBNB_CUDA(cudaGetLastError());
    e->launch_count++;
  }
  if (grad && b->rooted_finish) {
    RootedFinishParams r{};
    r.tree_count = T;
    r.taxon_count = b->taxon_count;
    r.rate_count = b->rate_count;
    r.children = b->At<int32_t>(b->children_at);
    r.fields = b->At<double>(b->rooted_fields_at);
    r.scaled_lengths = b->At<double>(b->lengths_at);
    r.grad = b->ResultGrad();
    r.rgrad = C > 1 ? b->ResultRateGrad() : nullptr;
    r.scratch = b->rooted_scratch.get();
    r.out = b->ResultRooted();
    if (inv) {
      r.inv_sums = b->ResultInvariant();
      r.models = b->At<ModelTables>(b->models_at);
      r.vtree_model = b->At<int32_t>(b->vtree_model_at);
      r.site_width = b->site_width;
    }
    const int block = 64;
    RootedFinishKernel<<<(T + block - 1) / block, block, 0, s>>>(r);
    SBNB_CUDA(cudaGetLastError());
    e->launch_count++;
  }
}

// How many doubles of the result array a fetch of these outputs copies.
size_t FetchCount(const sbnb_engine* e, const sbnb_batch* b, bool grad, bool rgrad, bool subst,
                  bool rooted = false, bool inv = false) {
  const bool was_grad = (b->last_mode == SBNB_MODE_BRANCH_GRADIENT);
  const size_t vtrees = was_grad ? b->vtree_count : b->tree_count;
  const size_t grad_count = static_cast<size_t>(b->tree_count) * b->node_count;
  const bool rates = rgrad && e->padded_categories > 1;
  if (rooted)
    return b->vtree_count + 2 * grad_count +
           static_cast<size_t>(b->tree_count) * (kOeSubstSums + kOeInvariantSums + b->RootedWidth());
  if (inv)
    return b->vtree_count + 2 * grad_count + static_cast<size_t>(b->tree_count) * (kOeSubstSums + kOeInvariantSums);
  if (subst) return b->vtree_count + 2 * grad_count + static_cast<size_t>(b->tree_count) * kOeSubstSums;
  return (grad || rates) ? b->vtree_count + (rates ? 2 : 1) * grad_count : vtrees;
}

// Results that have landed in page-locked memory -> the caller's arrays.
void Unpack(const sbnb_engine* e, const sbnb_batch* b, const double* landed, double* logl, double* grad,
            double* rgrad, double* subst, double* rooted = nullptr, double* inv = nullptr) {
  const bool was_grad = (b->last_mode == SBNB_MODE_BRANCH_GRADIENT);
  const size_t vtrees = was_grad ? b->vtree_count : b->tree_count;
  const size_t grad_count = static_cast<size_t>(b->tree_count) * b->node_count;
  if (logl) std::copy(landed, landed + vtrees, logl);
  if (grad) std::copy(landed + b->vtree_count, landed + b->vtree_count + grad_count, grad);
  if (rgrad) {
    if (e->padded_categories > 1) {
      std::copy(landed + b->vtree_count + grad_count, landed + b->vtree_count + 2 * grad_count, rgrad);
    } else {
      std::fill(rgrad, rgrad + grad_count, 0.0);
    }
  }
  const size_t subst_count = static_cast<size_t>(b->tree_count) * kOeSubstSums;
  if (subst) std::copy(landed + b->vtree_count + 2 * grad_count, landed + b->vtree_count + 2 * grad_count + subst_count, subst);
  const size_t inv_count = static_cast<size_t>(b->tree_count) * kOeInvariantSums;
  if (inv) std::copy(landed + b->vtree_count + 2 * grad_count + subst_count,
                     landed + b->vtree_count + 2 * grad_count + subst_count + inv_count, inv);
  if (rooted) {
    const double* from = landed + b->vtree_count + 2 * grad_count + subst_count + inv_count;
    std::copy(from, from + static_cast<size_t>(b->tree_count) * b->RootedWidth(), rooted);
  }
}

void Fetch(sbnb_engine* e, sbnb_batch* b, double* logl, double* grad, double* rgrad, double* subst = nullptr,
           double* rooted = nullptr, double* inv = nullptr) {
  NvtxRange range("sbnb fetch");
  SBNB_CUDA(cudaSetDevice(e->device));
  Require(b->last_mode >= 0, "sbnb_batch_fetch called before sbnb_batch_run.");
  const bool was_grad = (b->last_mode == SBNB_MODE_BRANCH_GRADIENT);
  Require(was_grad || (!grad && !rgrad), "No gradient available: the last run was a log-likelihood run.");
  if (subst) Require(was_grad && b->with_subst, "No substitution-gradient sums: the batch was not staged for them.");
  if (inv) Require(was_grad && b->invariant, "No invariable-site sums: the last run was not a gradient run of a +I model.");
  cudaStream_t s = e->stream;
  if (b->tree_count == 0) {
    SBNB_CUDA(cudaStreamSynchronize(s));
    return;
  }
  // One copy of what is asked for into page-locked memory, then out to the caller's arrays.
  if (rooted) Require(was_grad && b->rooted_finish, "No finished rooted gradients: the batch carries no time-tree fields.");
  const size_t count =
      FetchCount(e, b, grad != nullptr, rgrad != nullptr, subst != nullptr, rooted != nullptr, inv != nullptr);
  e->landing.Reset(count * sizeof(double));
  double* landed = e->landing.Take<double>(count);
  SBNB_CUDA(cudaMemcpyAsync(landed, b->results.get(), count * sizeof(double), cudaMemcpyDeviceToHost, s));
  e->d2h_bytes += count * sizeof(double);
  SBNB_CUDA(cudaStreamSynchronize(s));
  Unpack(e, b, landed, logl, grad, rgrad, subst, rooted, inv);
}

// Run + Fetch of the one-call entry points.  Once the same topology set has come in
// three times in a row (programs cached on the device, the same sequence run eagerly once), the launch
// sequence is captured into a CUDA graph and replayed: one launch call instead of
// 4-6 launches, 2 event records and a copy (the small-problem regime of
// BASELINE.json configs[0..1], where a call is tens of microseconds).
void RunAndFetch(sbnb_engine* e, sbnb_batch* b, int mode, bool rescaling, double* logl, double* grad,
                 double* rgrad, double* subst = nullptr, double* rooted = nullptr, double* inv = nullptr) {
  static const bool graphs_enabled = EnvInt("SBNB_GRAPHS", 1) != 0;
  sbnb_batch::Graph& graph = b->graphs[mode == SBNB_MODE_BRANCH_GRADIENT ? 1 : 0][rescaling ? 1 : 0];
  if (!graphs_enabled || b->tree_count == 0 || b->cache_hits < 1 || !graph.warm) {
    Run(e, b, mode, rescaling);
    Fetch(e, b, logl, grad, rgrad, subst, rooted, inv);
    graph.warm = b->cache_hits >= 1;  // (an eager run on cached programs: the next one may be captured)
    return;
  }
  SBNB_CUDA(cudaSetDevice(e->device));
  cudaStream_t s = e->stream;
  b->last_mode = mode;
  const size_t count =
      FetchCount(e, b, grad != nullptr, rgrad != nullptr, subst != nullptr, rooted != nullptr, inv != nullptr);
  e->landing.Reset(count * sizeof(double));
  double* landed = e->landing.Take<double>(count);
  auto signature = [&] {
    return std::vector<uintptr_t>{
        reinterpret_cast<uintptr_t>(b->input.get()),        reinterpret_cast<uintptr_t>(b->operands.get()),
        reinterpret_cast<uintptr_t>(b->results.get()),      reinterpret_cast<uintptr_t>(b->logl_partial.get()),
        reinterpret_cast<uintptr_t>(b->grad_partial.get()), reinterpret_cast<uintptr_t>(b->rgrad_partial.get()),
        reinterpret_cast<uintptr_t>(b->subst_partial.get()), reinterpret_cast<uintptr_t>(e->stack.get()),
        reinterpret_cast<uintptr_t>(e->stack_exps.get()),   reinterpret_cast<uintptr_t>(e->arena.get()),
        reinterpret_cast<uintptr_t>(e->fd_operands.get()),  reinterpret_cast<uintptr_t>(e->tips.get()),
        reinterpret_cast<uintptr_t>(e->weights.get()),      reinterpret_cast<uintptr_t>(landed),
        static_cast<uintptr_t>(count),                      static_cast<uintptr_t>(b->vtree_count),
        static_cast<uintptr_t>(b->with_subst),              static_cast<uintptr_t>(e->range_end - e->range_begin),
        static_cast<uintptr_t>(b->slots),                   reinterpret_cast<uintptr_t>(b->rooted_scratch.get()),
        reinterpret_cast<uintptr_t>(b->inv_partial.get()),  reinterpret_cast<uintptr_t>(e->invariant_masks.get())};
  };
  if (graph.exec == nullptr || graph.signature != signature()) {
    if (graph.exec) {
      cudaGraphExecDestroy(graph.exec);
      graph.exec = nullptr;
    }
    // (the previous two calls ran this very sequence: every buffer has its size, so
    //  nothing below allocates while the stream is capturing)
    const int64_t launches_before = e->launch_count;
    SBNB_CUDA(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
    cudaGraph_t recorded = nullptr;
    try {
      Run(e, b, mode, rescaling, /*timed=*/false);
      SBNB_CUDA(cudaMemcpyAsync(landed, b->results.get(), count * sizeof(double), cudaMemcpyDeviceToHost, s));
    } catch (...) {
      cudaStreamEndCapture(s, &recorded);
      if (recorded) cudaGraphDestroy(recorded);
      throw;
    }
    SBNB_CUDA(cudaStreamEndCapture(s, &recorded));
    graph.kernels = static_cast<int>(e->launch_count - launches_before);
    e->launch_count = launches_before;
    const cudaError_t status = cudaGraphInstantiate(&graph.exec, recorded, 0);
    cudaGraphDestroy(recorded);
    SBNB_CUDA(status);
    graph.signature = signature();  // (the capture itself may have moved nothing; taken after it on purpose)
  }
  SBNB_CUDA(cudaGraphLaunch(graph.exec, s));
  e->launch_count += graph.kernels;
  e->d2h_bytes += count * sizeof(double);
  SBNB_CUDA(cudaStreamSynchronize(s));
  Unpack(e, b, landed, logl, grad, rgrad, subst, rooted, inv);
}

RootedView ViewOf(const sbnb_tree_batch* trees, int t, int n) {
  const int N = 2 * n - 1;
  RootedView view{};
  view.branch_lengths = trees->branch_lengths + static_cast<size_t>(t) * N;
  view.rates = trees->rates + static_cast<size_t>(t) * (N - 1);
  view.node_heights = trees->node_heights ? trees->node_heights + static_cast<size_t>(t) * N : nullptr;
  view.node_bounds = trees->node_bounds ? trees->node_bounds + static_cast<size_t>(t) * N : nullptr;
  view.height_ratios =
      trees->height_ratios ? trees->height_ratios + static_cast<size_t>(t) * (n - 1) : nullptr;
  view.rate_count = trees->rate_count;
  return view;
}

// The tip codes of an alignment (walk_oe.cuh): states 0..3 stay, anything >= 4 is the gap
// code 4; nucleotide masks become codes 0..14, and 0 or > 15 is refused.
std::shared_ptr<const std::vector<uint8_t>> TipCodes(int32_t taxon_count, int64_t pattern_count,
                                                     const uint8_t* tips, int32_t encoding, bool* ambiguous) {
  auto codes = std::make_shared<std::vector<uint8_t>>(static_cast<size_t>(taxon_count) * pattern_count);
  *ambiguous = false;
  if (encoding == SBNB_TIPS_STATES) {
    for (size_t i = 0; i < codes->size(); i++) (*codes)[i] = tips[i] < 4 ? tips[i] : 4;
    return codes;
  }
  uint8_t code_of[16] = {};
  for (int code = 0; code < kTipCodes; code++) code_of[TipCodeMask(code)] = static_cast<uint8_t>(code);
  for (size_t i = 0; i < codes->size(); i++) {
    const uint8_t mask = tips[i];
    if (mask == 0 || mask > 15)
      Fail(SBNB_ERR_INVALID_ARGUMENT, "Invalid nucleotide mask " + std::to_string(mask) + " at taxon " +
                                          std::to_string(i / pattern_count) + ", pattern " +
                                          std::to_string(i % pattern_count) + " (masks are 1..15).");
    (*codes)[i] = code_of[mask];
    *ambiguous = *ambiguous || code_of[mask] >= kFirstAmbiguousCode;
  }
  return codes;
}

// Engine::Engine + FatBeagle::FatBeagle for one device.  `sibling` (a child of the same
// device group) shares its host copy of the alignment.
std::unique_ptr<sbnb_engine> CreateEngine(const char* substitution, const char* site, const char* clock,
                                          int32_t taxon_count, int64_t pattern_count, const uint8_t* tips,
                                          int32_t tip_encoding, const double* pattern_weights, int32_t device,
                                          const sbnb_engine* sibling) {
  Require(substitution && site && clock, "NULL model specification string.");
  Require(taxon_count >= 2, "Need at least 2 taxa.");
  Require(pattern_count >= 1, "Need at least 1 site pattern.");
  Require(tips && pattern_weights, "NULL tip_states / pattern_weights.");
  Require(tip_encoding == SBNB_TIPS_STATES || tip_encoding == SBNB_TIPS_NUCLEOTIDE_MASKS, "Unknown tip encoding.");
  auto engine = std::make_unique<sbnb_engine>();
  engine->spec = ModelSpec::Parse(substitution, site, clock);
  int device_count = 0;
  if (cudaGetDeviceCount(&device_count) != cudaSuccess || device_count < 1) {
    cudaGetLastError();
    Fail(SBNB_ERR_NO_DEVICE, "No CUDA device available: libsbn_b200 has no CPU fallback (cudaGetDeviceCount).");
  }
  Require(device >= 0 && device < device_count, "CUDA device ordinal out of range.");
  SBNB_CUDA(cudaSetDevice(device));
  engine->device = device;
  int sm_count = 0;
  SBNB_CUDA(cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, device));
  engine->sm_count = sm_count;
  engine->taxon_count = taxon_count;
  engine->pattern_count = pattern_count;
  engine->range_begin = 0;
  engine->range_end = pattern_count;
  engine->categories = engine->spec.category_count;
  engine->padded_categories = PadCategories(engine->categories);
  Require(engine->padded_categories > 0,
          "At most 32 rate categories are supported by the fused tree walk (libhmsbeagle_b200.so, the "
          "BEAGLE-compatible device library behind the unmodified FatBeagle, takes any number).");
  SBNB_CUDA(cudaStreamCreateWithFlags(&engine->stream, cudaStreamNonBlocking));
  SBNB_CUDA(cudaEventCreateWithFlags(&engine->staging_free, cudaEventDisableTiming));
  for (int i = 0; i < sbnb_engine::kWalkRing; i++) {
    SBNB_CUDA(cudaEventCreate(&engine->walk_begin[i]));
    SBNB_CUDA(cudaEventCreate(&engine->walk_end[i]));
  }
  if (sibling) {
    engine->host_tips = sibling->host_tips;
    engine->ambiguous = sibling->ambiguous;
    engine->host_weights = sibling->host_weights;
  } else {
    engine->host_tips = TipCodes(taxon_count, pattern_count, tips, tip_encoding, &engine->ambiguous);
    engine->host_weights = std::make_shared<std::vector<double>>(pattern_weights, pattern_weights + pattern_count);
  }
  if (const char* mode = std::getenv("SBNB_SUBSTITUTION_GRADIENT"))
    engine->substitution_mode = std::string(mode) == "fd" ? SBNB_SUBSTITUTION_FINITE_DIFFERENCES
                                                           : SBNB_SUBSTITUTION_ANALYTIC;
  UploadPatternRange(engine.get(), 0, pattern_count);
  return engine;
}

// The one-call forms of Engine's five methods.
void LogLikelihoods(sbnb_engine* e, const sbnb_tree_batch* trees, const double* params,
                    bool rescaling, bool rooted_semantics, bool add_jacobian, double* out) {
  Require(trees != nullptr, "NULL tree batch.");
  Require(out != nullptr || trees->tree_count == 0, "NULL output.");
  auto batch = Stage(e, trees, params, rooted_semantics, false, /*slide_root=*/false);
  RunAndFetch(e, batch.get(), SBNB_MODE_LOG_LIKELIHOOD, rescaling, out, nullptr, nullptr);
  if (add_jacobian) {
    Require(trees->tree_count == 0 || (trees->node_heights && trees->node_bounds),
            "Rooted log likelihoods need node_heights and node_bounds.");
    for (int t = 0; t < trees->tree_count; t++)
      out[t] += LogDetJacobianHeightRatios(batch->programs[t], ViewOf(trees, t, e->taxon_count));
  }
}

// Host finishing of a gradient evaluation (the O(n) tail of FatBeagle::Gradient,
// fat_beagle.cpp:467-545) from the raw per-tree sums over site patterns:
// logl[T (+ T * 2 * fd_coords)], grad[T][N] edge derivatives, rgrad[T][N] the same
// with d rate_c / d shape as scalers.  Needs no device: every input is a sum over
// patterns, so under site-pattern sharding the ranks all-reduce the raw sums
// and each runs this once.
void FinishGradients(const ModelSpec& spec, int n, const sbnb_tree_batch* trees, bool rooted, int fd_coords,
                     const double* logl, const double* grad, const double* rgrad,
                     const sbnb_gradient_out* out, const std::vector<TreeProgram>* programs = nullptr,
                     const double* params = nullptr, const double* subst_sums = nullptr,
                     const double* rooted_finished = nullptr, size_t rooted_width = 0,
                     const double* inv_sums = nullptr) {
  NvtxRange range("sbnb finish gradients");
  Require(trees != nullptr, "NULL tree batch.");
  Require(out != nullptr, "NULL gradient output.");
  const int T = trees->tree_count, N = 2 * n - 1;
  if (rooted)
    Require(T == 0 || (trees->node_heights && trees->node_bounds && trees->height_ratios),
            "Rooted gradients need node_heights, node_bounds and height_ratios.");
  const int categories = spec.category_count;
  // +I: the site-model row is [shape (if any) | proportion invariant]
  const int site_width = spec.SiteGradientSize();
  if (spec.invariant) Require(T == 0 || (params && inv_sums), "A +I site model needs the parameters and the +I sums.");
  ParallelOverTrees(T, [&](int t) {
    std::vector<double> g(N), lengths(N);
    TreeProgram rebuilt;
    if (!programs)
      rebuilt = BuildTreeProgram(trees->parent_ids + static_cast<size_t>(t) * (trees->node_count - 1),
                                 trees->node_count, n);
    const TreeProgram& tree = programs ? (*programs)[t] : rebuilt;
    std::copy(grad + static_cast<size_t>(t) * N, grad + static_cast<size_t>(t + 1) * N, g.begin());
    if (out->log_likelihood) out->log_likelihood[t] = logl[t];
    if (out->substitution_model && fd_coords > 0) {
      // Central differences; the rooted Jacobian term cancels (fat_beagle.cpp:431).
      const double* fd = logl + T + static_cast<size_t>(t) * 2 * fd_coords;
      for (int k = 0; k < fd_coords; k++)
        out->substitution_model[static_cast<size_t>(t) * fd_coords + k] =
            (fd[2 * k] - fd[2 * k + 1]) / (2. * kFiniteDifferenceDelta);
    }
    if (out->substitution_model && subst_sums != nullptr) {
      // Analytic: d logL / d theta = < W, B_theta > + d pi / d theta . R (model.hpp).
      const double* row = params + static_cast<size_t>(t) * spec.param_count;
      ModelTables tables;
      BuildModelTables(spec, row, &tables);
      SubstitutionDerivatives derivatives;
      BuildSubstitutionDerivatives(spec, row, tables, &derivatives);
      const double* sums = subst_sums + static_cast<size_t>(t) * kOeSubstSums;
      double r[4];
      for (int j = 0; j < 4; j++) r[j] = sums[16 + j];
      // +I: the invariant class adds pinv E_s to R_s (0 at pinv = 0, where E may be infinite)
      if (spec.invariant && tables.pinv != 0.0)
        for (int j = 0; j < 4; j++) r[j] += tables.pinv * inv_sums[static_cast<size_t>(t) * kOeInvariantSums + 1 + j];
      for (int k = 0; k < derivatives.count; k++) {
        double value = 0.0;
        for (int e = 0; e < 16; e++) value += sums[e] * derivatives.b[k][e];
        for (int j = 0; j < 4; j++) value += r[j] * derivatives.dfreqs[k][j];
        out->substitution_model[static_cast<size_t>(t) * derivatives.count + k] = value;
      }
    }
    if (rooted && rooted_finished != nullptr) {
      // RootedFinishKernel has done the O(n) tail on the device: [ratios | clock | site model]
      const double* row = rooted_finished + static_cast<size_t>(t) * rooted_width;
      if (out->ratios_root_height) std::copy(row, row + (n - 1), out->ratios_root_height + static_cast<size_t>(t) * (n - 1));
      if (out->clock_model)
        std::copy(row + (n - 1), row + (n - 1) + trees->rate_count,
                  out->clock_model + static_cast<size_t>(t) * trees->rate_count);
      if (out->site_model && spec.invariant) {
        std::copy(row + (rooted_width - site_width), row + rooted_width, out->site_model + static_cast<size_t>(t) * site_width);
      } else if (out->site_model && categories > 1) {
        out->site_model[t] = row[rooted_width - 1];
      }
      return;
    }
    if (out->site_model && (categories > 1 || spec.invariant)) {
      EffectiveBranchLengths(tree, trees, t, rooted, /*slide_root=*/true, N, lengths.data());
      double* site = out->site_model + static_cast<size_t>(t) * site_width;
      if (categories > 1)
        site[0] = DiscreteSiteModelGradient(N, lengths.data(), rgrad + static_cast<size_t>(t) * N);  // fat_beagle.cpp:389-398
      if (spec.invariant) {
        // d logL / d pinv = D + sum over edges of tau g / (1 - pinv): the rates are divided by 1 - pinv
        const double pinv = params[static_cast<size_t>(t) * spec.param_count + spec.Block("proportion invariant").first];
        site[site_width - 1] = inv_sums[static_cast<size_t>(t) * kOeInvariantSums] +
                               DiscreteSiteModelGradient(N, lengths.data(), g.data()) / (1.0 - pinv);
      }
    }
    if (rooted) {
      const RootedView view = ViewOf(trees, t, n);
      if (out->ratios_root_height) {
        const std::vector<double> ratios = RatioGradientOfBranchGradient(tree, view, g.data());
        std::copy(ratios.begin(), ratios.end(), out->ratios_root_height + static_cast<size_t>(t) * (n - 1));
      }
      if (out->clock_model) {
        const std::vector<double> clock = ClockGradient(tree, view, g.data());
        std::copy(clock.begin(), clock.end(), out->clock_model + static_cast<size_t>(t) * view.rate_count);
      }
    } else if (out->branch_lengths) {
      // "We want the fixed node to have a zero gradient" (fat_beagle.cpp:498-500).
      g[tree.child1[tree.root]] = 0.0;
      std::copy(g.begin(), g.end(), out->branch_lengths + static_cast<size_t>(t) * N);
    }
  });
}

void Gradients(sbnb_engine* e, const sbnb_tree_batch* trees, const double* params, bool rescaling,
               bool rooted, const sbnb_gradient_out* out) {
  Require(out != nullptr, "NULL gradient output.");
  Require(trees != nullptr, "NULL tree batch.");
  const int coords = e->spec.SubstitutionGradientSize();
  const bool wanted = coords > 0 && out->substitution_model != nullptr;
  const bool analytic = wanted && e->substitution_mode == SBNB_SUBSTITUTION_ANALYTIC;
  auto batch = Stage(e, trees, params, rooted, wanted && !analytic, /*slide_root=*/true, analytic);
  const int T = trees->tree_count, N = 2 * e->taxon_count - 1;
  const bool finished_on_device = batch->rooted_finish && T > 0;
  const bool inv = e->spec.invariant && T > 0;
  std::vector<double> logl(batch->vtree_count), grad(static_cast<size_t>(T) * N),
      rgrad(static_cast<size_t>(T) * N), subst((analytic || finished_on_device) ? static_cast<size_t>(T) * kOeSubstSums : 0),
      finished(finished_on_device ? static_cast<size_t>(T) * batch->RootedWidth() : 0),
      inv_sums(inv ? static_cast<size_t>(T) * kOeInvariantSums : 0);
  RunAndFetch(e, batch.get(), SBNB_MODE_BRANCH_GRADIENT, rescaling, logl.data(), grad.data(), rgrad.data(),
              analytic && T > 0 ? subst.data() : nullptr, finished_on_device ? finished.data() : nullptr,
              inv ? inv_sums.data() : nullptr);
  FinishGradients(e->spec, e->taxon_count, trees, rooted, batch->fd_coords, logl.data(), grad.data(),
                  rgrad.data(), out, &batch->programs, params, analytic && T > 0 ? subst.data() : nullptr,
                  finished_on_device ? finished.data() : nullptr, finished_on_device ? batch->RootedWidth() : 0,
                  inv ? inv_sums.data() : nullptr);
}


// ---------------------------------------------------------------------------
// Device groups (sbnb_engine_create_multi): the reference's Engine owns
// thread_count FatBeagles and fans a collection over them (engine.cpp:23-27,
// fat_beagle.hpp:119-149); here a group owns one child engine per GPU, one host
// thread + stream each, and the two shard axes of SURVEY.md 8e:
//   trees    -- child g evaluates a contiguous slice of the collection and writes its
//               rows of the caller's output arrays; no exchange step.
//   patterns -- every child walks ALL trees over its range of site patterns; the raw
//               per-tree sums (log-likelihoods, edge derivatives) of children 1.. are
//               added onto child 0's result array by PeerSumKernel, which reads the
//               peers' device memory directly over NVLink (or staged peer copies when
//               peer access is unavailable), in a fixed order; then one fetch and one
//               host finishing.

// One host thread per child; the first failure is rethrown on the calling thread.
template <typename F>
void ParallelOverChildren(sbnb_engine* group, F&& body) {
  const int G = static_cast<int>(group->children.size());
  std::vector<std::thread> threads;
  std::exception_ptr failure;
  std::mutex failure_mutex;
  for (int g = 0; g < G; g++) {
    threads.emplace_back([&, g] {
      try {
        FloatingPointEnvironmentKeeper keep_environment;
        body(g, group->children[g]);
      } catch (...) {
        std::lock_guard<std::mutex> lock(failure_mutex);
        if (!failure) failure = std::current_exception();
      }
    });
  }
  for (auto& thread : threads) thread.join();
  if (failure) std::rethrow_exception(failure);
}

// The trees [begin, end) of a batch as a batch of their own.
sbnb_tree_batch SliceTrees(const sbnb_tree_batch* trees, int n, int begin, int end) {
  sbnb_tree_batch slice = *trees;
  slice.tree_count = end - begin;
  const size_t nodes = trees->node_count;
  auto advance = [begin](const auto* base, size_t stride) { return base ? base + begin * stride : base; };
  slice.parent_ids = advance(trees->parent_ids, nodes - 1);
  slice.branch_lengths = advance(trees->branch_lengths, nodes);
  slice.rates = advance(trees->rates, nodes - 1);
  slice.node_heights = advance(trees->node_heights, nodes);
  slice.node_bounds = advance(trees->node_bounds, nodes);
  slice.height_ratios = advance(trees->height_ratios, static_cast<size_t>(n - 1));
  return slice;
}

// Pattern axis: stage + run on every child, sum the raw results onto child 0.
// Returns child 0's batch (results complete once its stream has been synchronised).
std::vector<BatchPtr> RunOverPatternShards(sbnb_engine* group, const sbnb_tree_batch* trees, const double* params,
                                           bool rooted, bool with_fd, bool slide_root, int mode, bool rescaling,
                                           bool with_subst = false) {
  const int G = static_cast<int>(group->children.size());
  std::vector<BatchPtr> batches;
  for (int g = 0; g < G; g++) batches.emplace_back(nullptr, BatchRecycler{group->children[g]});
  std::vector<cudaEvent_t> done(G, nullptr);
  ParallelOverChildren(group, [&](int g, sbnb_engine* child) {
    batches[g] = Stage(child, trees, params, rooted, with_fd, slide_root, with_subst);
    Run(child, batches[g].get(), mode, rescaling);
    if (g > 0) {
      SBNB_CUDA(cudaEventCreateWithFlags(&done[g], cudaEventDisableTiming));
      SBNB_CUDA(cudaEventRecord(done[g], child->stream));
    }
  });
  sbnb_engine* first = group->children[0];
  sbnb_batch* b0 = batches[0].get();
  if (trees->tree_count > 0 && G > 1) {
    SBNB_CUDA(cudaSetDevice(first->device));
    const bool grad = (mode == SBNB_MODE_BRANCH_GRADIENT);
    const int64_t edges = static_cast<int64_t>(b0->tree_count) * b0->node_count;
    const int64_t count =
        !grad ? b0->tree_count
              : (b0->invariant ? b0->vtree_count + 2 * edges + b0->tree_count * (kOeSubstSums + kOeInvariantSums)
                 : with_subst  ? b0->vtree_count + 2 * edges + b0->tree_count * kOeSubstSums
                               : b0->vtree_count + (first->padded_categories > 1 ? 2 : 1) * edges);
    PeerPointers peers{};
    peers.part[0] = b0->results.get();
    for (int g = 1; g < G; g++) {
      sbnb_engine* child = group->children[g];
      SBNB_CUDA(cudaStreamWaitEvent(first->stream, done[g], 0));
      int can_access = (child->device == first->device) ? 1 : 0;
      if (!can_access) {
        SBNB_CUDA(cudaDeviceCanAccessPeer(&can_access, first->device, child->device));
        if (can_access) {
          const cudaError_t status = cudaDeviceEnablePeerAccess(child->device, 0);
          if (status == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
          else if (status != cudaSuccess) can_access = 0, cudaGetLastError();
        }
      }
      if (can_access) {
        peers.part[g] = batches[g]->results.get();  // read in place, over NVLink
      } else {
        first->fd_operands.Reserve(static_cast<size_t>(count) * G);  // (free between runs) staging for peer copies
        double* staged = first->fd_operands.get() + static_cast<size_t>(count) * g;
        SBNB_CUDA(cudaMemcpyPeerAsync(staged, first->device, batches[g]->results.get(), child->device,
                                      count * sizeof(double), first->stream));
        peers.part[g] = staged;
      }
    }
    const int block = 256;
    PeerSumKernel<<<static_cast<int>((count + block - 1) / block), block, 0, first->stream>>>(
        b0->results.get(), peers, G, count);
    SBNB_CUDA(cudaGetLastError());
    first->launch_count++;
  }
  // The children's result arrays must outlive the sum: wait for it here.
  SBNB_CUDA(cudaSetDevice(first->device));
  SBNB_CUDA(cudaStreamSynchronize(first->stream));
  for (int g = 1; g < G; g++)
    if (done[g]) cudaEventDestroy(done[g]);
  return batches;
}

void GroupLogLikelihoods(sbnb_engine* group, const sbnb_tree_batch* trees, const double* params, bool rescaling,
                         bool rooted_semantics, bool add_jacobian, double* out) {
  Require(trees != nullptr, "NULL tree batch.");
  Require(out != nullptr || trees->tree_count == 0, "NULL output.");
  const int G = static_cast<int>(group->children.size()), T = trees->tree_count, n = group->taxon_count;
  const int K = group->spec.param_count;
  if (group->shard_axis == SBNB_SHARD_TREES) {
    ParallelOverChildren(group, [&](int g, sbnb_engine* child) {
      const int begin = static_cast<int>(static_cast<int64_t>(T) * g / G);
      const int end = static_cast<int>(static_cast<int64_t>(T) * (g + 1) / G);
      if (begin == end) return;
      const sbnb_tree_batch slice = SliceTrees(trees, n, begin, end);
      LogLikelihoods(child, &slice, params ? params + static_cast<size_t>(begin) * K : nullptr, rescaling,
                     rooted_semantics, add_jacobian, out + begin);
    });
    return;
  }
  auto batches = RunOverPatternShards(group, trees, params, rooted_semantics, false, false,
                                      SBNB_MODE_LOG_LIKELIHOOD, rescaling);
  Fetch(group->children[0], batches[0].get(), out, nullptr, nullptr);
  if (add_jacobian) {
    Require(T == 0 || (trees->node_heights && trees->node_bounds),
            "Rooted log likelihoods need node_heights and node_bounds.");
    for (int t = 0; t < T; t++) out[t] += LogDetJacobianHeightRatios(batches[0]->programs[t], ViewOf(trees, t, n));
  }
}

void GroupGradients(sbnb_engine* group, const sbnb_tree_batch* trees, const double* params, bool rescaling,
                    bool rooted, const sbnb_gradient_out* out) {
  Require(out != nullptr, "NULL gradient output.");
  Require(trees != nullptr, "NULL tree batch.");
  const int G = static_cast<int>(group->children.size()), T = trees->tree_count, n = group->taxon_count;
  const int N = 2 * n - 1, K = group->spec.param_count;
  const int fd_coords = group->spec.SubstitutionGradientSize();
  const bool wanted = fd_coords > 0 && out->substitution_model != nullptr;
  const bool analytic = wanted && group->substitution_mode == SBNB_SUBSTITUTION_ANALYTIC;
  if (group->shard_axis == SBNB_SHARD_TREES) {
    ParallelOverChildren(group, [&](int g, sbnb_engine* child) {
      const int begin = static_cast<int>(static_cast<int64_t>(T) * g / G);
      const int end = static_cast<int>(static_cast<int64_t>(T) * (g + 1) / G);
      if (begin == end) return;
      const sbnb_tree_batch slice = SliceTrees(trees, n, begin, end);
      sbnb_gradient_out rows = *out;
      auto advance = [begin](double* base, size_t width) { return base ? base + begin * width : base; };
      rows.log_likelihood = advance(out->log_likelihood, 1);
      rows.branch_lengths = advance(out->branch_lengths, N);
      rows.substitution_model = advance(out->substitution_model, fd_coords);
      rows.site_model = advance(out->site_model, group->spec.SiteGradientSize());
      rows.ratios_root_height = advance(out->ratios_root_height, n - 1);
      rows.clock_model = advance(out->clock_model, std::max(trees->rate_count, 0));
      Gradients(child, &slice, params ? params + static_cast<size_t>(begin) * K : nullptr, rescaling, rooted,
                &rows);
    });
    return;
  }
  auto batches = RunOverPatternShards(group, trees, params, rooted, wanted && !analytic, true,
                                      SBNB_MODE_BRANCH_GRADIENT, rescaling, analytic);
  sbnb_batch* b0 = batches[0].get();
  const bool inv = group->spec.invariant && T > 0;
  std::vector<double> logl(b0->vtree_count), grad(static_cast<size_t>(T) * N), rgrad(static_cast<size_t>(T) * N),
      subst(analytic ? static_cast<size_t>(T) * kOeSubstSums : 0), inv_sums(inv ? static_cast<size_t>(T) * kOeInvariantSums : 0);
  Fetch(group->children[0], b0, logl.data(), grad.data(), rgrad.data(), analytic && T > 0 ? subst.data() : nullptr,
        nullptr, inv ? inv_sums.data() : nullptr);
  FinishGradients(group->spec, n, trees, rooted, b0->fd_coords, logl.data(), grad.data(), rgrad.data(), out,
                  &b0->programs, params, analytic && T > 0 ? subst.data() : nullptr, nullptr, 0,
                  inv ? inv_sums.data() : nullptr);
}

bool IsGroup(const sbnb_engine* e) { return !e->children.empty(); }
void RequireSingleDevice(const sbnb_engine* e) {
  Require(!IsGroup(e), "The staged entry points work on one device: call them on an engine created with "
                       "sbnb_engine_create (a device group offers the one-call entry points).");
}

}  // namespace

extern "C" {

const char* sbnb_last_error(void) { return g_last_error.c_str(); }

int sbnb_device_count(void) {
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return count;
}

int sbnb_engine_create(const char* substitution, const char* site, const char* clock,
                       int32_t taxon_count, int64_t pattern_count, const uint8_t* tip_states,
                       const double* pattern_weights, int32_t device, sbnb_engine** out) {
  return sbnb_engine_create_encoded(substitution, site, clock, taxon_count, pattern_count, tip_states,
                                    SBNB_TIPS_STATES, pattern_weights, device, out);
}

int sbnb_engine_create_encoded(const char* substitution, const char* site, const char* clock,
                               int32_t taxon_count, int64_t pattern_count, const uint8_t* tips,
                               int32_t tip_encoding, const double* pattern_weights, int32_t device,
                               sbnb_engine** out) {
  return Guard([&] {
    Require(out != nullptr, "NULL output handle.");
    *out = nullptr;
    *out = CreateEngine(substitution, site, clock, taxon_count, pattern_count, tips, tip_encoding, pattern_weights,
                        device, nullptr)
               .release();
  });
}

int sbnb_engine_create_multi(const char* substitution, const char* site, const char* clock,
                             int32_t taxon_count, int64_t pattern_count, const uint8_t* tip_states,
                             const double* pattern_weights, const int32_t* devices, int32_t device_count,
                             int32_t shard_axis, sbnb_engine** out) {
  return sbnb_engine_create_multi_encoded(substitution, site, clock, taxon_count, pattern_count, tip_states,
                                          SBNB_TIPS_STATES, pattern_weights, devices, device_count, shard_axis, out);
}

int sbnb_engine_create_multi_encoded(const char* substitution, const char* site, const char* clock,
                                     int32_t taxon_count, int64_t pattern_count, const uint8_t* tips,
                                     int32_t tip_encoding, const double* pattern_weights, const int32_t* devices,
                                     int32_t device_count, int32_t shard_axis, sbnb_engine** out) {
  return Guard([&] {
    Require(out != nullptr, "NULL output handle.");
    *out = nullptr;
    Require(devices != nullptr && device_count >= 1 && device_count <= 16, "Need 1 to 16 device ordinals.");
    Require(shard_axis == SBNB_SHARD_TREES || shard_axis == SBNB_SHARD_PATTERNS, "Unknown shard axis.");
    Require(shard_axis == SBNB_SHARD_TREES || pattern_count >= device_count,
            "Cannot shard fewer site patterns than devices.");
    auto group = std::make_unique<sbnb_engine>();
    group->shard_axis = shard_axis;
    for (int g = 0; g < device_count; g++) {
      auto child = CreateEngine(substitution, site, clock, taxon_count, pattern_count, tips, tip_encoding,
                                pattern_weights, devices[g], group->children.empty() ? nullptr : group->children[0]);
      if (shard_axis == SBNB_SHARD_PATTERNS && device_count > 1)
        UploadPatternRange(child.get(), pattern_count * g / device_count, pattern_count * (g + 1) / device_count);
      group->children.push_back(child.release());
    }
    const sbnb_engine* first = group->children[0];
    group->spec = first->spec;
    group->device = first->device;
    group->taxon_count = first->taxon_count;
    group->pattern_count = first->pattern_count;
    group->categories = first->categories;
    group->padded_categories = first->padded_categories;
    group->ambiguous = first->ambiguous;
    group->substitution_mode = first->substitution_mode;
    *out = group.release();
  });
}

int sbnb_engine_set_substitution_gradient(sbnb_engine* engine, int32_t mode) {
  return Guard([&] {
    Require(engine != nullptr, "NULL engine.");
    Require(mode == SBNB_SUBSTITUTION_ANALYTIC || mode == SBNB_SUBSTITUTION_FINITE_DIFFERENCES,
            "Unknown substitution-gradient mode.");
    engine->substitution_mode = mode;
    for (sbnb_engine* child : engine->children) child->substitution_mode = mode;
  });
}

int32_t sbnb_engine_device_count(const sbnb_engine* engine) {
  if (!engine) return -1;
  return engine->children.empty() ? 1 : static_cast<int32_t>(engine->children.size());
}

void sbnb_engine_destroy(sbnb_engine* engine) {
  if (!engine) return;
  FloatingPointEnvironmentKeeper keep_caller_environment;
  cudaSetDevice(engine->device);
  delete engine;
}

int32_t sbnb_engine_param_count(const sbnb_engine* engine) {
  return engine ? engine->spec.param_count : -1;
}

int sbnb_engine_param_block(const sbnb_engine* engine, const char* key, int32_t* start,
                            int32_t* length) {
  return Guard([&] {
    Require(engine && key && start && length, "NULL argument.");
    const auto block = engine->spec.Block(key);
    *start = block.first;
    *length = block.second;
  });
}

int32_t sbnb_engine_category_count(const sbnb_engine* engine) {
  return engine ? engine->categories : -1;
}

int sbnb_log_likelihoods_unrooted(sbnb_engine* engine, const sbnb_tree_batch* trees,
                                  const double* params, int32_t rescaling, double* out) {
  return Guard([&] {
    Require(engine != nullptr, "NULL engine.");
    (IsGroup(engine) ? GroupLogLikelihoods : LogLikelihoods)(engine, trees, params, rescaling != 0, false, false, out);
  });
}

int sbnb_log_likelihoods_rooted(sbnb_engine* engine, const sbnb_tree_batch* trees,
                                const double* params, int32_t rescaling, double* out) {
  return Guard([&] {
    Require(engine != nullptr, "NULL engine.");
    (IsGroup(engine) ? GroupLogLikelihoods : LogLikelihoods)(engine, trees, params, rescaling != 0, true, true, out);
  });
}

int sbnb_unrooted_log_likelihoods_of_rooted(sbnb_engine* engine, const sbnb_tree_batch* trees,
                                            const double* params, int32_t rescaling, double* out) {
  return Guard([&] {
    Require(engine != nullptr, "NULL engine.");
    // fat_beagle.cpp:78-80: plain branch lengths, no rates, no Jacobian.
    Require(trees && trees->node_count == 2 * engine->taxon_count - 1,
            "Rooted trees must be bifurcating: node_count must be 2n-1.");
    (IsGroup(engine) ? GroupLogLikelihoods : LogLikelihoods)(engine, trees, params, rescaling != 0, false, false, out);
  });
}

int sbnb_gradients_unrooted(sbnb_engine* engine, const sbnb_tree_batch* trees, const double* params,
                            int32_t rescaling, const sbnb_gradient_out* out) {
  return Guard([&] {
    Require(engine != nullptr, "NULL engine.");
    (IsGroup(engine) ? GroupGradients : Gradients)(engine, trees, params, rescaling != 0, false, out);
  });
}

int sbnb_gradients_rooted(sbnb_engine* engine, const sbnb_tree_batch* trees, const double* params,
                          int32_t rescaling, const sbnb_gradient_out* out) {
  return Guard([&] {
    Require(engine != nullptr, "NULL engine.");
    (IsGroup(engine) ? GroupGradients : Gradients)(engine, trees, params, rescaling != 0, true, out);
  });
}

int sbnb_finish_gradients(const char* substitution, const char* site, const char* clock,
                          int32_t taxon_count, const sbnb_tree_batch* trees, int32_t rooted,
                          int32_t with_substitution_fd, const double* log_likelihoods,
                          const double* branch_gradients, const double* rate_gradients,
                          const sbnb_gradient_out* out) {
  return Guard([&] {
    Require(substitution && site && clock, "NULL model specification string.");
    Require(trees != nullptr, "NULL tree batch.");
    Require(taxon_count >= 3, "Need at least 3 taxa.");
    const ModelSpec spec = ModelSpec::Parse(substitution, site, clock);
    Require(!spec.invariant, std::string("The site model ") + site +
                                 " has invariable sites: finish with sbnb_finish_gradients_invariant, which takes "
                                 "the +I sums (sbnb_batch_fetch_invariant_sums).");
    Require(trees->tree_count == 0 || (trees->parent_ids && trees->branch_lengths),
            "NULL parent_ids / branch_lengths.");
    Require(trees->tree_count == 0 || (log_likelihoods && branch_gradients),
            "NULL log_likelihoods / branch_gradients.");
    Require(spec.category_count == 1 || trees->tree_count == 0 || rate_gradients != nullptr,
            "rate_gradients are required for a multi-category site model.");
    Require(!rooted || trees->tree_count == 0 || trees->rates != nullptr,
            "Rooted evaluation needs per-branch rates (RootedTree::rates_).");
    FinishGradients(spec, taxon_count, trees, rooted != 0,
                    with_substitution_fd ? spec.SubstitutionGradientSize() : 0, log_likelihoods,
                    branch_gradients, rate_gradients, out);
  });
}

int sbnb_finish_log_likelihoods_rooted(int32_t taxon_count, const sbnb_tree_batch* trees,
                                       double* log_likelihoods) {
  return Guard([&] {
    Require(trees != nullptr, "NULL tree batch.");
    Require(trees->tree_count == 0 || (log_likelihoods && trees->node_heights && trees->node_bounds),
            "Rooted log likelihoods need node_heights and node_bounds.");
    for (int t = 0; t < trees->tree_count; t++) {
      const TreeProgram tree = BuildTreeProgram(
          trees->parent_ids + static_cast<size_t>(t) * (trees->node_count - 1), trees->node_count, taxon_count);
      log_likelihoods[t] += LogDetJacobianHeightRatios(tree, ViewOf(trees, t, taxon_count));
    }
  });
}

int sbnb_batch_stage(sbnb_engine* engine, const sbnb_tree_batch* trees, const double* params,
                     int32_t stage_flags, sbnb_batch** out) {
  return Guard([&] {
    Require(engine && out, "NULL argument.");
    *out = nullptr;
    RequireSingleDevice(engine);
    // (unrooted batches are staged with the root slid as the reference's Gradient does:
    //  a no-op for trifurcating input; for bifurcating input the log-likelihood is the
    //  same by the pulley principle)
    Require(!((stage_flags & SBNB_STAGE_SUBSTITUTION_FD) && (stage_flags & SBNB_STAGE_SUBSTITUTION_ANALYTIC)),
            "A batch is staged for one substitution-gradient method.");
    *out = Stage(engine, trees, params, (stage_flags & SBNB_STAGE_ROOTED) != 0,
                 (stage_flags & SBNB_STAGE_SUBSTITUTION_FD) != 0, /*slide_root=*/true,
                 (stage_flags & SBNB_STAGE_SUBSTITUTION_ANALYTIC) != 0 && engine->spec.SubstitutionGradientSize() > 0)
               .release();
  });
}

int sbnb_batch_run(sbnb_engine* engine, sbnb_batch* batch, int32_t mode, int32_t rescaling) {
  return Guard([&] {
    Require(engine && batch, "NULL argument.");
    RequireSingleDevice(engine);
    Run(engine, batch, mode, rescaling != 0);
  });
}

int sbnb_batch_fetch(sbnb_engine* engine, sbnb_batch* batch, double* log_likelihoods,
                     double* branch_gradients, double* rate_gradients) {
  return Guard([&] {
    Require(engine && batch, "NULL argument.");
    RequireSingleDevice(engine);
    Fetch(engine, batch, log_likelihoods, branch_gradients, rate_gradients);
  });
}

int sbnb_batch_fetch_substitution_sums(sbnb_engine* engine, sbnb_batch* batch, double* sums) {
  return Guard([&] {
    Require(engine && batch && sums, "NULL argument.");
    RequireSingleDevice(engine);
    Fetch(engine, batch, nullptr, nullptr, nullptr, sums);
  });
}

int sbnb_finish_gradients_analytic(const char* substitution, const char* site, const char* clock,
                                   int32_t taxon_count, const sbnb_tree_batch* trees, int32_t rooted,
                                   const double* params, const double* log_likelihoods,
                                   const double* branch_gradients, const double* rate_gradients,
                                   const double* substitution_sums, const sbnb_gradient_out* out) {
  return Guard([&] {
    Require(substitution && site && clock, "NULL model specification string.");
    Require(trees != nullptr, "NULL tree batch.");
    Require(taxon_count >= 3, "Need at least 3 taxa.");
    const ModelSpec spec = ModelSpec::Parse(substitution, site, clock);
    Require(!spec.invariant, std::string("The site model ") + site +
                                 " has invariable sites: finish with sbnb_finish_gradients_invariant, which takes "
                                 "the +I sums (sbnb_batch_fetch_invariant_sums).");
    Require(trees->tree_count == 0 || (trees->parent_ids && trees->branch_lengths),
            "NULL parent_ids / branch_lengths.");
    Require(trees->tree_count == 0 || (log_likelihoods && branch_gradients),
            "NULL log_likelihoods / branch_gradients.");
    Require(spec.category_count == 1 || trees->tree_count == 0 || rate_gradients != nullptr,
            "rate_gradients are required for a multi-category site model.");
    Require(spec.param_count == 0 || trees->tree_count == 0 || params != nullptr,
            "NULL phylo model parameter matrix.");
    Require(!rooted || trees->tree_count == 0 || trees->rates != nullptr,
            "Rooted evaluation needs per-branch rates (RootedTree::rates_).");
    FinishGradients(spec, taxon_count, trees, rooted != 0, 0, log_likelihoods, branch_gradients, rate_gradients,
                    out, nullptr, params, spec.SubstitutionGradientSize() > 0 ? substitution_sums : nullptr);
  });
}

int sbnb_batch_fetch_invariant_sums(sbnb_engine* engine, sbnb_batch* batch, double* sums) {
  return Guard([&] {
    Require(engine && batch && sums, "NULL argument.");
    RequireSingleDevice(engine);
    Fetch(engine, batch, nullptr, nullptr, nullptr, nullptr, nullptr, sums);
  });
}

int sbnb_finish_gradients_invariant(const char* substitution, const char* site, const char* clock,
                                    int32_t taxon_count, const sbnb_tree_batch* trees, int32_t rooted,
                                    const double* params, const double* log_likelihoods,
                                    const double* branch_gradients, const double* rate_gradients,
                                    const double* substitution_sums, const double* invariant_sums,
                                    const sbnb_gradient_out* out) {
  return Guard([&] {
    Require(substitution && site && clock, "NULL model specification string.");
    Require(trees != nullptr, "NULL tree batch.");
    Require(taxon_count >= 3, "Need at least 3 taxa.");
    const ModelSpec spec = ModelSpec::Parse(substitution, site, clock);
    Require(spec.invariant, std::string("The site model ") + site + " has no invariable sites (+I).");
    Require(trees->tree_count == 0 || (trees->parent_ids && trees->branch_lengths),
            "NULL parent_ids / branch_lengths.");
    Require(trees->tree_count == 0 || (log_likelihoods && branch_gradients && invariant_sums && params),
            "NULL log_likelihoods / branch_gradients / invariant_sums / params.");
    Require(spec.category_count == 1 || trees->tree_count == 0 || rate_gradients != nullptr,
            "rate_gradients are required for a multi-category site model.");
    Require(!rooted || trees->tree_count == 0 || trees->rates != nullptr,
            "Rooted evaluation needs per-branch rates (RootedTree::rates_).");
    for (int t = 0; t < trees->tree_count; t++) {  // (the same refusal as at staging)
      const double pinv = params[static_cast<size_t>(t) * spec.param_count + spec.Block("proportion invariant").first];
      if (!(pinv >= 0.0 && pinv < 1.0)) Fail(SBNB_ERR_MODEL, "Proportion invariant must lie in [0, 1).");
    }
    FinishGradients(spec, taxon_count, trees, rooted != 0, 0, log_likelihoods, branch_gradients, rate_gradients,
                    out, nullptr, params, spec.SubstitutionGradientSize() > 0 ? substitution_sums : nullptr, nullptr,
                    0, invariant_sums);
  });
}

int sbnb_batch_device_results(sbnb_batch* batch, void** log_likelihoods, void** branch_gradients,
                              void** rate_gradients) {
  return Guard([&] {
    Require(batch != nullptr, "NULL batch.");
    // (one contiguous fp64 array: log-likelihoods, branch gradients, rate gradients)
    if (log_likelihoods) *log_likelihoods = batch->ResultLogl();
    if (branch_gradients) *branch_gradients = batch->ResultGrad();
    if (rate_gradients) *rate_gradients = batch->categories > 1 ? batch->ResultRateGrad() : nullptr;
  });
}

void sbnb_batch_destroy(sbnb_engine* engine, sbnb_batch* batch) {
  FloatingPointEnvironmentKeeper keep_caller_environment;
  if (engine) cudaSetDevice(engine->device);
  Recycle(engine, batch);
}

int32_t sbnb_batch_evaluation_count(const sbnb_batch* batch) {
  if (!batch) return -1;
  return batch->last_mode == SBNB_MODE_BRANCH_GRADIENT ? batch->vtree_count : batch->tree_count;
}

void* sbnb_engine_stream(sbnb_engine* engine) {
  if (!engine) return nullptr;
  return IsGroup(engine) ? engine->children[0]->stream : engine->stream;
}

int64_t sbnb_engine_launch_count(const sbnb_engine* engine) {
  if (!engine) return -1;
  int64_t count = engine->launch_count;
  for (const sbnb_engine* child : engine->children) count += child->launch_count;
  return count;
}

int sbnb_engine_transfer_bytes(const sbnb_engine* engine, int64_t* host_to_device,
                               int64_t* device_to_host) {
  return Guard([&] {
    Require(engine && host_to_device && device_to_host, "NULL argument.");
    *host_to_device = engine->h2d_bytes;
    *device_to_host = engine->d2h_bytes;
    for (const sbnb_engine* child : engine->children) {
      *host_to_device += child->h2d_bytes;
      *device_to_host += child->d2h_bytes;
    }
  });
}

int sbnb_engine_walk_timing(sbnb_engine* engine, double* total_ms, int64_t* samples,
                            int32_t reset) {
  return Guard([&] {
    Require(engine && total_ms && samples, "NULL argument.");
    RequireSingleDevice(engine);
    SBNB_CUDA(cudaSetDevice(engine->device));
    // oldest first, so that walk_last_ms ends up being the newest run
    for (int i = 0; i < sbnb_engine::kWalkRing; i++)
      HarvestWalkTiming(engine, static_cast<int>((engine->walk_runs + i) % sbnb_engine::kWalkRing));
    *total_ms = engine->walk_total_ms;
    *samples = engine->walk_samples;
    if (reset) {
      engine->walk_total_ms = 0.0;
      engine->walk_samples = 0;
    }
  });
}

double sbnb_batch_algorithmic_bytes(const sbnb_batch* batch, int32_t mode) {
  // SURVEY.md 8d: U = 32 C P bytes per partial; (2n-2) U per log-likelihood,
  // (10n-14) U per log-likelihood + branch gradient.
  if (!batch) return 0.0;
  const double n = batch->taxon_count;
  const double units = (mode == SBNB_MODE_BRANCH_GRADIENT) ? (10.0 * n - 14.0) : (2.0 * n - 2.0);
  return units * 32.0 * batch->categories * static_cast<double>(batch->patterns) * batch->tree_count;
}

int sbnb_engine_set_pattern_range(sbnb_engine* engine, int64_t begin, int64_t end) {
  return Guard([&] {
    Require(engine != nullptr, "NULL engine.");
    RequireSingleDevice(engine);
    Require(0 <= begin && begin < end && end <= engine->pattern_count,
            "Pattern range must satisfy 0 <= begin < end <= pattern_count.");
    SBNB_CUDA(cudaSetDevice(engine->device));
    UploadPatternRange(engine, begin, end);
  });
}

int sbnb_debug_tree_program(const int32_t* parent_ids, int32_t node_count, int32_t taxon_count,
                            int32_t* post_ops, int32_t* pre_ops, int32_t* slots) {
  return Guard([&] {
    Require(parent_ids && post_ops && pre_ops && slots, "NULL argument.");
    const TreeProgram program = BuildTreeProgram(parent_ids, node_count, taxon_count);
    static_assert(sizeof(PostOp) == 32 && sizeof(PreOp) == 32, "ops are 8 x int32");
    std::memcpy(post_ops, program.post.data(), program.post.size() * sizeof(PostOp));
    std::memcpy(pre_ops, program.pre.data(), program.pre.size() * sizeof(PreOp));
    slots[0] = program.post_slots;
    slots[1] = program.pre_slots;
  });
}

int sbnb_debug_model_tables(const char* substitution, const char* site, const char* clock,
                            const double* param_row, double* eigenvectors,
                            double* inverse_eigenvectors, double* eigenvalues, double* frequencies,
                            double* q, double* category_rates, double* category_weights,
                            double* category_rate_derivatives) {
  return Guard([&] {
    Require(substitution && site && clock, "NULL model specification string.");
    const ModelSpec spec = ModelSpec::Parse(substitution, site, clock);
    Require(spec.param_count == 0 || param_row != nullptr, "NULL parameter row.");
    ModelTables tables;
    BuildModelTables(spec, param_row, &tables);
    if (eigenvectors) std::copy(tables.evec, tables.evec + 16, eigenvectors);
    if (inverse_eigenvectors) std::copy(tables.ivec, tables.ivec + 16, inverse_eigenvectors);
    if (eigenvalues) std::copy(tables.eval, tables.eval + 4, eigenvalues);
    if (frequencies) std::copy(tables.freqs, tables.freqs + 4, frequencies);
    if (q) std::copy(tables.q, tables.q + 16, q);
    const int C = spec.category_count;
    if (category_rates) std::copy(tables.rates, tables.rates + C, category_rates);
    if (category_weights) std::copy(tables.weights, tables.weights + C, category_weights);
    if (category_rate_derivatives) std::copy(tables.drates, tables.drates + C, category_rate_derivatives);
  });
}

int sbnb_debug_substitution_derivatives(const char* substitution, const char* site, const char* clock,
                                        const double* param_row, double* b, double* dfreqs, int32_t* count) {
  return Guard([&] {
    Require(substitution && site && clock && b && dfreqs && count, "NULL argument.");
    const ModelSpec spec = ModelSpec::Parse(substitution, site, clock);
    Require(spec.param_count == 0 || param_row != nullptr, "NULL parameter row.");
    ModelTables tables;
    BuildModelTables(spec, param_row, &tables);
    SubstitutionDerivatives derivatives;
    BuildSubstitutionDerivatives(spec, param_row, tables, &derivatives);
    *count = derivatives.count;
    for (int t = 0; t < derivatives.count; t++) {
      std::copy(derivatives.b[t], derivatives.b[t] + 16, b + 16 * t);
      std::copy(derivatives.dfreqs[t], derivatives.dfreqs[t] + 4, dfreqs + 4 * t);
    }
  });
}

}  // extern "C"
