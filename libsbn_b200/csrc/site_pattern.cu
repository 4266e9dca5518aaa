// Site-pattern compression on the device: the C ABI of include/sbn_b200_patterns.h,
// replacing the reference's SitePattern::Compress (src/site_pattern.cpp:77-115) and
// its symbol table (site_pattern.cpp:15-45).
//
// HBM-bound byte/integer work over an alignment stored [taxon][site]; the characters are
// read where they lie (no symbolised copy):
//   HashKernel           4 sites per thread (32-bit loads along a taxon row, 8 taxa in
//                        flight): characters -> symbols 0..4 through a shared-memory
//                        table (already shifted into place), the symbols of 8 taxa
//                        packed into one word per site, two 32-bit MurmurHash3-style
//                        hashes per column updated once per 8 taxa, mixed into one
//                        64-bit key
//   InsertKernel         one thread per site: claim / find the column's slot in an
//                        open-addressing table (atomicCAS on the 64-bit key), then
//                        atomicMin of the site index (the pattern's first
//                        appearance) and atomicAdd of its multiplicity
//   FlagKernel           flags first appearances
//   ScanBlocksKernel / ScanSumsKernel
//                        exclusive prefix sum of the flags = pattern index in order
//                        of first appearance (deterministic; no sort)
//   EmitKernel           4 sites per thread: first appearances write their column
//                        (a 32-bit store where four neighbours are four consecutive
//                        patterns -- every site of an alignment without repeats), weight
//                        and (per slot) pattern index; a pattern that repeats is given a
//                        second, CONTIGUOUS (taxon-fastest) column for the check
//   TileKernel<false>    writes those contiguous columns, TileKernel<true> holds every
//                        site that repeats a pattern against its pattern's column byte
//                        for byte: a CTA stages a tile of 128 sites x 64 taxa in shared
//                        memory (coalesced 128-byte row reads), then lanes = taxa, 32
//                        consecutive bytes of the column per request (the first version
//                        gathered single bytes of the [taxon][pattern] output: 3.3 ms at
//                        1000 taxa x 1M sites with 50k patterns).  A 64-bit key shared
//                        by two different columns is caught -- the host then retries
//                        with another seed -- never silently merged
// There is no CPU path in this file.

#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/sbn_b200_patterns.h"
#include "common.hpp"
#include "device_common.cuh"

namespace sbnb {

namespace {

constexpr int kSitesPerThread = 4;
constexpr int kRowAlignment = 128;  // device rows are whole 128-site tiles
constexpr int kTileSites = 128, kTileTaxa = 64;
constexpr uint32_t kNoColumn = 0xffffffffu;
constexpr int64_t kLongRow = 1 << 16;  // host rows copied one by one from this length on
constexpr int kHashThreads = 256;
constexpr int kScanThreads = 256;
constexpr int kScanItems = 4;  // flags per thread -> 1024 per block
constexpr int kScanBlock = kScanThreads * kScanItems;
constexpr uint64_t kEmptyKey = ~0ull;
constexpr uint8_t kUnknownSymbol = 0xff;

// GetSymbolTable (site_pattern.cpp:15-45): DNA, degenerate nucleotides are gaps.
void BuildSymbolTable(uint8_t (&table)[256]) {
  std::memset(table, kUnknownSymbol, sizeof(table));
  const char* acgt = "ACGT";
  for (int i = 0; i < 4; i++) {
    table[static_cast<unsigned char>(acgt[i])] = static_cast<uint8_t>(i);
    table[static_cast<unsigned char>(acgt[i] - 'A' + 'a')] = static_cast<uint8_t>(i);
  }
  for (const char* c = "-NX?BDHKMRSUVWY"; *c; c++) table[static_cast<unsigned char>(*c)] = 4;
}

// The IUPAC nucleotide codes as masks of the states they allow (bit 0 = A, 1 = C, 2 = G,
// 3 = T), upper and lower case; U = T; N X ? - = 15 (missing).
void BuildMaskTable(uint8_t (&table)[256]) {
  std::memset(table, kUnknownSymbol, sizeof(table));
  static const struct {
    char symbol;
    uint8_t mask;
  } kCodes[] = {{'A', 1},  {'C', 2},  {'G', 4},  {'T', 8},  {'U', 8},  {'R', 5},  {'Y', 10}, {'S', 6},
                {'W', 9},  {'K', 12}, {'M', 3},  {'B', 14}, {'D', 13}, {'H', 11}, {'V', 7},  {'N', 15},
                {'X', 15}};
  for (const auto& code : kCodes) {
    table[static_cast<unsigned char>(code.symbol)] = code.mask;
    table[static_cast<unsigned char>(code.symbol - 'A' + 'a')] = code.mask;
  }
  table[static_cast<unsigned char>('?')] = 15;
  table[static_cast<unsigned char>('-')] = 15;
}

struct SymbolTable {
  uint8_t map[256];
};

__device__ __forceinline__ uint64_t Mix(uint64_t x) {  // splitmix64 finaliser
  x ^= x >> 30;
  x *= 0xbf58476d1ce4e5b9ull;
  x ^= x >> 27;
  x *= 0x94d049bb133111ebull;
  return x ^ (x >> 31);
}

// One MurmurHash3-style step: the word is multiplied, rotated and multiplied before it meets
// the state, and the state is rotated afterwards.  (Multiply-xor steps WITHOUT the rotations
// only carry differences upward: fed with packed words, two columns that differ in the
// top nibbles of two words then collide in every such hash at once -- 3 of the 238 patterns
// of the reference's flu alignment did; the verification caught it under every seed.)
__device__ __forceinline__ uint32_t HashStep(uint32_t h, uint32_t word, uint32_t c1, uint32_t c2, int r1, int r2,
                                             uint32_t m, uint32_t add) {
  uint32_t k = word * c1;
  k = __funnelshift_l(k, k, r1) * c2;
  h ^= k;
  return __funnelshift_l(h, h, r2) * m + add;
}

// *unknown = the least position t * site_count + site of an unknown character (all ones = none),
// so the report names the first one in (taxon, site) order whatever the timing.
// MASKS: the table holds nucleotide masks 1..15, and an unknown character hashes as 0.
template <bool MASKS>
__global__ void __launch_bounds__(kHashThreads) HashKernel(
    const uint8_t* __restrict__ sequences, uint64_t* __restrict__ keys, int32_t taxon_count, int64_t site_count,
    int64_t pitch, uint64_t seed, uint64_t key_mask, const SymbolTable table,
    unsigned long long* __restrict__ unknown) {
  // character -> its symbol as a 4-bit field already in the place of taxon i of a group of 8
  // (an unknown character: 0xf, the only value with bit 3 set; with MASKS, 0, the only zero field)
  __shared__ uint32_t shifted[8][256];
  for (int i = threadIdx.x; i < 8 * 256; i += blockDim.x) {
    const uint8_t symbol = table.map[i & 255];
    const uint32_t field = MASKS ? (symbol == kUnknownSymbol ? 0u : symbol) : (symbol & 0xfu);
    shifted[i >> 8][i & 255] = field << (4 * (i >> 8));
  }
  __syncthreads();
  const int64_t group = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int64_t site0 = group * kSitesPerThread;
  if (site0 >= site_count) return;
  // Two 32-bit hashes per column (32-bit integer multiply-adds; a 64-bit multiply is three
  // of them), mixed into the 64-bit key at the end.  They consume the symbols of 8 taxa at
  // a time, 4 bits each.
  uint32_t ha[kSitesPerThread], hb[kSitesPerThread];
  const uint32_t seed_low = static_cast<uint32_t>(seed), seed_high = static_cast<uint32_t>(seed >> 32);
#pragma unroll
  for (int k = 0; k < kSitesPerThread; k++) {
    ha[k] = 0x811c9dc5u ^ seed_low;
    hb[k] = 0x9e3779b9u + seed_high;
  }
  uint32_t seen = 0;  // bit 3 of a field = an unknown character (MASKS: of the zero-field test)
  const uint8_t* column = sequences + site0;
  for (int t0 = 0; t0 < taxon_count; t0 += 16) {
    // (a thread has one 4-byte load per taxon, so the loads of many taxa must be in flight
    //  together to cover the HBM latency: 16 measured 0.31 ms against 0.37 ms with 8 at
    //  1000 taxa x 1M sites)
    uint32_t word[16];
#pragma unroll
    for (int i = 0; i < 16; i++)
      word[i] = (t0 + i < taxon_count) ? *reinterpret_cast<const uint32_t*>(column + static_cast<int64_t>(t0 + i) * pitch)
                                       : 0x41414141u;  // (rows past the last taxon read as 'A' for every site)
#pragma unroll
    for (int half = 0; half < 2; half++) {
      if (t0 + 8 * half >= taxon_count) break;  // (same number of hash steps for every site)
      uint32_t packed[kSitesPerThread];
#pragma unroll
      for (int k = 0; k < kSitesPerThread; k++) packed[k] = 0;
#pragma unroll
      for (int i = 0; i < 8; i++) {
#pragma unroll
        for (int k = 0; k < kSitesPerThread; k++) packed[k] |= shifted[i][(word[8 * half + i] >> (8 * k)) & 0xffu];
      }
#pragma unroll
      for (int k = 0; k < kSitesPerThread; k++) {
        // (MASKS: a field is zero exactly when it borrows in packed - 0x11111111 without having
        //  had bit 3 set; the padding taxa of a group read as 'A' = 1)
        seen |= MASKS ? (packed[k] - 0x11111111u) & ~packed[k] : packed[k];
        ha[k] = HashStep(ha[k], packed[k], 0xcc9e2d51u, 0x1b873593u, 15, 13, 5u, 0xe6546b64u);  // (MurmurHash3's own)
        hb[k] = HashStep(hb[k], packed[k], 0x85ebca6bu, 0xc2b2ae35u, 16, 11, 9u, 0x7f4a7c15u);
      }
    }
  }
  if (seen & 0x88888888u) {
    // rare: the thread's first unknown character in (taxon, site) order (padding sites hold 'A')
    for (int t = 0; t < taxon_count; t++) {
      for (int k = 0; k < kSitesPerThread; k++) {
        const uint8_t c = column[static_cast<int64_t>(t) * pitch + k];
        if (table.map[c] == kUnknownSymbol && site0 + k < site_count) {
          atomicMin(unknown, static_cast<unsigned long long>(t * site_count + site0 + k));
          t = taxon_count;
          break;
        }
      }
    }
  }
#pragma unroll
  for (int k = 0; k < kSitesPerThread; k++) {
    if (site0 + k < site_count) {
      uint64_t key = Mix((static_cast<uint64_t>(ha[k]) << 32 | hb[k]) + 0x9e3779b97f4a7c15ull);
      key &= key_mask;  // all ones, except in the collision-handling test
      if (key == kEmptyKey) key = 0;
      keys[site0 + k] = key;
    }
  }
}

__global__ void InsertKernel(const uint64_t* __restrict__ keys, unsigned long long* __restrict__ table_keys,
                             uint32_t* __restrict__ table_first, uint32_t* __restrict__ table_count,
                             uint32_t* __restrict__ slot_of, int64_t site_count, uint32_t mask) {
  const int64_t site = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (site >= site_count) return;
  const uint64_t key = keys[site];
  uint32_t slot = static_cast<uint32_t>(Mix(key)) & mask;
  while (true) {
    const unsigned long long previous = atomicCAS(&table_keys[slot], kEmptyKey, key);
    if (previous == kEmptyKey || previous == key) break;
    slot = (slot + 1) & mask;
  }
  slot_of[site] = slot;
  atomicMin(&table_first[slot], static_cast<uint32_t>(site));
  atomicAdd(&table_count[slot], 1u);
}

__global__ void FlagKernel(const uint32_t* __restrict__ slot_of, const uint32_t* __restrict__ table_first,
                           uint32_t* __restrict__ flags, int64_t site_count) {
  const int64_t site = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (site < site_count) flags[site] = (table_first[slot_of[site]] == site) ? 1u : 0u;
}

// Block-local exclusive scan of 1024 flags; the block's total goes to block_sums.
__global__ void __launch_bounds__(kScanThreads) ScanBlocksKernel(const uint32_t* __restrict__ flags,
                                                                 uint32_t* __restrict__ index,
                                                                 uint32_t* __restrict__ block_sums,
                                                                 int64_t count) {
  __shared__ uint32_t warp_totals[kScanThreads / 32];
  const int64_t base = (static_cast<int64_t>(blockIdx.x) * kScanThreads + threadIdx.x) * kScanItems;
  uint32_t item[kScanItems], sum = 0;
#pragma unroll
  for (int k = 0; k < kScanItems; k++) {
    item[k] = (base + k < count) ? flags[base + k] : 0u;
    sum += item[k];
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t inclusive = sum;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t up = __shfl_up_sync(0xffffffffu, inclusive, d);
    if (lane >= d) inclusive += up;
  }
  if (lane == 31) warp_totals[warp] = inclusive;
  __syncthreads();
  uint32_t offset = 0, total = 0;
#pragma unroll
  for (int w = 0; w < kScanThreads / 32; w++) {
    if (w < warp) offset += warp_totals[w];
    total += warp_totals[w];
  }
  uint32_t running = offset + inclusive - sum;
#pragma unroll
  for (int k = 0; k < kScanItems; k++) {
    if (base + k < count) index[base + k] = running;
    running += item[k];
  }
  if (threadIdx.x == 0) block_sums[blockIdx.x] = total;
}

// One block: exclusive scan of the block totals in place, grand total to *total.
__global__ void __launch_bounds__(1024) ScanSumsKernel(uint32_t* __restrict__ block_sums, int64_t blocks,
                                                       unsigned long long* __restrict__ total) {
  __shared__ uint32_t warp_totals[32];
  __shared__ unsigned long long carry_shared;
  if (threadIdx.x == 0) carry_shared = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int64_t start = 0; start < blocks; start += 1024) {
    const int64_t i = start + threadIdx.x;
    const uint32_t value = (i < blocks) ? block_sums[i] : 0u;
    uint32_t inclusive = value;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t up = __shfl_up_sync(0xffffffffu, inclusive, d);
      if (lane >= d) inclusive += up;
    }
    if (lane == 31) warp_totals[warp] = inclusive;
    __syncthreads();
    uint32_t offset = 0, chunk_total = 0;
    for (int w = 0; w < 32; w++) {
      if (w < warp) offset += warp_totals[w];
      chunk_total += warp_totals[w];
    }
    const unsigned long long carry = carry_shared;
    if (i < blocks) block_sums[i] = static_cast<uint32_t>(carry + offset + inclusive - value);
    __syncthreads();
    if (threadIdx.x == 0) carry_shared = carry + chunk_total;
    __syncthreads();
  }
  if (threadIdx.x == 0) *total = carry_shared;
}

// characters of four sites -> their four symbols
__device__ __forceinline__ uint32_t MapWord(const uint8_t* map, uint32_t word) {
  return static_cast<uint32_t>(map[word & 0xffu]) | static_cast<uint32_t>(map[(word >> 8) & 0xffu]) << 8 |
         static_cast<uint32_t>(map[(word >> 16) & 0xffu]) << 16 | static_cast<uint32_t>(map[word >> 24]) << 24;
}

// flags / index / slot_of hold `pitch` entries (flags zero past the last site).
__global__ void __launch_bounds__(kHashThreads) EmitKernel(
    const uint8_t* __restrict__ sequences, const uint32_t* __restrict__ slot_of,
    const uint32_t* __restrict__ table_count, const uint32_t* __restrict__ flags, const uint32_t* __restrict__ index,
    const uint32_t* __restrict__ block_sums, uint8_t* __restrict__ patterns, double* __restrict__ weights,
    uint32_t* __restrict__ table_pattern, uint32_t* __restrict__ table_column,
    uint32_t* __restrict__ column_counter, int32_t taxon_count, int64_t site_count, int64_t pitch,
    const SymbolTable table) {
  __shared__ uint8_t map[256];
  for (int i = threadIdx.x; i < 256; i += blockDim.x) map[i] = table.map[i];
  __syncthreads();
  const int64_t site0 = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) * kSitesPerThread;
  if (site0 >= site_count) return;
  const uint4 flag4 = *reinterpret_cast<const uint4*>(flags + site0);
  const uint32_t flag[4] = {flag4.x, flag4.y, flag4.z, flag4.w};
  if (!(flag[0] | flag[1] | flag[2] | flag[3])) return;
  const uint4 index4 = *reinterpret_cast<const uint4*>(index + site0);
  const uint32_t local[4] = {index4.x, index4.y, index4.z, index4.w};
  int64_t p[4];
#pragma unroll
  for (int k = 0; k < 4; k++) {
    p[k] = -1;
    if (!flag[k]) continue;
    p[k] = static_cast<int64_t>(local[k]) + block_sums[(site0 + k) / kScanBlock];
    const uint32_t slot = slot_of[site0 + k];
    const uint32_t count = table_count[slot];
    weights[p[k]] = static_cast<double>(count);
    table_pattern[slot] = static_cast<uint32_t>(p[k]);
    // a pattern that repeats gets a contiguous column for the verification (ColumnsKernel)
    table_column[slot] = count > 1 ? atomicAdd(column_counter, 1u) : kNoColumn;
  }
  const bool four_in_a_row = flag[0] && flag[1] && flag[2] && flag[3] && p[1] == p[0] + 1 && p[2] == p[0] + 2 &&
                             p[3] == p[0] + 3 && (p[0] & 3) == 0;
  const uint8_t* source = sequences + site0;
  if (four_in_a_row) {
#pragma unroll 8
    for (int t = 0; t < taxon_count; t++)
      *reinterpret_cast<uint32_t*>(patterns + static_cast<int64_t>(t) * pitch + p[0]) =
          MapWord(map, *reinterpret_cast<const uint32_t*>(source + static_cast<int64_t>(t) * pitch));
    return;
  }
#pragma unroll 4
  for (int t = 0; t < taxon_count; t++) {
    const uint32_t symbols = MapWord(map, *reinterpret_cast<const uint32_t*>(source + static_cast<int64_t>(t) * pitch));
#pragma unroll
    for (int k = 0; k < 4; k++) {
      if (!flag[k]) continue;
      const uint8_t symbol = static_cast<uint8_t>(symbols >> (8 * k));
      patterns[static_cast<int64_t>(t) * pitch + p[k]] = symbol;
    }
  }
}

// One CTA per tile of 128 sites, staged 64 taxa at a time in shared memory, TRANSPOSED
// ([site][taxon]: a lane reads a row's sites lane, lane + 32, ... -- each request one full
// 32-byte sector -- and stores them 17 words apart, conflict-free), so that the four symbols
// of four consecutive taxa of a site are one word.  Half a warp then covers the 64 taxa of
// one site with one 32-bit access per lane to the pattern's contiguous column (columns are
// padded to whole 64-taxon chunks; the padding holds zeros on both sides).
//   VERIFY = false: first appearances of patterns that repeat write their column.
//   VERIFY = true: every repeat compares its symbols with its pattern's column.
template <bool VERIFY>
__global__ void __launch_bounds__(256) TileKernel(const uint8_t* __restrict__ sequences,
                                                  const uint32_t* __restrict__ slot_of,
                                                  const uint32_t* __restrict__ flags,
                                                  const uint32_t* __restrict__ table_column,
                                                  uint8_t* __restrict__ columns, int32_t taxon_count,
                                                  int64_t site_count, int64_t pitch, int64_t column_pitch,
                                                  const SymbolTable table, int32_t* __restrict__ collided) {
  constexpr int kSiteWords = kTileTaxa / 4 + 1;  // 17: the sites of a warp's store fall into 32 banks
  __shared__ uint8_t map[256];
  __shared__ uint32_t column_of[kTileSites];
  __shared__ uint32_t tile[kTileSites][kSiteWords];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  map[tid] = table.map[tid];
  const int64_t tile_site = static_cast<int64_t>(blockIdx.x) * kTileSites;
  uint32_t mine = kNoColumn;
  if (tid < kTileSites) {
    const int64_t site = tile_site + tid;
    // the sites this pass works on: repeats (VERIFY) or first appearances
    if (site < site_count && (flags[site] != 0) != VERIFY) mine = table_column[slot_of[site]];
    column_of[tid] = mine;
  }
  if (!__syncthreads_or(mine != kNoColumn)) return;  // nothing to do in this tile
  uint8_t* const tile_bytes = reinterpret_cast<uint8_t*>(tile);
  uint32_t difference = 0;
  for (int t0 = 0; t0 < taxon_count; t0 += kTileTaxa) {
    if (t0 > 0) __syncthreads();  // every warp is done with the previous rows
#pragma unroll
    for (int i = 0; i < kTileTaxa / 8; i++) {
      const int row = warp + 8 * i;
      const bool inside = t0 + row < taxon_count;
      const uint8_t* const source = sequences + static_cast<int64_t>(inside ? t0 + row : 0) * pitch + tile_site + lane;
#pragma unroll
      for (int j = 0; j < kTileSites / 32; j++) {
        const uint8_t symbol = inside ? map[source[32 * j]] : 0;
        tile_bytes[(lane + 32 * j) * (kSiteWords * 4) + row] = symbol;
      }
    }
    __syncthreads();
    // warp w: sites 16 w .. 16 w + 15, two per step; a half-warp's lanes = 16 words of 4 taxa
    const int word = lane & 15;
#pragma unroll
    for (int s = 0; s < kTileSites / 16; s++) {
      const int k = warp * (kTileSites / 8) + 2 * s + (lane >> 4);
      const uint32_t id = column_of[k];
      if (id == kNoColumn) continue;
      uint32_t* const theirs =
          reinterpret_cast<uint32_t*>(columns + static_cast<int64_t>(id) * column_pitch + t0) + word;
      if (VERIFY) {
        difference |= tile[k][word] ^ *theirs;
      } else {
        *theirs = tile[k][word];
      }
    }
  }
  if (VERIFY && difference != 0) *collided = 1;
}

// "Symbol 'c' not known." (SymbolTableAt, site_pattern.cpp:47-55), with a byte outside printable
// ASCII written as \xHH so that the message stays valid text.
std::string UnknownSymbolMessage(uint8_t c) {
  char symbol[8];
  if (c >= 0x20 && c <= 0x7e) {
    std::snprintf(symbol, sizeof(symbol), "%c", c);
  } else {
    std::snprintf(symbol, sizeof(symbol), "\\x%02x", c);
  }
  return std::string("Symbol '") + symbol + "' not known.";
}

void Compress(int32_t n, int64_t S, const char* sequences, bool masks, int32_t device, uint8_t* out_patterns,
              double* out_weights, int64_t* out_pattern_count, double* out_device_ms) {
  Require(n > 0, "Site pattern compression needs at least one sequence.");
  Require(S >= 0 && S < (1ll << 30), "Site count out of range [0, 2^30).");  // 32-bit site ids, 2S-slot table
  Require(out_pattern_count != nullptr, "out_pattern_count is NULL.");
  int device_count = 0;
  if (cudaGetDeviceCount(&device_count) != cudaSuccess || device_count == 0)
    Fail(SBNB_ERR_NO_DEVICE, "No usable CUDA device: libsbn_b200 has no CPU fallback.");
  Require(device >= 0 && device < device_count, "CUDA device index out of range.");
  SBNB_CUDA(cudaSetDevice(device));
  *out_pattern_count = 0;
  if (out_device_ms) *out_device_ms = 0.0;
  if (S == 0) return;
  // SBNB_DEBUG_TIMING: wall-clock stages of the call on stderr
  const bool timing = std::getenv("SBNB_DEBUG_TIMING") != nullptr;
  auto stage_clock = std::chrono::steady_clock::now();
  auto stage = [&](const char* what) {
    if (!timing) return;
    cudaDeviceSynchronize();
    const auto now = std::chrono::steady_clock::now();
    std::fprintf(stderr, "[sbnb_compress_site_patterns] %-22s %8.2f ms\n", what,
                 std::chrono::duration<double, std::milli>(now - stage_clock).count());
    stage_clock = now;
  };
  Require(sequences && out_patterns && out_weights, "NULL buffer passed to sbnb_compress_site_patterns.");

  const int64_t pitch = (S + kRowAlignment - 1) / kRowAlignment * kRowAlignment;
  uint32_t table_size = 1024;
  while (table_size < 2ull * static_cast<uint64_t>(S)) table_size <<= 1;
  const int64_t scan_blocks = (S + kScanBlock - 1) / kScanBlock;

  DeviceArray<uint8_t> d_sequences, d_patterns, d_columns;
  DeviceArray<uint64_t> d_keys;
  DeviceArray<unsigned long long> d_table_keys, d_total;
  DeviceArray<uint32_t> d_table_first, d_table_count, d_table_pattern, d_table_column, d_slot_of, d_flags, d_index,
      d_block_sums, d_column_counter;
  DeviceArray<int32_t> d_collided;
  DeviceArray<double> d_weights;
  d_sequences.Reserve(static_cast<size_t>(n) * pitch);
  d_keys.Reserve(S);
  d_table_keys.Reserve(table_size);
  d_table_first.Reserve(table_size);
  d_table_count.Reserve(table_size);
  d_table_pattern.Reserve(table_size);
  d_table_column.Reserve(table_size);
  d_column_counter.Reserve(1);
  d_slot_of.Reserve(pitch);
  d_flags.Reserve(pitch);
  d_index.Reserve(pitch);
  // a pattern that repeats also keeps its column contiguously (taxon-fastest) for the
  // verification: at most S / 2 patterns repeat
  const int64_t column_pitch = (static_cast<int64_t>(n) + kTileTaxa - 1) / kTileTaxa * kTileTaxa;
  d_columns.Reserve(static_cast<size_t>(S / 2 + 1) * column_pitch);
  SBNB_CUDA(cudaMemset(d_flags.get(), 0, static_cast<size_t>(pitch) * sizeof(uint32_t)));
  d_block_sums.Reserve(scan_blocks);
  d_total.Reserve(2);  // the pattern count, then the position of the first unknown character
  d_collided.Reserve(1);
  d_weights.Reserve(pitch);
  d_patterns.Reserve(static_cast<size_t>(n) * pitch);
  stage("device allocations");
  // the padding columns of the last row segment must hold valid characters
  SBNB_CUDA(cudaMemset(d_sequences.get(), 'A', static_cast<size_t>(n) * pitch));
  // (pageable host rows: a 2-D copy of 1000 rows of 1 MB runs at ~2 GB/s; row-by-row copies of
  //  long rows go through the driver's staging buffers several times faster)
  if (S >= kLongRow) {
    for (int32_t t = 0; t < n; t++)
      SBNB_CUDA(cudaMemcpyAsync(d_sequences.get() + static_cast<size_t>(t) * pitch,
                                sequences + static_cast<size_t>(t) * S, S, cudaMemcpyHostToDevice, 0));
  } else {
    SBNB_CUDA(cudaMemcpy2D(d_sequences.get(), pitch, sequences, S, S, n, cudaMemcpyHostToDevice));
  }

  stage("host -> device");
  SymbolTable table;
  if (masks) {
    BuildMaskTable(table.map);
  } else {
    BuildSymbolTable(table.map);
  }
  cudaEvent_t begin, end;
  SBNB_CUDA(cudaEventCreate(&begin));
  SBNB_CUDA(cudaEventCreate(&end));
  struct EventGuard {
    cudaEvent_t a, b;
    ~EventGuard() {
      cudaEventDestroy(a);
      cudaEventDestroy(b);
    }
  } event_guard{begin, end};

  const int site_blocks = static_cast<int>((S + 255) / 256);
  // Test hook: keep only the low bits of the column keys, so that different columns
  // share keys and the verification / rehash path is exercised.
  uint64_t key_mask = ~0ull;
  if (const char* bits = std::getenv("SBNB_DEBUG_PATTERN_KEY_BITS"))
    key_mask = (1ull << std::max(1, std::min(63, std::atoi(bits)))) - 1;
  int64_t pattern_count = 0;
  double device_ms = 0.0;
  bool done = false;
  for (uint64_t seed = 0; seed < 4 && !done; seed++) {
    SBNB_CUDA(cudaMemset(d_total.get() + 1, 0xff, sizeof(unsigned long long)));
    SBNB_CUDA(cudaMemset(d_collided.get(), 0, sizeof(int32_t)));
    SBNB_CUDA(cudaMemset(d_column_counter.get(), 0, sizeof(uint32_t)));
    SBNB_CUDA(cudaMemset(d_table_keys.get(), 0xff, static_cast<size_t>(table_size) * sizeof(uint64_t)));
    SBNB_CUDA(cudaMemset(d_table_first.get(), 0xff, static_cast<size_t>(table_size) * sizeof(uint32_t)));
    SBNB_CUDA(cudaMemset(d_table_count.get(), 0, static_cast<size_t>(table_size) * sizeof(uint32_t)));
    SBNB_CUDA(cudaEventRecord(begin));
    const int64_t groups = pitch / kSitesPerThread;
    (masks ? HashKernel<true> : HashKernel<false>)<<<static_cast<int>((groups + kHashThreads - 1) / kHashThreads),
                                                     kHashThreads>>>(
        d_sequences.get(), d_keys.get(), n, S, pitch, seed * 0x9e3779b97f4a7c15ull, key_mask, table, d_total.get() + 1);
    InsertKernel<<<site_blocks, 256>>>(d_keys.get(), d_table_keys.get(), d_table_first.get(),
                                       d_table_count.get(), d_slot_of.get(), S, table_size - 1);
    FlagKernel<<<site_blocks, 256>>>(d_slot_of.get(), d_table_first.get(), d_flags.get(), S);
    ScanBlocksKernel<<<static_cast<int>(scan_blocks), kScanThreads>>>(d_flags.get(), d_index.get(),
                                                                      d_block_sums.get(), S);
    ScanSumsKernel<<<1, 1024>>>(d_block_sums.get(), scan_blocks, d_total.get());
    // The output rows are written `pitch` apart (the pattern count is not known on
    // the host yet), so the whole pipeline is queued without a round trip.
    EmitKernel<<<static_cast<int>((groups + kHashThreads - 1) / kHashThreads), kHashThreads>>>(
        d_sequences.get(), d_slot_of.get(), d_table_count.get(), d_flags.get(), d_index.get(), d_block_sums.get(),
        d_patterns.get(), d_weights.get(), d_table_pattern.get(), d_table_column.get(), d_column_counter.get(), n, S,
        pitch, table);
    // the contiguous columns of the patterns that repeat, then every repeat held against its
    // pattern's column byte for byte
    TileKernel<false><<<static_cast<int>(pitch / kTileSites), 256>>>(d_sequences.get(), d_slot_of.get(), d_flags.get(),
                                                                     d_table_column.get(), d_columns.get(), n, S, pitch,
                                                                     column_pitch, table, d_collided.get());
    TileKernel<true><<<static_cast<int>(pitch / kTileSites), 256>>>(d_sequences.get(), d_slot_of.get(), d_flags.get(),
                                                                    d_table_column.get(), d_columns.get(), n, S, pitch,
                                                                    column_pitch, table, d_collided.get());
    SBNB_CUDA(cudaEventRecord(end));
    SBNB_CUDA(cudaGetLastError());
    SBNB_CUDA(cudaEventSynchronize(end));
    float ms = 0.f;
    SBNB_CUDA(cudaEventElapsedTime(&ms, begin, end));
    device_ms = ms;
    int32_t collided = 0;
    unsigned long long total[2] = {0, 0};
    SBNB_CUDA(cudaMemcpy(&collided, d_collided.get(), sizeof(collided), cudaMemcpyDeviceToHost));
    SBNB_CUDA(cudaMemcpy(total, d_total.get(), sizeof(total), cudaMemcpyDeviceToHost));
    if (total[1] != ~0ull)
      Fail(SBNB_ERR_INVALID_ARGUMENT, UnknownSymbolMessage(static_cast<uint8_t>(sequences[total[1]])));
    if (collided != 0) continue;  // two different columns shared a 64-bit key: rehash
    pattern_count = static_cast<int64_t>(total[0]);
    done = true;
  }
  if (!done) Fail(SBNB_ERR_CUDA, "Site pattern hashing collided under four seeds.");
  stage("kernels");
  if (pattern_count >= kLongRow) {
    for (int32_t t = 0; t < n; t++)
      SBNB_CUDA(cudaMemcpyAsync(out_patterns + static_cast<size_t>(t) * pattern_count,
                                d_patterns.get() + static_cast<size_t>(t) * pitch, pattern_count,
                                cudaMemcpyDeviceToHost, 0));
    SBNB_CUDA(cudaStreamSynchronize(0));
  } else {
    SBNB_CUDA(cudaMemcpy2D(out_patterns, pattern_count, d_patterns.get(), pitch, pattern_count, n,
                           cudaMemcpyDeviceToHost));
  }
  SBNB_CUDA(cudaMemcpy(out_weights, d_weights.get(), static_cast<size_t>(pattern_count) * sizeof(double),
                       cudaMemcpyDeviceToHost));
  stage("device -> host");
  *out_pattern_count = pattern_count;
  if (out_device_ms) *out_device_ms = device_ms;
}

}  // namespace

}  // namespace sbnb

extern "C" int sbnb_compress_site_patterns(int32_t taxon_count, int64_t site_count, const char* sequences,
                                           int32_t device, uint8_t* out_patterns, double* out_weights,
                                           int64_t* out_pattern_count, double* out_device_ms) {
  return sbnb::Guard([&] {
    sbnb::Compress(taxon_count, site_count, sequences, false, device, out_patterns, out_weights, out_pattern_count,
                   out_device_ms);
  });
}

extern "C" int sbnb_compress_site_patterns_encoded(int32_t taxon_count, int64_t site_count, const char* sequences,
                                                   int32_t tip_encoding, int32_t device, uint8_t* out_patterns,
                                                   double* out_weights, int64_t* out_pattern_count,
                                                   double* out_device_ms) {
  return sbnb::Guard([&] {
    sbnb::Require(tip_encoding == SBNB_TIPS_STATES || tip_encoding == SBNB_TIPS_NUCLEOTIDE_MASKS,
                  "Unknown tip encoding.");
    sbnb::Compress(taxon_count, site_count, sequences, tip_encoding == SBNB_TIPS_NUCLEOTIDE_MASKS, device,
                   out_patterns, out_weights, out_pattern_count, out_device_ms);
  });
}
