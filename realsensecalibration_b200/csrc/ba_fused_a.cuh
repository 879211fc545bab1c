// ba_fused_a.cuh -- Model A (camera, point) hot path, B200-first: two point-tile passes per LM iteration in
// which the residual and the analytic Jacobian never leave the SM.
//
// The materialised-Jacobian pipeline (ba_kernels.cuh, still used for Model B) moves ~1.3 kB per observation
// and iteration through HBM; on a B200 (measured ~6.5 TB/s against ~37 TFLOP/s fp64) recomputing the 2x9
// Jacobian of an observation (~150 flops) is cheaper than re-reading its 160 bytes, and the Schur complement's
// pair products are the only heavy arithmetic.  So:
//
//   pass 1  k_fa_pass1   per tile of points (a window of 480 or 1024 observations, all observations of a point in one
//                        tile), one CTA per tile:
//             A0  one 96-byte tile descriptor; the tile's camera tables (32-bit planes), points and work-item entry
//                 lists -> shared memory by cp.async; first observation / point range / work items -> registers
//             A1  one thread per observation: r, J_e, J_f in registers -> shared-memory record (22 doubles)
//             A2  one thread per point: E^T E, E^T r, LM diagonal, 3x3 Cholesky in registers, z = L^-1 E^T r
//                 (L, 1/diag, z -> shared memory and, as full lines, HBM: 72 B / point); then one thread per
//                 observation: U_i = L^-1 J_e,i^T, w_i = U_i^T z
//             B   one thread per WORK ITEM (a fixed list of <= 16 observation pairs of one camera pair, or <= 16
//                 observations of one camera, all inside the tile; items sorted by length and dealt boustrophedon so
//                 that the lanes of a warp run equally long loops; entries ordered once so that the lanes of a quarter
//                 warp gather from different banks): operands from shared memory, 36 resp. 33 accumulators in
//                 registers, one partial block -> HBM
//             modes: FA_FULL; FA_FIRST (iteration 0, Jacobi scaling inside the pass); FA_GRAD (cost and gradient only,
//                 after the last step of a solve); FA_NORMS (column norms only)
//   reduce  k_reduce_items   fixed-order sum of the partial blocks per camera pair / camera (two levels)
//   pass 2  k_fa_pass2   per tile: r, J again, back-substitution, Ceres' model cost change, candidate point,
//                        candidate cost -- one pass instead of four
//   K1      k_fa_jac     the standalone residual + Jacobian (ba_cuda_eval, generic pipeline) on the same tiles
//
// Every list is static (built once per problem with stable radix sorts) and every sum runs in a fixed order:
// deterministic segmented reduction with shared-memory staging, no floating-point atomics.
// Replaces ReprojectionError + AutoDiff (Test1_BundleAdjustment/bundle_adjustmenter.cpp:106-148) and, inside
// Ceres, SchurEliminator::Eliminate / BackSubstitute.
#pragma once
#include <cuda_pipeline.h>

#include <chrono>
#include <cstdio>

#include "ba_kernels.cuh"
#include "ba_structure.cuh"

namespace ba {

constexpr int FA_TOBS_DEFAULT = 256;         // observation window of a tile (BA_FA_TOBS overrides, for tuning)
constexpr int FA_KMAX = 64;                  // max observations of one point (fused path)
constexpr int FA_TPTS = 4096;                // max points of a tile (a forced cut every FA_TPTS points: keep it rare)
constexpr int FA_TCAM = 48;                  // camera tables staged in shared memory per tile (more: read from L2)
constexpr int FA_CH_PAIR = 16;               // pairs per pair item (BA_FA_CH_PAIR overrides, for tuning)
constexpr int FA_CH_RED = 64;                // partial blocks per first-level reduction chunk
constexpr int FA_NVC = 33;                   // per camera: 21 packed upper F^T F | 6 F^T r | 6 sum of v_i
constexpr int FA_MAX_THREADS = 512;          // launch bound: 1 x 512, 2 x 256 or 4 x 128 threads per SM at <= 128 registers
constexpr int FA_THREADS_DEFAULT = 128;      // BA_FA_THREADS overrides, for tuning
constexpr int FA_REC = 22;                   // doubles per observation record in shared memory (pass 1)
constexpr int FA_REC2 = 10;                  // pass 2
constexpr int FA_PENT_MAX = 6144;            // pair entries staged in shared memory per tile (24 KB)
constexpr size_t FA_SMEM_MAX = 231000;      // dynamic shared memory per CTA (232448 opt-in limit minus the static part)
constexpr int FA_LS = 10;                    // per point in shared memory: L10 L20 L21 | 1/L00 1/L11 1/L22 | z (3) | pad
constexpr int FA_PS2 = 7;                    // pass 2 / k_fa_jac, per point in shared memory: x_e (3, then the candidate) | scale (3) | pad (odd stride)
constexpr int FA_FULL = 0, FA_NORMS = 1, FA_GRAD = 2, FA_FIRST = 3;   // modes of k_fa_pass1
constexpr int FA_JAC_THREADS = 128;          // k_fa_jac: four CTAs per SM
constexpr int FA_RECJ = 18;                  // k_fa_jac: doubles staged per observation (J_e 6 | J_f 12), in a per-warp buffer

// Everything a CTA needs to know about its tile in one 96-byte record (one L2 round trip instead of a chain of
// dependent pointer loads): built once per problem by k_fa_tile_desc.
struct __align__(16) FaTile {
  int64_t pt0, ob0, cam0, pe0, ce0, pitem0, citem0;    // first point / observation / camera-list entry / pair entry / camera entry / items
  int32_t npts, nobs, ncam, npe, nce, npitem, ncitem;  // counts (unclamped)
  int32_t pad_[3];
};
static_assert(sizeof(FaTile) == 96, "FaTile is loaded as six 16-byte words");
static_assert(TAB == 32, "one lane per table field when the tables are staged");


__global__ void k_fa_tile_desc(int n_tiles, const int64_t* __restrict__ tile_pt_ptr, const int64_t* __restrict__ e_ptr,
                               const int64_t* __restrict__ tile_cam_ptr, const int64_t* __restrict__ tile_pent_ptr,
                               const int64_t* __restrict__ tile_cent_ptr, const int64_t* __restrict__ tile_pitem_ptr,
                               const int64_t* __restrict__ tile_citem_ptr, FaTile* __restrict__ out) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_tiles) return;
  const int64_t cap32 = INT32_MAX;
  FaTile T;
  T.pt0 = tile_pt_ptr[t];
  const int64_t pt1 = tile_pt_ptr[t + 1];
  T.ob0 = e_ptr[T.pt0];
  T.npts = (int32_t)(pt1 - T.pt0);
  T.nobs = (int32_t)(e_ptr[pt1] - T.ob0);
  T.cam0 = tile_cam_ptr[t];   T.ncam = (int32_t)min(tile_cam_ptr[t + 1] - T.cam0, cap32);
  T.pe0 = tile_pent_ptr[t];   T.npe = (int32_t)min(tile_pent_ptr[t + 1] - T.pe0, cap32);
  T.ce0 = tile_cent_ptr[t];   T.nce = (int32_t)min(tile_cent_ptr[t + 1] - T.ce0, cap32);
  T.pitem0 = tile_pitem_ptr[t]; T.npitem = (int32_t)min(tile_pitem_ptr[t + 1] - T.pitem0, cap32);
  T.citem0 = tile_citem_ptr[t]; T.ncitem = (int32_t)min(tile_citem_ptr[t + 1] - T.citem0, cap32);
  T.pad_[0] = T.pad_[1] = T.pad_[2] = 0;
  out[t] = T;
}

// The partial blocks of one kind (one per work item) and how they are summed per target, in a fixed order
// (k_reduce_items, then k_reduce_final): the same lists for single tiles and for strips.
struct ReduceList {
  DVec<int32_t> items;          // item ids grouped by target (stable)
  DVec<int64_t> tgt_ptr;        // n_targets + 1 into items
  Chunks ch;                    // chunks over tgt_ptr
  DVec<double> part, red1;      // partial blocks (per item), first-level sums (per chunk)
};

// work items of one kind (pair items or camera items)
struct ItemSet {
  int64_t n_ent = 0;
  int n_items = 0, n_targets = 0, n_groups = 0;
  DVec<int32_t> ent;            // sorted entries (pair: li | lj << 16 ; camera: li)
  DVec<int64_t> item_begin;     // n_items
  DVec<int64_t> item_end;       // n_items
  DVec<int64_t> tile_item_ptr;  // n_tiles + 1
  DVec<int32_t> item_target;    // n_items: destination block / camera
  // groups = distinct (tile, target)
  DVec<int64_t> group_ptr;      // n_groups + 1 into ent
  DVec<int32_t> group_target;   // n_groups
  DVec<int64_t> tile_group_ptr; // n_tiles + 1
};

struct FusedA {
  bool ready = false;
  int n_tiles = 0, tobs = FA_TOBS_DEFAULT, kmax = 0, cap = 0, threads = FA_THREADS_DEFAULT, threads2 = FA_THREADS_DEFAULT, ch_cam = 16, ch_pair = FA_CH_PAIR;
  DVec<int64_t> tile_pt_ptr;    // n_tiles + 1
  DVec<int64_t> tile_pent_ptr;  // n_tiles + 1: the tile's slice of pairs.ent (entries are tile-major)
  DVec<int64_t> tile_cent_ptr;  // n_tiles + 1: the tile's slice of cams.ent
  ItemSet pairs, cams;
  ReduceList red_pairs, red_cams; // over the items' partial blocks
  DVec<uint32_t> ob_meta;       // per observation: local point | camera slot << 16 (k_fa_ob_meta)
  DVec<FaTile> tiles;           // n_tiles descriptors
  DVec<double> camacc, Lz;
  // shared-memory geometry, from the maxima over the tiles of this problem (so that small tiles co-reside on an SM)
  int pts_cap = FA_TPTS;        // points of the fullest tile
  int tcam = FA_TCAM;           // camera tables staged per tile (cameras beyond are read from L2)
  int tcs = FA_TCAM + 1;        // stride of one table field in shared memory (odd: conflict-free staging)
  int pent_cap = 0;             // pair entries staged per tile (entries beyond are read from L2)
  size_t smem1() const {
    return ((size_t)cap * FA_REC + (size_t)pts_cap * FA_LS + (size_t)tcs * TAB) * 8 + ((size_t)pent_cap + cap) * 4 + (size_t)cap * 2;
  }
  size_t smem2() const { return ((size_t)cap * FA_REC2 + (size_t)pts_cap * FA_PS2 + (size_t)tcs * (TAB + 16)) * 8; }
  size_t smemj(int threads) const { return ((size_t)threads * FA_RECJ + (size_t)pts_cap * FA_PS2 + (size_t)tcs * TAB) * 8 + (size_t)cap * 20; }
};

__global__ void k_fa_tile_flags(const int64_t* __restrict__ e_ptr, int64_t ne, int tobs, int32_t* __restrict__ flag, int* __restrict__ kmax) {
  const int64_t pt = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (pt >= ne) return;
  atomicMax(kmax, (int)min(e_ptr[pt + 1] - e_ptr[pt], (int64_t)INT32_MAX));
  int f = 0;
  if (pt > 0) f = (e_ptr[pt] / tobs != e_ptr[pt - 1] / tobs) || (pt / FA_TPTS != (pt - 1) / FA_TPTS);
  flag[pt] = f;
}

// ordered observation pairs of a point, keyed by (tile, destination block)
__global__ void k_fa_pair_fill(const int64_t* __restrict__ e_ptr, const int32_t* __restrict__ ob_f, int64_t ne, int64_t nf,
                               const int64_t* __restrict__ off, const int32_t* __restrict__ tile_of_pt, const int64_t* __restrict__ tile_pt_ptr,
                               const uint64_t* __restrict__ dest_keys, int ndest, const uint64_t* __restrict__ dh_keys,
                               const int32_t* __restrict__ dh_val, uint64_t dh_mask, int dh_shift, uint64_t* __restrict__ keys,
                               int32_t* __restrict__ vals) {
  const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e >= ne) return;
  int64_t o = off[e];
  const int tile = tile_of_pt[e];
  const int64_t ob0 = e_ptr[tile_pt_ptr[tile]];
  for (int64_t i = e_ptr[e]; i < e_ptr[e + 1]; ++i)
    for (int64_t j = e_ptr[e]; j < e_ptr[e + 1]; ++j)
      if (ob_f[i] <= ob_f[j]) {
        const uint64_t fk = (uint64_t)ob_f[i] * nf + ob_f[j];
        const int64_t d = dh_keys ? (int64_t)dh_find(dh_keys, dh_val, dh_mask, dh_shift, fk) : lower_bound_u64(dest_keys, ndest, fk);
        keys[o] = (uint64_t)tile * (uint64_t)ndest + (uint64_t)d;
        vals[o] = (int32_t)(i - ob0) | ((int32_t)(j - ob0) << 16);
        ++o;
      }
}
// the same pairs keyed by (tile, camera slot of i, camera slot of j) in 32 bits (GroupDecode mode 1); one thread per
// observation i (a thread per point walks up to 64^2 pairs alone), output in the same order as k_fa_pair_fill
__global__ void k_fa_pair_fill32(const int64_t* __restrict__ e_ptr, const int32_t* __restrict__ ob_e, const int32_t* __restrict__ ob_f,
                                 int64_t nb, const int64_t* __restrict__ off, const int32_t* __restrict__ tile_of_pt,
                                 const int64_t* __restrict__ tile_pt_ptr, const uint32_t* __restrict__ ob_meta, int sb,
                                 uint32_t* __restrict__ keys, int32_t* __restrict__ vals) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= nb) return;
  const int64_t e = ob_e[i];
  const int64_t b = e_ptr[e], n = e_ptr[e + 1];
  const int32_t fi = ob_f[i];
  int64_t o = off[e];
  for (int64_t ii = b; ii < i; ++ii) {   // pairs of the earlier observations of this point
    const int32_t f = ob_f[ii];
    for (int64_t j = b; j < n; ++j) o += (f <= ob_f[j]) ? 1 : 0;
  }
  const uint32_t tile = (uint32_t)tile_of_pt[e];
  const int64_t ob0 = e_ptr[tile_pt_ptr[tile]];
  const uint32_t head = (tile << (2 * sb)) | ((ob_meta[i] >> 16) << sb);
  for (int64_t j = b; j < n; ++j)
    if (fi <= ob_f[j]) {
      keys[o] = head | (ob_meta[j] >> 16);
      vals[o] = (int32_t)(i - ob0) | ((int32_t)(j - ob0) << 16);
      ++o;
    }
}
__global__ void k_fa_max_diff(int n, const int64_t* __restrict__ ptr, int* __restrict__ out) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) atomicMax(out, (int)min(ptr[t + 1] - ptr[t], (int64_t)INT32_MAX));
}
__global__ void k_fa_cam_fill(const int32_t* __restrict__ ob_e, const int32_t* __restrict__ ob_f, int64_t nb, int64_t nf,
                              const int64_t* __restrict__ e_ptr, const int32_t* __restrict__ tile_of_pt, const int64_t* __restrict__ tile_pt_ptr,
                              uint64_t* __restrict__ keys, int32_t* __restrict__ vals) {
  const int64_t o = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (o >= nb) return;
  const int tile = tile_of_pt[ob_e[o]];
  keys[o] = (uint64_t)tile * (uint64_t)nf + (uint64_t)ob_f[o];
  vals[o] = (int32_t)(o - e_ptr[tile_pt_ptr[tile]]);
}
// How a group key splits into (tile, target).  mode 0: key = tile * n_targets + target (64-bit keys).  mode 1 (pair items
// when the camera slots of a tile fit sb bits): key = tile << 2 sb | slot_i << sb | slot_j in 32 bits -- two thirds of the
// sort traffic and one radix pass less on the 144 M pair entries of the 30 M-observation problem; the destination block
// is then looked up once per GROUP (camera pair of the tile) instead of once per pair.
struct GroupDecode {
  int mode = 0, sb = 0, key_bits = 64;
  uint64_t n_targets = 1, nf = 0;
  const int64_t* tile_cam_ptr = nullptr;
  const int32_t* tile_cams = nullptr;
  const uint64_t* dh_keys = nullptr;
  const int32_t* dh_val = nullptr;
  uint64_t dh_mask = 0;
  int dh_shift = 0;
};
template <typename K>
__global__ void k_fa_group_meta(int ng, const K* __restrict__ group_key, GroupDecode D, int32_t* __restrict__ group_target,
                                int32_t* __restrict__ group_tile) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= ng) return;
  const uint64_t key = (uint64_t)group_key[g];
  if (D.mode == 0) {
    group_target[g] = (int32_t)(key % D.n_targets);
    group_tile[g] = (int32_t)(key / D.n_targets);
  } else {
    const uint64_t m = ((uint64_t)1 << D.sb) - 1;
    const int tile = (int)(key >> (2 * D.sb));
    const int64_t c0 = D.tile_cam_ptr[tile];
    const uint64_t ci = (uint64_t)D.tile_cams[c0 + (int64_t)((key >> D.sb) & m)], cj = (uint64_t)D.tile_cams[c0 + (int64_t)(key & m)];
    group_target[g] = dh_find(D.dh_keys, D.dh_val, D.dh_mask, D.dh_shift, ci * D.nf + cj);
    group_tile[g] = tile;
  }
}
// per item: end, target, and the key (tile, descending length) the items are re-ordered by
__global__ void k_fa_item_meta(int n_items, const int32_t* __restrict__ seg, const int64_t* __restrict__ begin, int ch,
                               const int64_t* __restrict__ group_ptr, const int32_t* __restrict__ group_target,
                               const int32_t* __restrict__ group_tile, int64_t* __restrict__ item_end, int32_t* __restrict__ item_target,
                               uint64_t* __restrict__ sort_key) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_items) return;
  const int g = seg[i];
  const int64_t end = min(begin[i] + ch, group_ptr[g + 1]);
  item_end[i] = end;
  item_target[i] = group_target[g];
  sort_key[i] = (uint64_t)group_tile[g] * 64u + (uint64_t)(63 - min((int)(end - begin[i]), 63));
}
template <typename T>
__global__ void k_fa_gather(const T* __restrict__ src, const int32_t* __restrict__ perm, int n, T* __restrict__ dst) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = src[perm[i]];
}
__global__ void k_fa_key_tile(const uint64_t* __restrict__ key, int n, int32_t* __restrict__ tile) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) tile[i] = (int32_t)(key[i] / 64u);
}
__global__ void k_fa_group_tile(int n_tiles, const int64_t* __restrict__ tile_group_ptr, int32_t* __restrict__ group_tile) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_tiles) return;
  for (int64_t g = tile_group_ptr[t]; g < tile_group_ptr[t + 1]; ++g) group_tile[g] = t;
}
// per observation: local point index inside its tile (low 16 bits) | slot of its camera in the tile's camera list
// (= rank of its (tile, camera) group in the tile; high 16 bits): everything pass 1 / pass 2 / k_fa_jac need to know
// about an observation besides its image point, in one 4-byte load
__global__ void k_fa_ob_meta(int ng, const int64_t* __restrict__ group_ptr, const int32_t* __restrict__ group_tile,
                             const int64_t* __restrict__ tile_group_ptr, const int32_t* __restrict__ ent, const int64_t* __restrict__ e_ptr,
                             const int64_t* __restrict__ tile_pt_ptr, const int32_t* __restrict__ ob_e, uint32_t* __restrict__ ob_meta) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= ng) return;
  const int tile = group_tile[g];
  const int64_t pt0 = tile_pt_ptr[tile];
  const int64_t ob0 = e_ptr[pt0];
  const uint32_t slot = (uint32_t)min((int64_t)65535, (int64_t)g - tile_group_ptr[tile]);
  for (int64_t q = group_ptr[g]; q < group_ptr[g + 1]; ++q) {
    const int64_t o = ob0 + ent[q];
    ob_meta[o] = (uint32_t)(ob_e[o] - pt0) | (slot << 16);
  }
}

// per tile: slice of an entry list (entries are sorted tile-major, groups are tile-major) and the maxima the
// shared-memory geometry is sized by; stat = {max points, max cameras, max pair entries}
__global__ void k_fa_tile_ent_ptr(int n_tiles, const int64_t* __restrict__ tile_group_ptr, const int64_t* __restrict__ group_ptr,
                                  int64_t* __restrict__ tile_ent_ptr) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t <= n_tiles) tile_ent_ptr[t] = group_ptr[tile_group_ptr[t]];
}
__global__ void k_fa_tile_stats(int n_tiles, const int64_t* __restrict__ tile_pt_ptr, const int64_t* __restrict__ tile_cam_ptr,
                                const int64_t* __restrict__ tile_pent_ptr, int* __restrict__ stat) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_tiles) return;
  atomicMax(stat + 0, (int)(tile_pt_ptr[t + 1] - tile_pt_ptr[t]));
  atomicMax(stat + 1, (int)(tile_cam_ptr[t + 1] - tile_cam_ptr[t]));
  atomicMax(stat + 2, (int)min(tile_pent_ptr[t + 1] - tile_pent_ptr[t], (int64_t)INT32_MAX));
}

struct FaLap {  // BA_CUDA_TIMING=2: wall clock of the build phases on stderr (synchronises the stream at every lap)
  cudaStream_t st;
  bool on;
  std::chrono::steady_clock::time_point t;
  explicit FaLap(cudaStream_t s) : st(s), t(std::chrono::steady_clock::now()) {
    const char* e = std::getenv("BA_CUDA_TIMING");
    on = e && std::atoi(e) >= 2;
  }
  void lap(const char* what) {
    if (!on) return;
    cudaStreamSynchronize(st);
    const auto n = std::chrono::steady_clock::now();
    std::fprintf(stderr, "[ba_cuda timing]   fused: %-24s %9.3f ms\n", what, 1e3 * std::chrono::duration<double>(n - t).count());
    t = n;
  }
};

inline int env_int(const char* name, int lo, int hi, int fallback) {
  if (const char* env = std::getenv(name)) { const int v = std::atoi(env); if (v >= lo && v <= hi) return v; }
  return fallback;
}

// Bank-aware order of the entries inside the work items.  In phase B of pass 1 the eight lanes of a quarter warp
// gather 16-byte pieces of eight different observation records; two records whose indices agree modulo 8 sit in the
// same banks (record stride 22 doubles = 11 x 16 B), and with entries in arbitrary order 60 % of the shared-memory
// wavefronts of the kernel were such replays (ncu, profiles/).  The order of the entries inside an item is free, so
// for every eight items that share a quarter warp (consecutive item indices of a tile) the entries are permuted
// greedily: in step t the lanes pick, in turn, a remaining entry whose record classes are still unused in that step.
// One warp per tile, lane = group of eight items.  Static, so the sums stay in a fixed order.
__global__ void k_fa_bank_order(int n_tiles, const int64_t* __restrict__ tile_item_ptr, const int64_t* __restrict__ item_begin,
                                const int64_t* __restrict__ item_end, int32_t* __restrict__ ent, int is_pair) {
  const int tile = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (tile >= n_tiles) return;
  const int64_t i0 = tile_item_ptr[tile], i1 = tile_item_ptr[tile + 1];
  const int full = is_pair ? 2 : 1;
  for (int64_t g0 = i0 + 8 * lane; g0 < i1; g0 += 8 * 32) {
    int64_t b[8];
    int len[8], maxlen = 0;
#pragma unroll
    for (int l = 0; l < 8; ++l) {
      const bool on = g0 + l < i1;
      b[l] = on ? item_begin[g0 + l] : 0;
      len[l] = on ? (int)(item_end[g0 + l] - b[l]) : 0;
      maxlen = max(maxlen, len[l]);
    }
    for (int t = 0; t < maxlen; ++t) {
      unsigned used_i = 0, used_j = 0;
#pragma unroll
      for (int l = 0; l < 8; ++l) {
        if (t >= len[l]) continue;
        int32_t* E = ent + b[l];
        int best = t, best_score = -1;
        for (int c = t; c < len[l] && best_score < full; ++c) {
          const int32_t e = E[c];
          int score = ((used_i >> (e & 7)) & 1) ? 0 : 1;
          if (is_pair) score += ((used_j >> ((e >> 16) & 7)) & 1) ? 0 : 1;
          if (score > best_score) { best_score = score; best = c; }
        }
        const int32_t e = E[best];
        if (best != t) { E[best] = E[t]; E[t] = e; }
        used_i |= 1u << (e & 7);
        if (is_pair) used_j |= 1u << ((e >> 16) & 7);
      }
    }
  }
}

// keys (tile * n_targets + target) with their entries -> sorted entries, groups, items of <= ch entries ordered by
// (tile, descending length), the reduction lists R over the items
template <typename K>
inline int build_items(ItemSet& I, ReduceList& R, DVec<K>& keys, DVec<int32_t>& vals, int64_t n, int n_tiles, int64_t n_targets, int ch,
                       bool is_pair, const GroupDecode& D, cudaStream_t st) {
  I.n_ent = n; I.n_targets = (int)n_targets;
  FaLap L(st);
  DVec<K> ks, gkey;
  DVec<int64_t> gcnt;
  DVec<int32_t> nruns, group_tile;
  BA_TRY(ks.alloc(n)); BA_TRY(I.ent.alloc(n));
  if (n > 0)
    BA_TRY(cub_call([&](void* t, size_t& b) {
      return cub::DeviceRadixSort::SortPairs(t, b, keys.p, ks.p, vals.p, I.ent.p, (int)n, 0, D.key_bits, st);
    }));
  keys.release(); vals.release();
  L.lap("items: sort entries");
  BA_TRY(gkey.alloc(n)); BA_TRY(gcnt.alloc(n + 1)); BA_TRY(nruns.alloc(1));
  int32_t ng = 0;
  if (n > 0) {
    BA_TRY(cub_call([&](void* t, size_t& b) { return cub::DeviceRunLengthEncode::Encode(t, b, ks.p, gkey.p, gcnt.p, nruns.p, (int)n, st); }));
    BA_CUDA_TRY(cudaMemcpyAsync(&ng, nruns.p, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    BA_CUDA_TRY(cudaStreamSynchronize(st));
  }
  ks.release();
  I.n_groups = ng;
  BA_TRY(I.group_ptr.alloc(ng + 1)); BA_TRY(I.group_target.alloc(ng)); BA_TRY(group_tile.alloc(ng));
  BA_CUDA_TRY(cudaMemsetAsync(gcnt.p + ng, 0, sizeof(int64_t), st));
  BA_TRY(cub_call([&](void* t, size_t& b) { return cub::DeviceScan::ExclusiveSum(t, b, gcnt.p, I.group_ptr.p, ng + 1, st); }));
  k_fa_group_meta<K><<<grid_for(ng, 256), 256, 0, st>>>(ng, gkey.p, D, I.group_target.p, group_tile.p);
  BA_TRY(I.tile_group_ptr.alloc((size_t)n_tiles + 1));
  k_seg_ptr<int32_t><<<grid_for(ng > n_tiles + 1 ? ng : n_tiles + 1, 256), 256, 0, st>>>(group_tile.p, ng, n_tiles, I.tile_group_ptr.p);
  L.lap("items: groups");
  Chunks C;
  BA_TRY(build_chunks(C, I.group_ptr.p, ng, ch, st));
  L.lap("items: chunks");
  const int ni = C.n;
  I.n_items = ni;
  DVec<int64_t> end0;
  DVec<int32_t> tgt0, perm, iota, item_tile;
  DVec<uint64_t> skey, skey_sorted;
  BA_TRY(end0.alloc(ni)); BA_TRY(tgt0.alloc(ni)); BA_TRY(skey.alloc(ni)); BA_TRY(skey_sorted.alloc(ni)); BA_TRY(perm.alloc(ni));
  BA_TRY(iota.alloc(ni)); BA_TRY(item_tile.alloc(ni));
  k_fa_item_meta<<<grid_for(ni, 256), 256, 0, st>>>(ni, C.seg.p, C.begin.p, ch, I.group_ptr.p, I.group_target.p, group_tile.p, end0.p, tgt0.p, skey.p);
  k_iota<<<grid_for(ni, 256), 256, 0, st>>>(iota.p, ni, 0);
  if (ni > 0)
    BA_TRY(cub_call([&](void* t, size_t& b) {
      return cub::DeviceRadixSort::SortPairs(t, b, skey.p, skey_sorted.p, iota.p, perm.p, ni, 0, bits_for((uint64_t)n_tiles * 64u), st);
    }));
  BA_TRY(I.item_begin.alloc(ni)); BA_TRY(I.item_end.alloc(ni)); BA_TRY(I.item_target.alloc(ni));
  k_fa_gather<int64_t><<<grid_for(ni, 256), 256, 0, st>>>(C.begin.p, perm.p, ni, I.item_begin.p);
  k_fa_gather<int64_t><<<grid_for(ni, 256), 256, 0, st>>>(end0.p, perm.p, ni, I.item_end.p);
  k_fa_gather<int32_t><<<grid_for(ni, 256), 256, 0, st>>>(tgt0.p, perm.p, ni, I.item_target.p);
  k_fa_key_tile<<<grid_for(ni, 256), 256, 0, st>>>(skey_sorted.p, ni, item_tile.p);
  BA_TRY(I.tile_item_ptr.alloc((size_t)n_tiles + 1));
  k_seg_ptr<int32_t><<<grid_for(ni > n_tiles + 1 ? ni : n_tiles + 1, 256), 256, 0, st>>>(item_tile.p, ni, n_tiles, I.tile_item_ptr.p);
  L.lap("items: sort items");
  if (env_int("BA_FA_BANK_ORDER", 0, 1, 1))
    k_fa_bank_order<<<grid_for(n_tiles, 4), 128, 0, st>>>(n_tiles, I.tile_item_ptr.p, I.item_begin.p, I.item_end.p, I.ent.p, is_pair ? 1 : 0);
  L.lap("items: bank order");
  BA_TRY(sort_to_csr(I.item_target.p, iota.p, ni, n_targets, R.tgt_ptr, R.items, st));
  BA_TRY(build_chunks(R.ch, R.tgt_ptr.p, (int)n_targets, FA_CH_RED, st));
  L.lap("items: reduction lists");
  BA_CUDA_TRY(cudaStreamSynchronize(st));
  BA_CUDA_TRY(cudaGetLastError());
  return BA_OK;
}

// Returns BA_ERR_UNSUPPORTED when the problem does not fit the fused path (a point with more than FA_KMAX
// observations, or nothing to do): the caller then keeps the generic pipeline.
inline int build_fused_a_tobs(FusedA& F, const Structure& S, cudaStream_t st, int tobs);

// Tile geometry: measured on B200 (profiles/README.md), a problem whose points carry many observation pairs
// (cfg5: 4.8 pairs per observation) wants the largest tile shared memory can hold (the partial blocks written per
// work item, 288 B each, are what the kernel pays for in HBM) and 512 threads on it; a sparse one (cfg4: 3 pairs
// per observation) runs best on 480-observation tiles, two CTAs of 256 threads per SM.  BA_FA_TOBS / BA_FA_THREADS /
// BA_FA_THREADS2 / BA_FA_CH_CAM override, for tuning.  A geometry that does not fit is retried at half the tile.
inline int build_fused_a(FusedA& F, const Structure& S, cudaStream_t st) {
  F.ready = false;
  if (S.ne == 0 || S.nb == 0 || S.nslots != 1) return BA_ERR_UNSUPPORTED;
  const int64_t np = S.npairs - S.nf;   // ordered incidence pairs, counted when the structure was built
  if (np >= (int64_t)INT32_MAX) return BA_ERR_UNSUPPORTED;
  const bool dense_pairs = (double)np >= 4.0 * (double)S.nb;
  int tobs = env_int("BA_FA_TOBS", 64, 1024, dense_pairs ? 1024 : 480);
  for (;; tobs /= 2) {
    F.threads = env_int("BA_FA_THREADS", 32, FA_MAX_THREADS, tobs >= 768 ? 512 : 256) / 32 * 32;
    F.threads2 = env_int("BA_FA_THREADS2", 32, FA_MAX_THREADS, tobs >= 768 ? 256 : 128) / 32 * 32;
    F.ch_cam = env_int("BA_FA_CH_CAM", 1, 63, 16);
    F.ch_pair = env_int("BA_FA_CH_PAIR", 1, 63, dense_pairs ? FA_CH_PAIR : 12);  // measured: cfg4 12, cfg5 16
    const int rc = build_fused_a_tobs(F, S, st, tobs);
    if (rc != BA_ERR_UNSUPPORTED || tobs <= 128 || F.kmax > FA_KMAX) return rc;
  }
}

inline int build_fused_a_tobs(FusedA& F, const Structure& S, cudaStream_t st, int tobs) {
  F.ready = false;
  const int64_t ne = S.ne, nb = S.nb, nf = S.nf;
  F.tobs = tobs;
  FaLap L(st);
  DVec<int32_t> flag, tile_of_pt;
  DVec<int> kmax;
  BA_TRY(flag.alloc(ne)); BA_TRY(tile_of_pt.alloc(ne)); BA_TRY(kmax.alloc_zero(1, st));
  k_fa_tile_flags<<<grid_for(ne, 256), 256, 0, st>>>(S.e_ptr.p, ne, F.tobs, flag.p, kmax.p);
  BA_TRY(cub_call([&](void* t, size_t& b) { return cub::DeviceScan::InclusiveSum(t, b, flag.p, tile_of_pt.p, (int)ne, st); }));
  int last_tile = 0;
  BA_CUDA_TRY(cudaMemcpyAsync(&F.kmax, kmax.p, sizeof(int), cudaMemcpyDeviceToHost, st));
  BA_CUDA_TRY(cudaMemcpyAsync(&last_tile, tile_of_pt.p + (ne - 1), sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  BA_CUDA_TRY(cudaStreamSynchronize(st));
  if (F.kmax > FA_KMAX) return BA_ERR_UNSUPPORTED;
  F.cap = F.tobs + F.kmax;
  F.n_tiles = last_tile + 1;
  BA_TRY(F.tile_pt_ptr.alloc((size_t)F.n_tiles + 1));
  k_seg_ptr<int32_t><<<grid_for(ne > F.n_tiles + 1 ? ne : F.n_tiles + 1, 256), 256, 0, st>>>(tile_of_pt.p, ne, F.n_tiles, F.tile_pt_ptr.p);
  L.lap("tiles");
  // camera items, the tile camera lists and the per-observation word (local point | camera slot)
  int max_tile_cams = 0;
  {
    DVec<uint64_t> keys;
    DVec<int32_t> vals, group_tile;
    DVec<int> mx;
    BA_TRY(keys.alloc(nb)); BA_TRY(vals.alloc(nb)); BA_TRY(mx.alloc_zero(1, st));
    k_fa_cam_fill<<<grid_for(nb, 256), 256, 0, st>>>(S.ob_e.p, S.ob_f0.p, nb, nf, S.e_ptr.p, tile_of_pt.p, F.tile_pt_ptr.p, keys.p, vals.p);
    GroupDecode D;
    D.n_targets = (uint64_t)nf; D.key_bits = bits_for((uint64_t)F.n_tiles * (uint64_t)nf);
    BA_TRY(build_items<uint64_t>(F.cams, F.red_cams, keys, vals, nb, F.n_tiles, nf, F.ch_cam, false, D, st));
    const int ng = F.cams.n_groups;
    BA_TRY(group_tile.alloc(ng)); BA_TRY(F.ob_meta.alloc(nb));
    // group -> tile from the tile_group_ptr CSR (groups are tile-major)
    k_fa_group_tile<<<grid_for(F.n_tiles, 256), 256, 0, st>>>(F.n_tiles, F.cams.tile_group_ptr.p, group_tile.p);
    k_fa_ob_meta<<<grid_for(ng, 256), 256, 0, st>>>(ng, F.cams.group_ptr.p, group_tile.p, F.cams.tile_group_ptr.p, F.cams.ent.p, S.e_ptr.p,
                                                    F.tile_pt_ptr.p, S.ob_e.p, F.ob_meta.p);
    k_fa_max_diff<<<grid_for(F.n_tiles, 256), 256, 0, st>>>(F.n_tiles, F.cams.tile_group_ptr.p, mx.p);
    BA_CUDA_TRY(cudaMemcpyAsync(&max_tile_cams, mx.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    BA_CUDA_TRY(cudaStreamSynchronize(st));
  }
  L.lap("camera items");
  // pair items
  {
    DVec<int64_t> cnt, off;
    BA_TRY(cnt.alloc(ne + 1)); BA_TRY(off.alloc(ne + 1));
    k_pair_count<<<grid_for(ne + 1, 128), 128, 0, st>>>(S.e_ptr.p, S.ob_f0.p, ne, cnt.p);
    BA_TRY(cub_call([&](void* t, size_t& b) { return cub::DeviceScan::ExclusiveSum(t, b, cnt.p, off.p, (int)(ne + 1), st); }));
    int64_t np = 0;
    BA_CUDA_TRY(cudaMemcpyAsync(&np, off.p + ne, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    BA_CUDA_TRY(cudaStreamSynchronize(st));
    if (np >= (int64_t)INT32_MAX) return BA_ERR_UNSUPPORTED;
    DVec<int32_t> vals;
    BA_TRY(vals.alloc(np));
    const int sb = bits_for((uint64_t)std::max(max_tile_cams - 1, 1));
    const int tb = bits_for((uint64_t)std::max(F.n_tiles - 1, 1));
    GroupDecode D;
    D.n_targets = (uint64_t)S.ndest; D.nf = (uint64_t)nf;
    if (S.dh_keys.n && 2 * sb + tb <= 32 && env_int("BA_FA_KEY32", 0, 1, 1)) {   // 32-bit keys (tile, camera slot i, camera slot j)
      DVec<uint32_t> keys;
      BA_TRY(keys.alloc(np));
      k_fa_pair_fill32<<<grid_for(nb, 256), 256, 0, st>>>(S.e_ptr.p, S.ob_e.p, S.ob_f0.p, nb, off.p, tile_of_pt.p, F.tile_pt_ptr.p, F.ob_meta.p,
                                                          sb, keys.p, vals.p);
      L.lap("pair fill (32-bit keys)");
      D.mode = 1; D.sb = sb; D.key_bits = 2 * sb + tb;
      D.tile_cam_ptr = F.cams.tile_group_ptr.p; D.tile_cams = F.cams.group_target.p;
      D.dh_keys = S.dh_keys.p; D.dh_val = S.dh_val.p; D.dh_mask = S.dh_mask; D.dh_shift = S.dh_shift;
      BA_TRY(build_items<uint32_t>(F.pairs, F.red_pairs, keys, vals, np, F.n_tiles, S.ndest, F.ch_pair, true, D, st));
    } else {
      DVec<uint64_t> keys;
      BA_TRY(keys.alloc(np));
      k_fa_pair_fill<<<grid_for(ne, 128), 128, 0, st>>>(S.e_ptr.p, S.ob_f0.p, ne, nf, off.p, tile_of_pt.p, F.tile_pt_ptr.p, S.dest_keys.p,
                                                        S.ndest, S.dh_keys.n ? S.dh_keys.p : nullptr, S.dh_val.p, S.dh_mask, S.dh_shift, keys.p,
                                                        vals.p);
      L.lap("pair fill");
      D.key_bits = bits_for((uint64_t)F.n_tiles * (uint64_t)S.ndest);
      BA_TRY(build_items<uint64_t>(F.pairs, F.red_pairs, keys, vals, np, F.n_tiles, S.ndest, F.ch_pair, true, D, st));
    }
  }
  {  // per-tile slices of the entry lists; shared-memory geometry from the fullest tile
    const int nt = F.n_tiles;
    BA_TRY(F.tile_pent_ptr.alloc((size_t)nt + 1)); BA_TRY(F.tile_cent_ptr.alloc((size_t)nt + 1));
    k_fa_tile_ent_ptr<<<grid_for(nt + 1, 256), 256, 0, st>>>(nt, F.pairs.tile_group_ptr.p, F.pairs.group_ptr.p, F.tile_pent_ptr.p);
    k_fa_tile_ent_ptr<<<grid_for(nt + 1, 256), 256, 0, st>>>(nt, F.cams.tile_group_ptr.p, F.cams.group_ptr.p, F.tile_cent_ptr.p);
    DVec<int> stat;
    BA_TRY(stat.alloc_zero(3, st));
    k_fa_tile_stats<<<grid_for(nt, 256), 256, 0, st>>>(nt, F.tile_pt_ptr.p, F.cams.tile_group_ptr.p, F.tile_pent_ptr.p, stat.p);
    int h[3] = {0, 0, 0};
    BA_CUDA_TRY(cudaMemcpyAsync(h, stat.p, sizeof(h), cudaMemcpyDeviceToHost, st));
    BA_CUDA_TRY(cudaStreamSynchronize(st));
    F.pts_cap = std::max(1, std::min(h[0], FA_TPTS));
    F.tcam = std::max(1, std::min(h[1], FA_TCAM));
    F.tcs = F.tcam | 1;
    F.pent_cap = std::min(h[2], FA_PENT_MAX);
    F.pent_cap += F.pent_cap & 1;  // keeps the int32 areas 8-byte sized
    if (F.smem1() > FA_SMEM_MAX) {   // stage fewer pair entries (the rest is read from L2) before giving up
      const size_t excess = (F.smem1() - FA_SMEM_MAX + 7) / 8 * 2;
      F.pent_cap = (size_t)F.pent_cap > excess ? F.pent_cap - (int)excess : 0;
    }
    if (F.smem1() > FA_SMEM_MAX || F.smem2() > FA_SMEM_MAX || F.smemj(FA_JAC_THREADS) > FA_SMEM_MAX) return BA_ERR_UNSUPPORTED;
  }
  L.lap("pair items, geometry");
  BA_TRY(F.tiles.alloc((size_t)F.n_tiles));
  k_fa_tile_desc<<<grid_for(F.n_tiles, 256), 256, 0, st>>>(F.n_tiles, F.tile_pt_ptr.p, S.e_ptr.p, F.cams.tile_group_ptr.p, F.tile_pent_ptr.p,
                                                          F.tile_cent_ptr.p, F.pairs.tile_item_ptr.p, F.cams.tile_item_ptr.p, F.tiles.p);
  BA_TRY(F.red_pairs.part.alloc((size_t)F.pairs.n_items * 36)); BA_TRY(F.red_cams.part.alloc((size_t)F.cams.n_items * FA_NVC));
  BA_TRY(F.red_pairs.red1.alloc((size_t)F.red_pairs.ch.n * 36)); BA_TRY(F.red_cams.red1.alloc((size_t)F.red_cams.ch.n * FA_NVC));
  BA_TRY(F.camacc.alloc((size_t)nf * FA_NVC + 2 + 64));  // tail: shard-local gradient scalars (ba_cuda.cu, kMaxWorld)
  BA_TRY(F.Lz.alloc((size_t)ne * 9));
  BA_CUDA_TRY(cudaStreamSynchronize(st));
  BA_CUDA_TRY(cudaGetLastError());
  F.ready = true;
  return BA_OK;
}

// ---------------------------------------------------------------------------------------
// residual + Jacobian of one Model A observation (the arithmetic of k_jac_a)
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ void fa_linearize(const double* __restrict__ T, const double* X, const double* s, double2 ob, double* r,
                                             double* je, double* jf) {
  double q[3];
  mat3_vec(T, X, q);
  const double p0 = q[0] + T[18], p1 = q[1] + T[19], p2 = q[2] + T[20];
  r[0] = T[21] * p0 / p2 + T[23] - ob.x;
  r[1] = T[22] * p1 / p2 + T[24] - ob.y;
  const double iz = 1.0 / p2;
  const double a = T[21] * iz, bb = -T[21] * p0 * iz * iz, cc = T[22] * iz, dd = -T[22] * p1 * iz * iz;
  double D[9];
  rot_deriv(T + 9, T[25] != 0.0 ? X : q, D);
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    jf[k] = (a * D[k] + bb * D[6 + k]) * T[26 + k];
    jf[6 + k] = (cc * D[3 + k] + dd * D[6 + k]) * T[26 + k];
  }
  jf[3] = a * T[29]; jf[4] = 0.0;        jf[5] = bb * T[31];
  jf[9] = 0.0;       jf[10] = cc * T[30]; jf[11] = dd * T[31];
  je[0] = (a * T[0] + bb * T[6]) * s[0]; je[1] = (a * T[1] + bb * T[7]) * s[1]; je[2] = (a * T[2] + bb * T[8]) * s[2];
  je[3] = (cc * T[3] + dd * T[6]) * s[0]; je[4] = (cc * T[4] + dd * T[7]) * s[1]; je[5] = (cc * T[5] + dd * T[8]) * s[2];
}

// 3x3 Cholesky with reciprocal diagonal: Lp = {L10, L20, L21, 1/L00, 1/L11, 1/L22}; M symmetric, upper part read
__device__ __forceinline__ bool fa_chol3(const double* M /* m00 m01 m02 m11 m12 m22 */, double* Lp) {
  const double d0 = M[0];
  if (!(d0 > 0.0) || !isfinite(d0)) return false;
  const double i0 = rsqrt(d0);
  const double l10 = M[1] * i0, l20 = M[2] * i0;
  const double d1 = M[3] - l10 * l10;
  if (!(d1 > 0.0) || !isfinite(d1)) return false;
  const double i1 = rsqrt(d1);
  const double l21 = (M[4] - l20 * l10) * i1;
  const double d2 = M[5] - l20 * l20 - l21 * l21;
  if (!(d2 > 0.0) || !isfinite(d2)) return false;
  Lp[0] = l10; Lp[1] = l20; Lp[2] = l21; Lp[3] = i0; Lp[4] = i1; Lp[5] = rsqrt(d2);
  return true;
}
__device__ __forceinline__ void fa_fwd3(const double* Lp, double* x) {  // x <- L^-1 x
  x[0] *= Lp[3];
  x[1] = (x[1] - Lp[0] * x[0]) * Lp[4];
  x[2] = (x[2] - Lp[1] * x[0] - Lp[2] * x[1]) * Lp[5];
}
__device__ __forceinline__ void fa_bwd3(const double* Lp, double* x) {  // x <- L^-T x
  x[2] *= Lp[5];
  x[1] = (x[1] - Lp[2] * x[2]) * Lp[4];
  x[0] = (x[0] - Lp[0] * x[1] - Lp[1] * x[2]) * Lp[3];
}

struct FaParams {
  // structure
  const FaTile* tiles;
  const int64_t* e_ptr; const int32_t* ob_f; const uint32_t* ob_meta; const double2* uv;
  const int32_t* tile_cams;
  const int64_t* pitem_begin; const int64_t* pitem_end; const int32_t* pent;
  const int64_t* citem_begin; const int64_t* citem_end; const int32_t* cent;
  int cap, pts_cap, tcam, tcs, pent_cap;
  // state
  const double* xe; const double* se; const double* tab_f; const double* radius;
  double min_diag, max_diag;
  // pass 1 outputs
  double* partP; double* partC; double* Lz; double* se_out;
  double* cost_partial; double* gmax_partial; double* g2_partial;
  // pass 2 inputs / outputs
  const double* yf; const double* tabc_f; double* xe_c;
  double* mcc_partial; double* x2_partial; double* d2_partial; double* cand_partial;
  // standalone residual + Jacobian (k_fa_jac)
  double* RES; double* JE; double* JF;
  int* status;
  LossSpec loss;   // robust loss on every observation (type 0 = none, the reference)
};

// Ceres' Corrector on one observation: r, J_e, J_f scaled by sqrt(rho'(|r|^2)); returns the cost term rho
__device__ __forceinline__ double fa_apply_loss(const LossSpec L, double* r, double* je, double* jf) {
  const double s = r[0] * r[0] + r[1] * r[1];
  if (L.type == 0) return s;
  double rho, w;
  loss_apply(L, s, &rho, &w);
  r[0] *= w; r[1] *= w;
#pragma unroll
  for (int k = 0; k < 6; ++k) je[k] *= w;
#pragma unroll
  for (int k = 0; k < 12; ++k) jf[k] *= w;
  return rho;
}

__device__ __forceinline__ FaTile fa_load_tile(const FaTile* __restrict__ p) {
  FaTile T;
  const int4* s = reinterpret_cast<const int4*>(p);
  int4* d = reinterpret_cast<int4*>(&T);
#pragma unroll
  for (int k = 0; k < 6; ++k) d[k] = __ldg(s + k);
  return T;
}

// The tile's camera tables -> shared memory as 32-bit planes [2 * field + half][slot]: a thread reads field f of ITS
// camera with two 4-byte loads, and the lanes of a warp (different cameras of the tile) then hit different banks for
// up to 32 slots; as 8-byte words only 16 slots are conflict free and the table reads replayed 1.9x (ncu).
// One warp per camera row: the (uniform) camera ids of four rows are fetched first, then lane f copies field f of
// each row with two 4-byte cp.async, so nothing of this waits in a register; the caller commits and waits on the
// pipeline.  nfields <= 32; field_map = nullptr copies fields 0 .. nfields-1.
__device__ __forceinline__ void fa_stage_tables_async(const FaParams& P, const FaTile& T, const double* __restrict__ tab, double* tabs,
                                                      int nfields, const int* field_map) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const int ncam = min(T.ncam, P.tcam);
  const int src_f = lane < nfields ? (field_map ? field_map[lane] : lane) : 0;
  uint32_t* planes = reinterpret_cast<uint32_t*>(tabs);
  for (int s0 = warp; s0 < ncam; s0 += 4 * nw) {
    int32_t cam[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) { const int s = s0 + u * nw; cam[u] = s < ncam ? __ldg(P.tile_cams + T.cam0 + s) : -1; }
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (cam[u] >= 0 && lane < nfields) {
        const uint32_t* src = reinterpret_cast<const uint32_t*>(tab + (int64_t)TAB * cam[u] + src_f);
        uint32_t* dst = planes + (size_t)(2 * lane) * P.tcs + (s0 + u * nw);
        __pipeline_memcpy_async(dst, src, 4);
        __pipeline_memcpy_async(dst + P.tcs, src + 1, 4);
      }
  }
}
__device__ __forceinline__ double fa_table_field(const double* tabs, int tcs, int f, int slot) {
  const uint32_t* planes = reinterpret_cast<const uint32_t*>(tabs);
  const uint32_t lo = planes[(size_t)(2 * f) * tcs + slot], hi = planes[(size_t)(2 * f + 1) * tcs + slot];
  return __hiloint2double((int)hi, (int)lo);
}
__device__ __forceinline__ void fa_get_table(const FaParams& P, const double* tabs, const double* __restrict__ tab, int slot, int32_t cam,
                                             double* T) {
  if (slot < P.tcam) {
#pragma unroll
    for (int f = 0; f < TAB; ++f) T[f] = fa_table_field(tabs, P.tcs, f, slot);
  } else {
    load_tab(tab, cam, T);
  }
}

// three / four tile scalars through one barrier: warp trees, then warp 0 folds the per-warp values (the same fixed
// tree as block_sum / block_max); result valid in thread 0
__device__ __forceinline__ void fa_block_reduce(double* v, const bool* is_max, int n, double* red /* [n][32] */) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  for (int k = 0; k < n; ++k) {
    v[k] = is_max[k] ? warp_max(v[k]) : warp_sum(v[k]);
    if (lane == 0) red[32 * k + warp] = v[k];
  }
  __syncthreads();
  if (warp == 0)
    for (int k = 0; k < n; ++k) {
      const double x = lane < nw ? red[32 * k + lane] : 0.0;
      v[k] = is_max[k] ? warp_max(x) : warp_sum(x);
    }
}

// item index of a tile dealt boustrophedon over the threads: round r, thread t -> r * T + (r odd ? T - 1 - t : t);
// the camera items are dealt from the other end, so they go first to the threads whose pair items were the shortest
__device__ __forceinline__ int fa_item_index(int r, bool reverse) {
  const int t = (int)threadIdx.x, n = (int)blockDim.x;
  return r * n + ((((r & 1) != 0) != reverse) ? n - 1 - t : t);
}

// MODE FA_FULL: linearise and eliminate.  MODE FA_NORMS: iteration 0 only, unscaled Jacobian; writes the Jacobi scaling
// of the points and the camera items (their F^T F diagonals are the camera column norms); no Schur products.
// MODE FA_GRAD: cost and gradient only (scaled Jacobian, camera items, no Cholesky, no Schur products) -- the
// evaluation after the last step of a solve, where Ceres evaluates the Jacobian too but never eliminates it.
// MODE FA_FIRST: iteration 0 in ONE pass.  The Jacobi scaling of a point is local to its tile: it is computed from the
// unscaled E^T E, written out, and applied to the point's records before anything is eliminated.  The cameras' scaling
// needs the global column norms, so the camera side stays unscaled here (scale fields of the tables = 1) and the reduced
// results (F^T F, F^T r, sum v, Schur products) are scaled afterwards, per block (k_fa_scale_cams / k_fa_scale_pairs).
//
// Latency plan (the kernel is bound by dependent round trips, not by bytes or flops): the tile descriptor is one
// load; the camera tables, the tile's points (x_e, scale) and the work-item entry lists arrive by cp.async while the
// threads fetch, into registers, the first observation, the first point range and the first work items they will
// handle -- so every phase after the first barrier starts from shared memory or registers.
template <int MODE>
__global__ void __launch_bounds__(FA_MAX_THREADS, 1) k_fa_pass1(FaParams P) {
  constexpr bool NORMS = MODE == FA_NORMS, FIRST = MODE == FA_FIRST, FULL = MODE == FA_FULL || FIRST, UNIT = NORMS || FIRST;
  extern __shared__ double smem[];
  double* rec = smem;                                   // [cap][FA_REC]: U (6) | Jf (12) | r (2) | w (2)
  double* Ls = rec + (size_t)P.cap * FA_REC;            // [pts_cap][FA_LS]: x_e (3) | scale (3), then L (6) | z (3)
  double* tabs = Ls + (size_t)P.pts_cap * FA_LS;        // [TAB][tcs]
  int32_t* pent_s = reinterpret_cast<int32_t*>(tabs + (size_t)P.tcs * TAB);  // [pent_cap] the tile's pair entries
  int32_t* cent_s = pent_s + P.pent_cap;                // [cap] the tile's camera-item entries
  uint16_t* oblp = reinterpret_cast<uint16_t*>(cent_s + P.cap);  // [cap] local point of an observation
  __shared__ double red[96];
  const int tile = blockIdx.x, tid = threadIdx.x, nthr = blockDim.x;
  const FaTile T = fa_load_tile(P.tiles + tile);
  const int64_t pt0 = T.pt0, ob0 = T.ob0, pe0 = T.pe0, ce0 = T.ce0;
  const int nobs = T.nobs, npts = T.npts;
  const int npe = FULL ? min(T.npe, P.pent_cap) : 0;
  const int nce = min(T.nce, P.cap);
  // group 1 (needed by A1): camera tables, points
  fa_stage_tables_async(P, T, P.tab_f, tabs, TAB, nullptr);
  for (int i = tid; i < 3 * npts; i += nthr) {
    const int lp = i / 3, k = i - 3 * lp;
    __pipeline_memcpy_async(Ls + lp * FA_LS + k, P.xe + 3 * pt0 + i, 8);
    if (!UNIT) __pipeline_memcpy_async(Ls + lp * FA_LS + 3 + k, P.se + 3 * pt0 + i, 8);
  }
  __pipeline_commit();
  // group 2 (needed by B): the work-item entry lists
  for (int i = tid; i < npe; i += nthr) __pipeline_memcpy_async(pent_s + i, P.pent + pe0 + i, 4);
  for (int i = tid; i < nce; i += nthr) __pipeline_memcpy_async(cent_s + i, P.cent + ce0 + i, 4);
  __pipeline_commit();
  // registers: first work items, first point range, first observation of this thread
  int pq0 = 0, pq1 = 0, cq0 = 0, cq1 = 0, pl0 = 0, pl1 = 0;
  if (FULL && tid < T.npitem) {
    pq0 = (int)(P.pitem_begin[T.pitem0 + tid] - pe0);
    pq1 = (int)(P.pitem_end[T.pitem0 + tid] - pe0);
  }
  if (nthr - 1 - tid < T.ncitem) {
    cq0 = (int)(P.citem_begin[T.citem0 + (nthr - 1 - tid)] - ce0);
    cq1 = (int)(P.citem_end[T.citem0 + (nthr - 1 - tid)] - ce0);
  }
  if (tid < npts) {
    pl0 = (int)(P.e_ptr[pt0 + tid] - ob0);
    pl1 = (int)(P.e_ptr[pt0 + tid + 1] - ob0);
  }
  uint32_t m_n = 0;
  double2 uv_n = make_double2(0.0, 0.0);
  if (tid < nobs) { m_n = P.ob_meta[ob0 + tid]; uv_n = P.uv[ob0 + tid]; }
  __pipeline_wait_prior(1);
  __syncthreads();
  // ---- A1: one thread per observation (the next round's inputs are in flight while this one computes) ----
  double sq = 0.0;
  for (int l = tid; l < nobs; l += nthr) {
    const int lp = (int)(m_n & 0xffffu), slot = (int)(m_n >> 16);
    const double2 ob = uv_n;
    if (l + nthr < nobs) { const int64_t o = ob0 + l + nthr; m_n = P.ob_meta[o]; uv_n = P.uv[o]; }
    double Tt[TAB];
    if (slot < P.tcam) {
#pragma unroll
      for (int f = 0; f < TAB; ++f) Tt[f] = fa_table_field(tabs, P.tcs, f, slot);
    } else {
      load_tab(P.tab_f, P.ob_f[ob0 + l], Tt);
    }
    const double* xs = Ls + lp * FA_LS;
    const double X[3] = {xs[0], xs[1], xs[2]};
    double s[3] = {1.0, 1.0, 1.0};
    if (!UNIT) { s[0] = xs[3]; s[1] = xs[4]; s[2] = xs[5]; }
    double r[2], je[6], jf[12];
    fa_linearize(Tt, X, s, ob, r, je, jf);
    sq += fa_apply_loss(P.loss, r, je, jf);
    double2* R2 = reinterpret_cast<double2*>(rec + (size_t)l * FA_REC);
#pragma unroll
    for (int k = 0; k < 3; ++k) R2[k] = make_double2(je[2 * k], je[2 * k + 1]);
#pragma unroll
    for (int k = 0; k < 6; ++k) R2[3 + k] = make_double2(jf[2 * k], jf[2 * k + 1]);
    R2[9] = make_double2(r[0], r[1]);
    R2[10] = make_double2(0.0, 0.0);
    oblp[l] = (uint16_t)lp;
  }
  __syncthreads();
  // ---- A2a: one thread per point ----
  double gmx = 0.0, g2 = 0.0;
  const double radius = *P.radius;
  for (int lp = tid; lp < npts; lp += nthr) {
    const int64_t e = pt0 + lp;
    int l0 = pl0, l1 = pl1;
    if (lp != tid) { l0 = (int)(P.e_ptr[e] - ob0); l1 = (int)(P.e_ptr[e + 1] - ob0); }
    double M[6] = {0, 0, 0, 0, 0, 0}, g[3] = {0, 0, 0};  // m00 m01 m02 m11 m12 m22
    for (int l = l0; l < l1; ++l) {
      const double* R = rec + (size_t)l * FA_REC;
#pragma unroll
      for (int rr = 0; rr < 2; ++rr) {
        const double j0 = R[3 * rr], j1 = R[3 * rr + 1], j2 = R[3 * rr + 2], rv = R[18 + rr];
        M[0] += j0 * j0; M[1] += j0 * j1; M[2] += j0 * j2; M[3] += j1 * j1; M[4] += j1 * j2; M[5] += j2 * j2;
        g[0] += j0 * rv; g[1] += j1 * rv; g[2] += j2 * rv;
      }
    }
    if (NORMS) {
      P.se_out[3 * e] = 1.0 / (1.0 + sqrt(M[0])); P.se_out[3 * e + 1] = 1.0 / (1.0 + sqrt(M[3])); P.se_out[3 * e + 2] = 1.0 / (1.0 + sqrt(M[5]));
      continue;
    }
    double* ls = Ls + lp * FA_LS;
    if (FIRST) {  // Jacobi scaling of this point from the unscaled column norms; E^T E, E^T r and the records in scaled columns
      const double s0 = 1.0 / (1.0 + sqrt(M[0])), s1 = 1.0 / (1.0 + sqrt(M[3])), s2 = 1.0 / (1.0 + sqrt(M[5]));
      P.se_out[3 * e] = s0; P.se_out[3 * e + 1] = s1; P.se_out[3 * e + 2] = s2;
      ls[3] = s0; ls[4] = s1; ls[5] = s2;
      M[0] *= s0 * s0; M[1] *= s0 * s1; M[2] *= s0 * s2; M[3] *= s1 * s1; M[4] *= s1 * s2; M[5] *= s2 * s2;
      g[0] *= s0; g[1] *= s1; g[2] *= s2;
      for (int l = l0; l < l1; ++l) {
        double* R = rec + (size_t)l * FA_REC;
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) { R[3 * rr] *= s0; R[3 * rr + 1] *= s1; R[3 * rr + 2] *= s2; }
      }
    }
    if (l1 > l0) {  // |x - Plus(x, -g)| of the unscaled gradient (TrustRegionMinimizer::EvaluateGradientAndJacobian)
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const double xv = ls[k];
        const double d = xv - (xv + (-(g[k] / ls[3 + k])));
        gmx = fmax(gmx, fabs(d)); g2 += d * d;
      }
    }
    if (!FULL) continue;
    {
      const double da = sqrt(fmin(fmax(M[0], P.min_diag), P.max_diag) / radius);
      const double db = sqrt(fmin(fmax(M[3], P.min_diag), P.max_diag) / radius);
      const double dc = sqrt(fmin(fmax(M[5], P.min_diag), P.max_diag) / radius);
      M[0] += da * da; M[3] += db * db; M[5] += dc * dc;
    }
    double Lp[6];
    if (!fa_chol3(M, Lp)) {
      atomicOr(P.status, 1);
      Lp[0] = Lp[1] = Lp[2] = 0.0; Lp[3] = Lp[4] = Lp[5] = 1.0;
    }
    fa_fwd3(Lp, g);  // z
#pragma unroll
    for (int k = 0; k < 6; ++k) ls[k] = Lp[k];
#pragma unroll
    for (int k = 0; k < 3; ++k) ls[6 + k] = g[k];
  }
  __pipeline_wait_prior(0);
  __syncthreads();
  // ---- A2b: one thread per observation: U = L^-1 J_e^T (rows), w = U^T z; L | z of the tile leave as full lines ----
  if (FULL) {
    for (int i = tid; i < 9 * npts; i += nthr) { const int lp = i / 9; P.Lz[9 * pt0 + i] = Ls[lp * FA_LS + (i - 9 * lp)]; }
    for (int l = tid; l < nobs; l += nthr) {
      double* R = rec + (size_t)l * FA_REC;
      const double* ls = Ls + (int)oblp[l] * FA_LS;
      double Lp[6], z[3];
#pragma unroll
      for (int k = 0; k < 6; ++k) Lp[k] = ls[k];
#pragma unroll
      for (int k = 0; k < 3; ++k) z[k] = ls[6 + k];
#pragma unroll
      for (int rr = 0; rr < 2; ++rr) {
        double u[3] = {R[3 * rr], R[3 * rr + 1], R[3 * rr + 2]};
        fa_fwd3(Lp, u);
        R[3 * rr] = u[0]; R[3 * rr + 1] = u[1]; R[3 * rr + 2] = u[2];
        R[20 + rr] = u[0] * z[0] + u[1] * z[1] + u[2] * z[2];
      }
    }
    __syncthreads();
  }
  // ---- B: one thread per work item ----
  if (FULL) {
    for (int r = 0; r * nthr < T.npitem; ++r) {
      const int idx = fa_item_index(r, false);
      if (idx >= T.npitem) continue;
      const int64_t it = T.pitem0 + idx;
      int q = pq0, q1 = pq1;
      if (r > 0) { q = (int)(P.pitem_begin[it] - pe0); q1 = (int)(P.pitem_end[it] - pe0); }
      double acc[36];
#pragma unroll
      for (int k = 0; k < 36; ++k) acc[k] = 0.0;
      for (; q < q1; ++q) {
        const int32_t cur = q < npe ? pent_s[q] : P.pent[pe0 + q];
        const double2* Ri = reinterpret_cast<const double2*>(rec + (size_t)(cur & 0xffff) * FA_REC);
        const double2* Rj = reinterpret_cast<const double2*>(rec + (size_t)((cur >> 16) & 0xffff) * FA_REC);
        double ui[6], uj[6], fj[12];
#pragma unroll
        for (int k = 0; k < 3; ++k) { const double2 a = Ri[k], b = Rj[k]; ui[2 * k] = a.x; ui[2 * k + 1] = a.y; uj[2 * k] = b.x; uj[2 * k + 1] = b.y; }
#pragma unroll
        for (int k = 0; k < 6; ++k) { const double2 b = Rj[3 + k]; fj[2 * k] = b.x; fj[2 * k + 1] = b.y; }
        const double g00 = ui[0] * uj[0] + ui[1] * uj[1] + ui[2] * uj[2], g01 = ui[0] * uj[3] + ui[1] * uj[4] + ui[2] * uj[5];
        const double g10 = ui[3] * uj[0] + ui[4] * uj[1] + ui[5] * uj[2], g11 = ui[3] * uj[3] + ui[4] * uj[4] + ui[5] * uj[5];
        double t0[6], t1[6];
#pragma unroll
        for (int b = 0; b < 6; ++b) { t0[b] = g00 * fj[b] + g01 * fj[6 + b]; t1[b] = g10 * fj[b] + g11 * fj[6 + b]; }
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          const double2 f0 = Ri[3 + k], f1 = Ri[6 + k];   // J_f,i rows 0 / 1, columns 2k, 2k+1
#pragma unroll
          for (int b = 0; b < 6; ++b) {
            acc[(2 * k) * 6 + b] += f0.x * t0[b] + f1.x * t1[b];
            acc[(2 * k + 1) * 6 + b] += f0.y * t0[b] + f1.y * t1[b];
          }
        }
      }
      double2* out = reinterpret_cast<double2*>(P.partP + (size_t)it * 36);
#pragma unroll
      for (int k = 0; k < 18; ++k) out[k] = make_double2(acc[2 * k], acc[2 * k + 1]);
    }
  }
  for (int r = 0; r * nthr < T.ncitem; ++r) {
    const int idx = fa_item_index(r, true);
    if (idx >= T.ncitem) continue;
    const int64_t it = T.citem0 + idx;
    int q = cq0, q1 = cq1;
    if (r > 0) { q = (int)(P.citem_begin[it] - ce0); q1 = (int)(P.citem_end[it] - ce0); }
    double acc[FA_NVC];
#pragma unroll
    for (int k = 0; k < FA_NVC; ++k) acc[k] = 0.0;
    for (; q < q1; ++q) {
      const double2* R2 = reinterpret_cast<const double2*>(rec + (size_t)cent_s[q] * FA_REC);
      double jf[12];
#pragma unroll
      for (int k = 0; k < 6; ++k) { const double2 v = R2[3 + k]; jf[2 * k] = v.x; jf[2 * k + 1] = v.y; }
      const double2 rv = R2[9], wv = R2[10];
      int c = 0;
#pragma unroll
      for (int a = 0; a < 6; ++a)
#pragma unroll
        for (int b = a; b < 6; ++b) acc[c++] += jf[a] * jf[b] + jf[6 + a] * jf[6 + b];
#pragma unroll
      for (int a = 0; a < 6; ++a) { acc[21 + a] += jf[a] * rv.x + jf[6 + a] * rv.y; acc[27 + a] += jf[a] * wv.x + jf[6 + a] * wv.y; }
    }
    double* out = P.partC + (size_t)it * FA_NVC;
#pragma unroll
    for (int k = 0; k < FA_NVC; ++k) out[k] = acc[k];
  }
  if (!NORMS) {  // cost and gradient-norm partials of the tile (fixed tree, one barrier)
    double v[3] = {sq, g2, gmx};
    const bool mx[3] = {false, false, true};
    fa_block_reduce(v, mx, 3, red);
    if (tid == 0) { P.cost_partial[tile] = v[0]; P.g2_partial[tile] = v[1]; P.gmax_partial[tile] = v[2]; }
  }
}

__device__ __constant__ int kFaCandFields[16] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 18, 19, 20, 21, 22, 23, 24};  // R | t | fx fy ppx ppy

// back-substitution, model cost change, candidate point and candidate cost of one tile
__global__ void __launch_bounds__(FA_MAX_THREADS, 1) k_fa_pass2(FaParams P) {
  extern __shared__ double smem[];
  double* rec = smem;                                   // [cap][FA_REC2]: J_e (6) | r (2) | J_f yf (2)
  double* Xs = rec + (size_t)P.cap * FA_REC2;           // [pts_cap][FA_PS2]
  double* tabs = Xs + (size_t)P.pts_cap * FA_PS2;       // [TAB][tcs] tables at x
  double* tabc = tabs + (size_t)P.tcs * TAB;            // [16][tcs] tables at the candidate (R, t, intrinsics)
  __shared__ double red[128];
  const int tile = blockIdx.x, tid = threadIdx.x, nthr = blockDim.x;
  const FaTile T = fa_load_tile(P.tiles + tile);
  const int64_t pt0 = T.pt0, ob0 = T.ob0;
  const int nobs = T.nobs, npts = T.npts;
  fa_stage_tables_async(P, T, P.tab_f, tabs, TAB, nullptr);
  for (int i = tid; i < 3 * npts; i += nthr) {
    const int lp = i / 3, k = i - 3 * lp;
    __pipeline_memcpy_async(Xs + lp * FA_PS2 + k, P.xe + 3 * pt0 + i, 8);
    __pipeline_memcpy_async(Xs + lp * FA_PS2 + 3 + k, P.se + 3 * pt0 + i, 8);
  }
  __pipeline_commit();
  fa_stage_tables_async(P, T, P.tabc_f, tabc, 16, kFaCandFields);   // needed by the last loop only
  __pipeline_commit();
  int pl0 = 0, pl1 = 0;
  if (tid < npts) {
    pl0 = (int)(P.e_ptr[pt0 + tid] - ob0);
    pl1 = (int)(P.e_ptr[pt0 + tid + 1] - ob0);
  }
  uint32_t m_n = 0;
  int32_t c_n = 0;
  double2 uv_n = make_double2(0.0, 0.0);
  if (tid < nobs) { m_n = P.ob_meta[ob0 + tid]; c_n = P.ob_f[ob0 + tid]; uv_n = P.uv[ob0 + tid]; }
  __pipeline_wait_prior(1);
  __syncthreads();
  for (int l = tid; l < nobs; l += nthr) {
    const int lp = (int)(m_n & 0xffffu), slot = (int)(m_n >> 16);
    const int32_t c = c_n;
    const double2 ob = uv_n;
    if (l + nthr < nobs) { const int64_t o = ob0 + l + nthr; m_n = P.ob_meta[o]; c_n = P.ob_f[o]; uv_n = P.uv[o]; }
    double y[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) y[k] = __ldg(P.yf + 6 * (int64_t)c + k);
    double Tt[TAB];
    fa_get_table(P, tabs, P.tab_f, slot, c, Tt);
    const double* xs = Xs + lp * FA_PS2;
    const double X[3] = {xs[0], xs[1], xs[2]};
    const double s[3] = {xs[3], xs[4], xs[5]};
    double r[2], je[6], jf[12];
    fa_linearize(Tt, X, s, ob, r, je, jf);
    fa_apply_loss(P.loss, r, je, jf);
    double q0 = 0.0, q1 = 0.0;
#pragma unroll
    for (int k = 0; k < 6; ++k) { q0 += jf[k] * y[k]; q1 += jf[6 + k] * y[k]; }
    double2* R2 = reinterpret_cast<double2*>(rec + (size_t)l * FA_REC2);
#pragma unroll
    for (int k = 0; k < 3; ++k) R2[k] = make_double2(je[2 * k], je[2 * k + 1]);
    R2[3] = make_double2(r[0], r[1]);
    R2[4] = make_double2(q0, q1);
  }
  // the last loop's first observation: in flight across the point phase
  uint32_t m2 = 0;
  double2 uv2 = make_double2(0.0, 0.0);
  if (tid < nobs) { m2 = P.ob_meta[ob0 + tid]; uv2 = P.uv[ob0 + tid]; }
  __syncthreads();
  double mcc = 0.0, x2 = 0.0, d2 = 0.0;
  for (int lp = tid; lp < npts; lp += nthr) {
    const int64_t e = pt0 + lp;
    int l0 = pl0, l1 = pl1;
    if (lp != tid) { l0 = (int)(P.e_ptr[e] - ob0); l1 = (int)(P.e_ptr[e + 1] - ob0); }
    const double* in = P.Lz + 9 * e;
    double Lp[6], t[3];
#pragma unroll
    for (int k = 0; k < 6; ++k) Lp[k] = in[k];
#pragma unroll
    for (int k = 0; k < 3; ++k) t[k] = in[6 + k];
    for (int l = l0; l < l1; ++l) {
      const double* R = rec + (size_t)l * FA_REC2;
#pragma unroll
      for (int rr = 0; rr < 2; ++rr) {
        double u[3] = {R[3 * rr], R[3 * rr + 1], R[3 * rr + 2]};
        fa_fwd3(Lp, u);
        const double q = R[8 + rr];
        t[0] -= u[0] * q; t[1] -= u[1] * q; t[2] -= u[2] * q;
      }
    }
    fa_bwd3(Lp, t);  // y_e
    // Ceres: model_cost_change = -(J step)^T (r + J step / 2) with step = -y; the caller negates the sum
    for (int l = l0; l < l1; ++l) {
      const double* R = rec + (size_t)l * FA_REC2;
#pragma unroll
      for (int rr = 0; rr < 2; ++rr) {
        const double m = -(R[3 * rr] * t[0] + R[3 * rr + 1] * t[1] + R[3 * rr + 2] * t[2]) - R[8 + rr];
        mcc += m * (R[6 + rr] + m / 2.0);
      }
    }
    double* xs = Xs + lp * FA_PS2;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const double xv = xs[k];
      const double c = xv + (-(t[k]) * xs[3 + k]);
      P.xe_c[3 * e + k] = c;
      xs[k] = c;
      if (l1 > l0) { x2 += xv * xv; const double d = xv - c; d2 += d * d; }
    }
  }
  __pipeline_wait_prior(0);
  __syncthreads();
  double sq = 0.0;
  for (int l = tid; l < nobs; l += nthr) {
    const int lp = (int)(m2 & 0xffffu), slot = (int)(m2 >> 16);
    const double2 ob = uv2;
    if (l + nthr < nobs) { const int64_t o = ob0 + l + nthr; m2 = P.ob_meta[o]; uv2 = P.uv[o]; }
    double C[16];
    if (slot < P.tcam) {
#pragma unroll
      for (int f = 0; f < 16; ++f) C[f] = fa_table_field(tabc, P.tcs, f, slot);
    } else {
      const double* Tc = P.tabc_f + TAB * (int64_t)P.ob_f[ob0 + l];
#pragma unroll
      for (int f = 0; f < 16; ++f) C[f] = __ldg(Tc + kFaCandFields[f]);
    }
    const double* xs = Xs + lp * FA_PS2;
    const double X[3] = {xs[0], xs[1], xs[2]};
    double q[3];
    mat3_vec(C, X, q);
    const double p0 = q[0] + C[9], p1 = q[1] + C[10], p2 = q[2] + C[11];
    const double r0 = C[12] * p0 / p2 + C[14] - ob.x;
    const double r1 = C[13] * p1 / p2 + C[15] - ob.y;
    double sc = r0 * r0 + r1 * r1;
    if (P.loss.type != 0) { double w; loss_apply(P.loss, sc, &sc, &w); }
    sq += sc;
  }
  double v[4] = {mcc, x2, d2, sq};
  const bool mx[4] = {false, false, false, false};
  fa_block_reduce(v, mx, 4, red);
  if (tid == 0) { P.mcc_partial[tile] = v[0]; P.x2_partial[tile] = v[1]; P.d2_partial[tile] = v[2]; P.cand_partial[tile] = v[3]; }
}

// Standalone residual + Jacobian of Model A (what ba_cuda_eval and the generic pipeline materialise): the tile
// prologue of pass 1 (descriptor, tables and points by cp.async, the first observation in registers), then every warp
// works on its own: 32 consecutive observations per round, r leaves directly (16 B per thread, contiguous), the J_e and
// J_f records go through a per-warp staging buffer (__syncwarp only) and leave as full 128-byte lines.  The staging
// buffers are packed exactly like the global arrays, so the copy-out reads consecutive 16-byte units; the writes are
// conflict free too (J_e: 3 units per lane, odd stride; J_f: 6 units per lane, the lanes with bit 2 set write their
// units one step ahead of the others).  ~31 KB of shared memory, 128 registers: four CTAs of 128 threads per SM.
// Replaces k_jac_a whenever the tile structure exists: k_jac_a reads a 256-byte table per observation through L1
// (32 different lines per warp load) and is bound by that, not by HBM.
__global__ void __launch_bounds__(FA_JAC_THREADS, 4) k_fa_jac(FaParams P) {
  extern __shared__ double smem[];
  const int tile = blockIdx.x, tid = threadIdx.x, nthr = blockDim.x, lane = tid & 31, warp = tid >> 5;
  double* wje = smem + (size_t)warp * (32 * FA_RECJ);   // [32][6] of this warp
  double* wjf = wje + 32 * 6;                           // [32][12]
  double2* uv_s = reinterpret_cast<double2*>(smem + (size_t)(nthr >> 5) * (32 * FA_RECJ));   // [cap] image points of the tile
  double* Xs = reinterpret_cast<double*>(uv_s + P.cap);  // [pts_cap][FA_PS2]
  double* tabs = Xs + (size_t)P.pts_cap * FA_PS2;       // table planes
  uint32_t* meta_s = reinterpret_cast<uint32_t*>(tabs + (size_t)P.tcs * TAB);   // [cap] local point | camera slot << 16
  __shared__ double red[32];
  const FaTile T = fa_load_tile(P.tiles + tile);
  const int64_t pt0 = T.pt0, ob0 = T.ob0;
  const int nobs = T.nobs, npts = T.npts;
  // everything the tile reads arrives by cp.async: the loop below touches global memory only to store
  fa_stage_tables_async(P, T, P.tab_f, tabs, TAB, nullptr);
  for (int i = tid; i < 3 * npts; i += nthr) {
    const int lp = i / 3, k = i - 3 * lp;
    __pipeline_memcpy_async(Xs + lp * FA_PS2 + k, P.xe + 3 * pt0 + i, 8);
    __pipeline_memcpy_async(Xs + lp * FA_PS2 + 3 + k, P.se + 3 * pt0 + i, 8);
  }
  for (int i = tid; i < nobs; i += nthr) {
    __pipeline_memcpy_async(uv_s + i, P.uv + ob0 + i, 16);
    __pipeline_memcpy_async(meta_s + i, P.ob_meta + ob0 + i, 4);
  }
  __pipeline_commit();
  __pipeline_wait_prior(0);
  __syncthreads();
  double sq = 0.0;
  double2* RES2 = reinterpret_cast<double2*>(P.RES);
  const bool ahead = (lane & 4) != 0;
  for (int base = warp * 32; base < nobs; base += nthr) {   // warp-uniform: 32 consecutive observations per round
    const int l = base + lane;
    const bool on = l < nobs;
    if (on) {
      const uint32_t m = meta_s[l];
      const int lp = (int)(m & 0xffffu), slot = (int)(m >> 16);
      const double2 ob = uv_s[l];
      double Tt[TAB];
      if (slot < P.tcam) {
#pragma unroll
        for (int f = 0; f < TAB; ++f) Tt[f] = fa_table_field(tabs, P.tcs, f, slot);
      } else {
        load_tab(P.tab_f, P.ob_f[ob0 + l], Tt);
      }
      const double* xs = Xs + lp * FA_PS2;
      const double X[3] = {xs[0], xs[1], xs[2]};
      const double s[3] = {xs[3], xs[4], xs[5]};
      double r[2], je[6], jf[12];
      fa_linearize(Tt, X, s, ob, r, je, jf);
      sq += fa_apply_loss(P.loss, r, je, jf);
      RES2[ob0 + l] = make_double2(r[0], r[1]);
      double2* E2 = reinterpret_cast<double2*>(wje) + 3 * lane;
#pragma unroll
      for (int k = 0; k < 3; ++k) E2[k] = make_double2(je[2 * k], je[2 * k + 1]);
      double2* F2 = reinterpret_cast<double2*>(wjf) + 6 * lane;
#pragma unroll
      for (int st = 0; st < 6; ++st) {
        const int k0 = st, k1 = (st + 1) % 6;
        F2[ahead ? k1 : k0] = ahead ? make_double2(jf[2 * k1], jf[2 * k1 + 1]) : make_double2(jf[2 * k0], jf[2 * k0 + 1]);
      }
    }
    __syncwarp();
    const int nv = min(32, nobs - base);
    const double2* se2 = reinterpret_cast<const double2*>(wje);
    const double2* sf2 = reinterpret_cast<const double2*>(wjf);
    double2* je_out = reinterpret_cast<double2*>(P.JE + 6 * (ob0 + base));
    double2* jf_out = reinterpret_cast<double2*>(P.JF + 12 * (ob0 + base));
#pragma unroll
    for (int m = 0; m < 3; ++m) { const int g = lane + 32 * m; if (g < 3 * nv) je_out[g] = se2[g]; }
#pragma unroll
    for (int m = 0; m < 6; ++m) { const int g = lane + 32 * m; if (g < 6 * nv) jf_out[g] = sf2[g]; }
    __syncwarp();
  }
  sq = block_sum(sq, red);
  if (tid == 0) P.cost_partial[tile] = sq;
}

// FA_FIRST / SA_FIRST: the reduced camera-side results of the unscaled pass, brought to Jacobi-scaled camera columns
// (NVC = FA_NVC on tiles; SA_NVC on strips, whose tail holds diag F^T F)
template <int NVC>
__global__ void k_fa_scale_cams(int64_t nf, const double* __restrict__ sf, double* __restrict__ camacc) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= nf * NVC) return;
  const int64_t c = t / NVC;
  const int v = (int)(t % NVC);
  double f;
  if (v < 21) {  // packed upper (a <= b) of F^T F
    int a = 0, rem = v;
    while (rem >= 6 - a) { rem -= 6 - a; ++a; }
    f = sf[6 * c + a] * sf[6 * c + a + rem];
  } else if (NVC == 33 || v < 33) {
    f = sf[6 * c + (v - 21) % 6];   // F^T r, sum of v
  } else {
    f = sf[6 * c + (v - 33)] * sf[6 * c + (v - 33)];   // diag F^T F (strips)
  }
  camacc[t] *= f;
}
__global__ void k_fa_scale_pairs(int ndest, const int32_t* __restrict__ dest_fa, const int32_t* __restrict__ dest_fb,
                                 const double* __restrict__ sf, double* __restrict__ Pacc) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= (int64_t)ndest * 36) return;
  const int d = (int)(t / 36), v = (int)(t % 36);
  Pacc[t] *= sf[6 * (int64_t)dest_fa[d] + v / 6] * sf[6 * (int64_t)dest_fb[d] + v % 6];
}

// first level: one warp per chunk of <= ch partial blocks of one target, lane = value, sequential over the blocks
template <int NV>
__global__ void __launch_bounds__(128)
k_reduce_items(int nchunks, int ch, const int32_t* __restrict__ chunk_seg, const int64_t* __restrict__ chunk_begin,
               const int64_t* __restrict__ tgt_ptr, const int32_t* __restrict__ items, const double* __restrict__ part, double* __restrict__ out) {
  const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (c >= nchunks) return;
  const int64_t begin = chunk_begin[c];
  const int64_t end = min(begin + ch, tgt_ptr[chunk_seg[c] + 1]);
  // lanes fetch 32 item ids at a time, then eight independent block loads are in flight per lane; the sum itself
  // stays strictly sequential in list order
  double a0 = 0.0, a1 = 0.0;  // values lane, lane + 32
  for (int64_t base = begin; base < end; base += 32) {
    const int n = (int)min((int64_t)32, end - base);
    const int32_t mine = lane < n ? items[base + lane] : 0;
    for (int k = 0; k < n; k += 8) {
      double x0[8], x1[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int32_t id = __shfl_sync(0xffffffffu, mine, (k + u) & 31);
        const bool on = k + u < n;
        x0[u] = on ? part[(int64_t)id * NV + lane] : 0.0;
        x1[u] = (on && lane + 32 < NV) ? part[(int64_t)id * NV + lane + 32] : 0.0;
      }
#pragma unroll
      for (int u = 0; u < 8; ++u)
        if (k + u < n) { a0 += x0[u]; a1 += x1[u]; }
    }
  }
  out[(int64_t)c * NV + lane] = a0;
  if (lane + 32 < NV) out[(int64_t)c * NV + lane + 32] = a1;
}
// second level: one warp per target over its chunk partials
template <int NV>
__global__ void __launch_bounds__(128)
k_reduce_final(int ntargets, const int32_t* __restrict__ seg_first, const double* __restrict__ part1, double* __restrict__ out) {
  const int t = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (t >= ntargets) return;
  const int c0 = seg_first[t], c1 = seg_first[t + 1];
  for (int v = lane; v < NV; v += 32) {
    double a = 0.0;
    for (int c = c0; c < c1; ++c) a += part1[(int64_t)c * NV + v];
    out[(int64_t)t * NV + v] = a;
  }
}

// folds up to 4 partial arrays in one launch: blockIdx.x = which; op 0 = sum, 1 = max
struct FoldJob { const double* partial[4]; int slot[4]; int is_max[4]; int n[4] = {0, 0, 0, 0}; };   // n[k] > 0 overrides the common length
__global__ void k_fold_multi(FoldJob J, int n, double* out) {
  __shared__ double sm[32];
  const double* partial = J.partial[blockIdx.x];
  if (J.n[blockIdx.x] > 0) n = J.n[blockIdx.x];
  double v = 0.0;
  if (J.is_max[blockIdx.x]) {
    for (int i = threadIdx.x; i < n; i += blockDim.x) v = fmax(v, partial[i]);
    v = block_max(v, sm);
  } else {
    for (int i = threadIdx.x; i < n; i += blockDim.x) v += partial[i];
    v = block_sum(v, sm);
  }
  if (threadIdx.x == 0) out[J.slot[blockIdx.x]] = v;
}

}  // namespace ba
