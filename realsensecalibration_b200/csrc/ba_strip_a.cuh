// ba_strip_a.cuh -- Model A pass 1, second generation: the Schur complement accumulators stay in registers
// across a STRIP of consecutive point tiles.
//
// What the first fused pass 1 (ba_fused_a.cuh, k_fa_pass1) paid for, measured with ncu on the 30 M-observation
// problem: one 288-byte partial block per (tile, camera pair) -- 5.4 GB written per launch and read back by
// k_reduce_items -- and shared-memory bank conflicts on the pair gathers (41 % of all wavefronts).  Here:
//
//   * one CTA of 512 threads walks a strip of L consecutive tiles.  A thread OWNS one destination block of the
//     reduced camera system (a camera pair, 36 accumulators) or one camera (the diagonal block and the camera sums,
//     39 accumulators) for the whole strip and writes it once, at the end of the strip: the partial blocks shrink
//     from one per (tile, pair) to one per (strip, pair).  Which thread owns what is planned per strip at build time
//     from the pair counts (heavy pairs / cameras are split over several threads, the lightest pairs of a strip
//     that do not fit go to one "flush" warp that still writes per tile).
//   * the observation records of a tile sit in shared memory at CLASS-ALIGNED positions: position mod 8 = camera
//     slot mod 8.  The eight lanes of a quarter warp own eight pairs (a, a + d) with consecutive a, so the records
//     they gather in one step lie in eight different 16-byte bank groups whatever the entries are: the gathers are
//     conflict free by construction instead of by a greedy entry order.
//   * the diagonal blocks are accumulated as F^T (I - U^T U) F together with the camera sums by the camera threads
//     (one pass over a camera's records instead of two work-item kinds), and the structural zeros of the 2 x 6
//     camera Jacobian are skipped in the pair products (92 instead of 108 FMAs).
//   * every per-tile input (image points, per-position words, point ranges, points, entry lists, segment table) is a
//     contiguous, 16-byte aligned slice built once per problem and arrives by cp.async.bulk (TMA, SASS UBLKCP) on
//     two mbarriers, prefetched one tile ahead while the current tile computes.
//
// Everything is static and every sum runs in a fixed order: bitwise reproducible, no floating-point atomics.
// Replaces, inside Ceres, SchurEliminator::Eliminate behind Test1_BundleAdjustment/main.cpp:82-86.
#pragma once
#include "ba_fused_a.cuh"

namespace ba {

constexpr int SA_NT = 512;          // threads per CTA = owner slots per strip
constexpr int SA_NCS_MAX = 64;      // cameras per strip (tables staged, 6-bit slots)
constexpr int SA_NVC = 39;          // per camera: 21 packed upper of F^T(I - U^T U)F | 6 F^T r | 6 sum v | 6 diag F^T F
constexpr int SA_REC = 22;          // doubles per record: U (6) | J_f (12) | r (2) | w (2)
constexpr int SA_NF_CAP = 1024;     // flush destinations per strip
constexpr int SA_POS_MAX = 4096;    // record positions per tile (12-bit entries)
constexpr int SA_CM_MAX = 8;        // owner threads per camera
constexpr int SA_TYPE_IDLE = 0, SA_TYPE_PAIR = 1, SA_TYPE_FLUSH = 2, SA_TYPE_CAM = 3;
constexpr int SA_FULL = 0, SA_GRAD = 2, SA_FIRST = 3;

__host__ __device__ inline int sa_xs_len(int pts_cap) { return (3 * pts_cap + 4 + 1) & ~1; }   // doubles, even: keeps 16-byte alignment

struct __align__(16) SaTile {
  int64_t pt0, ob0, pos0, ent0, pidx0, fout0;   // first point / sorted observation / position slot / entry / index slot / flush output
  int32_t npts, nobs, npos, nent;
};
static_assert(sizeof(SaTile) == 64, "SaTile is loaded as four 16-byte words");
struct __align__(16) SaStrip {
  int64_t cam0, pout0, cout0;       // first camera-list entry, first pair output block, first camera output block
  int32_t tile0, ntiles, ncs, nflush;
  int32_t flush_t0;                 // first thread of the flush warp (-1: none)
  int32_t npp, ncact, cbase;        // persistent pairs (layer stride), active cameras (layer stride), first camera thread
};
static_assert(sizeof(SaStrip) == 64, "SaStrip");

struct StripA {
  bool ready = false;
  int n_tiles = 0, n_strips = 0, tobs = 0, L = 0, kmax = 0;
  int cap_pos = 0, pts_cap = 0, ncs_cap = 0, tcs = 0, ent_cap = 0, pidx_cap = 0, segw = 0, nobs_cap = 0;
  int64_t n_pout = 0, n_fout = 0, n_cout = 0;
  DVec<int64_t> tile_pt_ptr;
  DVec<SaTile> tiles;
  DVec<SaStrip> strips;
  DVec<int32_t> strip_cams;
  DVec<int64_t> strip_cam_ptr;
  DVec<uint32_t> slot_out;      // [n_strips][SA_NT]: type << 30 | output rank inside the strip
  DVec<uint32_t> pm;            // per position: local point | camera slot << 12 | 1 << 31
  DVec<double2> puv;            // per position: image point
  DVec<uint16_t> pidx;          // per tile: positions of the observations in point order, then the point ranges
  DVec<int32_t> ent;            // per tile: entries by owner slot
  DVec<uint16_t> seg;           // [n_tiles][segw]: first entry of every owner slot
  DVec<uint32_t> ob_meta;       // per sorted observation: local point | camera slot << 16 (pass 2, k_fa_jac)
  ReduceList red_pairs, red_cams; // the partial blocks per strip and camera pair / camera
  size_t smem() const {
    size_t b = ((size_t)cap_pos * SA_REC + (size_t)tcs * TAB + 2 * (size_t)sa_xs_len(pts_cap)) * 8;
    b += (size_t)cap_pos * 16 + (size_t)cap_pos * 4 + (size_t)pidx_cap * 2 + (size_t)ent_cap * 4 + (size_t)segw * 2 + 64;
    return b;
  }
};

// ---------------------------------------------------------------------------------------
// build
// ---------------------------------------------------------------------------------------
__global__ void k_sa_strip_keys(int64_t nb, const int32_t* __restrict__ ob_e, const int32_t* __restrict__ ob_f,
                                const int32_t* __restrict__ tile_of_pt, int L, int64_t nf, uint64_t* __restrict__ keys) {
  const int64_t o = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (o < nb) keys[o] = (uint64_t)(tile_of_pt[ob_e[o]] / L) * (uint64_t)nf + (uint64_t)ob_f[o];
}
__global__ void k_sa_split_keys(int ng, const uint64_t* __restrict__ ukeys, int64_t nf, int32_t* __restrict__ gstrip, int32_t* __restrict__ gcam) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= ng) return;
  gstrip[g] = (int32_t)(ukeys[g] / (uint64_t)nf);
  gcam[g] = (int32_t)(ukeys[g] % (uint64_t)nf);
}
// camera slot of every observation inside its strip; the per-observation word of pass 2 / k_fa_jac
__global__ void k_sa_obs_slot(int64_t nb, const int32_t* __restrict__ ob_e, const int32_t* __restrict__ ob_f,
                              const int32_t* __restrict__ tile_of_pt, const int64_t* __restrict__ tile_pt_ptr, int L,
                              const int64_t* __restrict__ strip_cam_ptr, const int32_t* __restrict__ strip_cams,
                              uint8_t* __restrict__ ob_slot, uint32_t* __restrict__ ob_meta) {
  const int64_t o = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (o >= nb) return;
  const int32_t e = ob_e[o], tile = tile_of_pt[e], strip = tile / L, cam = ob_f[o];
  int64_t lo = strip_cam_ptr[strip], hi = strip_cam_ptr[strip + 1];
  const int64_t c0 = lo;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (strip_cams[mid] < cam) lo = mid + 1; else hi = mid;
  }
  const uint32_t slot = (uint32_t)min((int64_t)255, lo - c0);
  ob_slot[o] = (uint8_t)slot;
  ob_meta[o] = (uint32_t)(e - tile_pt_ptr[tile]) | (slot << 16);
}

__device__ __forceinline__ int sa_class(int ncs, int slot, int l) { return ncs >= 8 ? (slot & 7) : (l & 7); }
// Positions per class of a tile: the fullest class would set the size of the record area of EVERY tile (shared memory
// is sized by the maximum), so a class only gets nobs / 8 + 6 % aligned positions; the few observations beyond take
// the positions other classes leave free (their gathers may then conflict, nothing else changes).
__device__ __forceinline__ int sa_class_rows(int nobs, int max_class) { return min(max_class, (nobs * 17 / 16 + 7) / 8); }

// per tile: record positions needed (8 x the fullest class), entries (pairs + observations), index slots; maxima;
// duplicate (point, camera) observations are flagged (the strip path then is not used)
// stat: 0 max npos, 1 max npts, 2 max nent, 3 max nobs, 4 duplicate flag, 5 max index slots
__global__ void __launch_bounds__(256)
k_sa_tile_sizes(int n_tiles, int L, const int64_t* __restrict__ tile_pt_ptr, const int64_t* __restrict__ e_ptr,
                const uint8_t* __restrict__ ob_slot, const int64_t* __restrict__ strip_cam_ptr, int64_t* __restrict__ tile_npos,
                int64_t* __restrict__ tile_nent, int64_t* __restrict__ tile_npidx, int* __restrict__ stat) {
  __shared__ int cls[8];
  __shared__ int npair, dup;
  const int t = blockIdx.x;
  if (threadIdx.x < 8) cls[threadIdx.x] = 0;
  if (threadIdx.x == 0) { npair = 0; dup = 0; }
  __syncthreads();
  const int64_t pt0 = tile_pt_ptr[t], pt1 = tile_pt_ptr[t + 1];
  const int64_t ob0 = e_ptr[pt0];
  const int nobs = (int)(e_ptr[pt1] - ob0), npts = (int)(pt1 - pt0);
  const int strip = t / L;
  const int ncs = (int)(strip_cam_ptr[strip + 1] - strip_cam_ptr[strip]);
  for (int l = threadIdx.x; l < nobs; l += blockDim.x) atomicAdd(&cls[sa_class(ncs, ob_slot[ob0 + l], l)], 1);
  for (int lp = threadIdx.x; lp < npts; lp += blockDim.x) {
    const int64_t b = e_ptr[pt0 + lp], n = e_ptr[pt0 + lp + 1];
    const int k = (int)(n - b);
    atomicAdd(&npair, k * (k - 1) / 2);
    for (int64_t i = b; i < n; ++i)
      for (int64_t j = i + 1; j < n; ++j)
        if (ob_slot[i] == ob_slot[j]) dup = 1;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int mx = 0;
    for (int c = 0; c < 8; ++c) mx = max(mx, cls[c]);
    const int npos = 8 * sa_class_rows(nobs, mx);
    const int nent = (npair + nobs + 3) & ~3;
    const int npidx = ((nobs + 7) & ~7) + ((npts + 1 + 7) & ~7);
    tile_npos[t] = npos; tile_nent[t] = nent; tile_npidx[t] = npidx;
    atomicMax(stat + 0, npos); atomicMax(stat + 1, npts); atomicMax(stat + 2, nent); atomicMax(stat + 3, nobs);
    if (dup) atomicMax(stat + 4, 1);
    atomicMax(stat + 5, npidx);
  }
}

// per tile: descriptor, record positions (warp c assigns class c in observation order), the position-ordered words
// and image points, the point ranges
__global__ void __launch_bounds__(256)
k_sa_tile_fill(int n_tiles, int L, const int64_t* __restrict__ tile_pt_ptr, const int64_t* __restrict__ e_ptr,
               const int32_t* __restrict__ ob_e, const uint8_t* __restrict__ ob_slot, const double2* __restrict__ uv,
               const int64_t* __restrict__ strip_cam_ptr, const int64_t* __restrict__ pos0, const int64_t* __restrict__ ent0,
               const int64_t* __restrict__ pidx0, const int64_t* __restrict__ tile_npos, const int64_t* __restrict__ tile_nent,
               SaTile* __restrict__ tiles, uint32_t* __restrict__ pm, double2* __restrict__ puv, uint16_t* __restrict__ pidx) {
  const int t = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t pt0 = tile_pt_ptr[t], pt1 = tile_pt_ptr[t + 1];
  const int64_t ob0 = e_ptr[pt0];
  const int nobs = (int)(e_ptr[pt1] - ob0), npts = (int)(pt1 - pt0);
  const int strip = t / L;
  const int ncs = (int)(strip_cam_ptr[strip + 1] - strip_cam_ptr[strip]);
  const int64_t P0 = pos0[t], I0 = pidx0[t];
  if (threadIdx.x == 0) {
    SaTile T;
    T.pt0 = pt0; T.ob0 = ob0; T.pos0 = P0; T.ent0 = ent0[t]; T.pidx0 = I0; T.fout0 = 0;
    T.npts = npts; T.nobs = nobs; T.npos = (int32_t)tile_npos[t]; T.nent = (int32_t)tile_nent[t];
    tiles[t] = T;
  }
  __shared__ int cnt[8], free0[9], ovf0[9];
  const int R = (int)(tile_npos[t] / 8);
  if (warp < 8) {   // class counts
    int n = 0;
    for (int l0 = 0; l0 < nobs; l0 += 32) {
      const int l = l0 + lane;
      const bool mine = l < nobs && sa_class(ncs, (int)ob_slot[ob0 + l], l) == warp;
      n += __popc(__ballot_sync(0xffffffffu, mine));
    }
    if (lane == 0) cnt[warp] = n;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int f = 0, o = 0;
    for (int c = 0; c < 8; ++c) { free0[c] = f; ovf0[c] = o; f += R - min(cnt[c], R); o += max(cnt[c] - R, 0); }
    free0[8] = f; ovf0[8] = o;
  }
  __syncthreads();
  if (warp < 8) {
    int base = 0;
    for (int l0 = 0; l0 < nobs; l0 += 32) {
      const int l = l0 + lane;
      const int slot = l < nobs ? (int)ob_slot[ob0 + l] : 0;
      const bool mine = l < nobs && sa_class(ncs, slot, l) == warp;
      const unsigned m = __ballot_sync(0xffffffffu, mine);
      if (mine) {
        const int r = base + __popc(m & ((1u << lane) - 1u));
        int pos = warp + 8 * r;
        if (r >= R) {   // the k-th position left free by the other classes
          const int k = ovf0[warp] + (r - R);
          int c = 0;
          while (c < 7 && free0[c + 1] <= k) ++c;
          pos = c + 8 * (min(cnt[c], R) + (k - free0[c]));
        }
        pidx[I0 + l] = (uint16_t)pos;
        pm[P0 + pos] = (uint32_t)(ob_e[ob0 + l] - pt0) | ((uint32_t)slot << 12) | 0x80000000u;
        puv[P0 + pos] = uv[ob0 + l];
      }
      base += __popc(m);
    }
  }
  const int64_t B0 = I0 + ((nobs + 7) & ~7);
  for (int lp = threadIdx.x; lp <= npts; lp += blockDim.x) pidx[B0 + lp] = (uint16_t)(e_ptr[pt0 + lp] - ob0);
}

struct SaPlanParams {
  int n_strips, L, n_tiles, ncs_cap, nf_cap;
  int cam_budget;               // camera threads per strip (whole warps): the observations of a camera are dealt over its threads
  int by_count;                 // owner slots in order of descending pair count instead of (diagonal, first camera)
  int balance;                  // deal the warps over the four SM sub-partitions by load
  int arrange;                  // class-aware order inside every group of 32 owner slots
  const int64_t* tile_pt_ptr; const int64_t* e_ptr; const uint8_t* ob_slot; const int64_t* strip_cam_ptr;
  uint32_t* dslot;              // [n_strips][ncs_cap^2]: rank | copies << 12, or 1 << 31 | flush index; ~0 = no such pair
  uint32_t* cslot;              // [n_strips][ncs_cap]: owner threads of the camera; 0 = camera without observations
  uint16_t* cthr;               // [n_strips][ncs_cap][SA_CM_MAX]: the owner threads (layer major: consecutive cameras in consecutive lanes)
  uint32_t* slot_out;           // [n_strips][SA_NT]
  uint16_t* slot_dest;          // [n_strips][SA_NT]: sa << 8 | sb (pair), s (camera)
  uint16_t* thr_of;             // [n_strips][SA_NT]: logical owner slot -> thread (warps dealt over the four SM sub-partitions by load)
  uint16_t* fl_dest;            // [n_strips][nf_cap]
  int32_t* counts;              // [n_strips][8]: npout, ncout, nflush, flush_t0, npp, -, cbase, ok
};

// One CTA per strip: pair counts per camera-slot pair, then thread 0 plans the owner slots.
__global__ void __launch_bounds__(256) k_sa_strip_plan(SaPlanParams P) {
  __shared__ int cnt[SA_NCS_MAX * SA_NCS_MAX];
  __shared__ int camobs[SA_NCS_MAX];
  __shared__ uint16_t pdest[SA_NT];
  __shared__ uint8_t pcopies[SA_NT];
  const int strip = blockIdx.x, tid = threadIdx.x;
  const int ncs = (int)(P.strip_cam_ptr[strip + 1] - P.strip_cam_ptr[strip]);
  for (int i = tid; i < SA_NCS_MAX * SA_NCS_MAX; i += blockDim.x) cnt[i] = 0;
  if (tid < SA_NCS_MAX) camobs[tid] = 0;
  __syncthreads();
  const int t0 = strip * P.L, t1 = min(P.n_tiles, t0 + P.L);
  const int64_t pt0 = P.tile_pt_ptr[t0], pt1 = P.tile_pt_ptr[t1];
  for (int64_t e = pt0 + tid; e < pt1; e += blockDim.x) {
    const int64_t b = P.e_ptr[e], n = P.e_ptr[e + 1];
    for (int64_t i = b; i < n; ++i) {
      const int si = P.ob_slot[i];
      atomicAdd(&camobs[si], 1);
      for (int64_t j = i + 1; j < n; ++j) {
        const int sj = P.ob_slot[j];
        if (si != sj) atomicAdd(&cnt[min(si, sj) * SA_NCS_MAX + max(si, sj)], 1);
      }
    }
  }
  __syncthreads();
  uint32_t* dslot = P.dslot + (size_t)strip * P.ncs_cap * P.ncs_cap;
  uint32_t* cslot = P.cslot + (size_t)strip * P.ncs_cap;
  uint32_t* sout = P.slot_out + (size_t)strip * SA_NT;
  uint16_t* sdest = P.slot_dest + (size_t)strip * SA_NT;
  for (int i = tid; i < P.ncs_cap * P.ncs_cap; i += blockDim.x) dslot[i] = 0xffffffffu;
  for (int i = tid; i < P.ncs_cap; i += blockDim.x) cslot[i] = 0u;
  for (int i = tid; i < SA_NT; i += blockDim.x) { sout[i] = 0u; sdest[i] = 0; }
  __syncthreads();
  __shared__ uint16_t item_ab[SA_NT], sort_ab[SA_NT];
  __shared__ int item_cnt[SA_NT], sort_cnt[SA_NT];
  __shared__ int sh[9];
  __shared__ double shd[1];
  __shared__ uint8_t cm[SA_NCS_MAX];
  if (tid == 0) {
  long long WC = 0, WP = 0;
  int n_pairs = 0, n_cact = 0, max_cnt = 0;
  for (int s = 0; s < ncs; ++s) { WC += camobs[s]; n_cact += camobs[s] > 0 ? 1 : 0; }
  for (int a = 0; a < ncs; ++a)
    for (int b = a + 1; b < ncs; ++b) {
      const int c = cnt[a * SA_NCS_MAX + b];
      if (c > 0) { WP += c; ++n_pairs; max_cnt = max(max_cnt, c); }
    }
  // camera threads: a fixed budget of whole warps, dealt over the cameras in proportion to their observations
  int n_cslots = 0;
  {
    // at least cam_budget threads; when the pairs of the strip leave threads over (a sparse problem), the cameras get
    // them: the camera threads are the longest lanes of phase B otherwise
    int budget = max(P.cam_budget, (n_cact + 31) & ~31);
    budget = max(budget, ((SA_NT - n_pairs) & ~31) - 32);
    budget = min(budget, min(SA_NT - 64, SA_CM_MAX * n_cact));
    budget = max(budget, n_cact);
    int used = 0;
    for (int s = 0; s < ncs; ++s) {
      int m = 0;
      if (camobs[s] > 0) m = min(SA_CM_MAX, 1 + (int)(((long long)(budget - n_cact) * camobs[s]) / max(WC, 1LL)));
      cm[s] = (uint8_t)m; used += m;
    }
    for (int round = 0; round < SA_CM_MAX && used < budget; ++round)   // what rounding down left over, one more each in camera order
      for (int s = 0; s < ncs && used < budget; ++s)
        if (camobs[s] > 0 && cm[s] < SA_CM_MAX) { ++cm[s]; ++used; }
    n_cslots = used;
  }
  const int cbase = SA_NT - n_cslots;
  const int avail = cbase;
  const double target = fmax((double)WP / max(avail, 1), 1e-9);   // pairs per pair thread and strip
  bool flush = false, ok = true;
  int mcap = 1, thr = 1, extra = 0, flush_t0 = -1;
  if (n_pairs <= avail) {
    mcap = n_pairs > 0 ? min(255, avail / n_pairs) : 1;
  } else {   // the lightest pairs go to one flush warp below the camera threads
    flush = true;
    const int fw = avail / 32 - 1;
    if (fw < 1) ok = false;
    flush_t0 = 32 * max(fw, 0);
    const int budget = flush_t0;
    // smallest threshold whose pairs fit; the remaining budget goes to pairs one count lighter, in slot order
    int lo = 1, hi = max_cnt + 1;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      int n = 0;
      for (int a = 0; a < ncs; ++a)
        for (int b = a + 1; b < ncs; ++b) n += cnt[a * SA_NCS_MAX + b] >= mid ? 1 : 0;
      if (n <= budget) hi = mid; else lo = mid + 1;
    }
    thr = lo;
    int n = 0;
    for (int a = 0; a < ncs; ++a)
      for (int b = a + 1; b < ncs; ++b) n += cnt[a * SA_NCS_MAX + b] >= thr ? 1 : 0;
    extra = budget - n;
  }
  // persistent pairs, collected in (diagonal, first camera) order; the lightest go to the flush list
  int npp = 0, nfl = 0;
  for (int d = 1; d < ncs && ok; ++d)
    for (int a = 0; a + d < ncs; ++a) {
      const int b = a + d, c = cnt[a * SA_NCS_MAX + b];
      if (c <= 0) continue;
      bool keep = true;
      if (flush) {
        keep = c >= thr;
        if (!keep && c == thr - 1 && extra > 0) { keep = true; --extra; }
      }
      if (keep) {
        item_ab[npp] = (uint16_t)((a << 8) | b);
        item_cnt[npp] = c;
        ++npp;
      } else {
        if (nfl >= P.nf_cap) { ok = false; break; }
        dslot[a * P.ncs_cap + b] = 0x80000000u | (uint32_t)nfl;
        P.fl_dest[(size_t)strip * P.nf_cap + nfl] = (uint16_t)((a << 8) | b);
        ++nfl;
      }
    }
  {
    int fw_pairs = 0;   // pair products of the flush list per strip
    for (int a = 0; a < ncs; ++a)
      for (int b = a + 1; b < ncs; ++b)
        if (dslot[a * P.ncs_cap + b] != 0xffffffffu && (dslot[a * P.ncs_cap + b] & 0x80000000u)) fw_pairs += cnt[a * SA_NCS_MAX + b];
    sh[8] = fw_pairs;
  }
  sh[0] = npp; sh[1] = nfl; sh[2] = ok ? 1 : 0; sh[3] = flush ? 1 : 0; sh[4] = mcap; sh[5] = flush_t0; sh[6] = n_cslots; sh[7] = n_cact;
  shd[0] = target;
  }
  __syncthreads();
  // Owner slots: in collection order -- (diagonal, first camera): a quarter warp owns eight pairs (a, a + d) with
  // consecutive a, whose records lie in eight different bank groups -- or (BA_SA_ORDER=1) by descending pair count, rank
  // sorted by all threads with ties in collection order.  Measured on the 30 M-observation problem the first is faster
  // (pass 1 5.6 vs 5.95 ms): the conflict-free gathers are worth more than lanes of equal length.
  const int npp = sh[0];
  for (int i = tid; i < npp; i += blockDim.x) {
    const int c = item_cnt[i];
    int r = i;
    if (P.by_count) {
      r = 0;
      for (int j = 0; j < npp; ++j) { const int cj = item_cnt[j]; r += (cj > c || (cj == c && j < i)) ? 1 : 0; }
    }
    sort_ab[r] = item_ab[i]; sort_cnt[r] = c;
  }
  __syncthreads();
  // inside every group of 32 (a warp): quarter warps whose eight pairs have eight different first-camera classes and
  // eight different second-camera classes (mod 8) where the group allows it, so that the records a quarter warp
  // gathers in one step lie in different bank groups
  if (P.arrange && tid < (npp + 31) / 32) {
    const int g0 = 32 * tid, n = min(32, npp - g0);
    uint16_t ab[32]; int cc[32]; bool used[32];
    for (int i = 0; i < n; ++i) { ab[i] = sort_ab[g0 + i]; cc[i] = sort_cnt[g0 + i]; used[i] = false; }
    int o = 0;
    for (int qd = 0; qd < 4 && o < n; ++qd) {
      unsigned ua = 0, ub = 0;
      int taken = 0;
      for (int i = 0; i < n && taken < 8; ++i) {
        if (used[i]) continue;
        const unsigned ca = 1u << ((ab[i] >> 8) & 7), cb = 1u << (ab[i] & 7);
        if ((ua & ca) || (ub & cb)) continue;
        ua |= ca; ub |= cb; used[i] = true; ++taken;
        sort_ab[g0 + o] = ab[i]; sort_cnt[g0 + o] = cc[i]; ++o;
      }
      for (int i = 0; i < n && taken < 8; ++i) {   // no conflict-free candidate left: fill in order
        if (used[i]) continue;
        used[i] = true; ++taken;
        sort_ab[g0 + o] = ab[i]; sort_cnt[g0 + o] = cc[i]; ++o;
      }
    }
  }
  __syncthreads();
  {
    const bool flush = sh[3] != 0;
    const int mcap = sh[4];
    const double target = shd[0];
    for (int r = tid; r < npp; r += blockDim.x) {
      const int a = sort_ab[r] >> 8, b = sort_ab[r] & 0xff;
      const int m = flush ? 1 : min(mcap, max(1, (int)((double)sort_cnt[r] / target + 0.5)));
      dslot[a * P.ncs_cap + b] = (uint32_t)r | ((uint32_t)m << 12);
      pdest[r] = sort_ab[r];
      pcopies[r] = (uint8_t)m;
      item_cnt[r] = sort_cnt[r] / m;   // pairs per owner thread of this pair (item_cnt is free now)
    }
  }
  __syncthreads();
  if (tid != 0) return;
  auto item_w = [&](int r) { return item_cnt[r]; };
  const bool ok = sh[2] != 0, flush = sh[3] != 0;
  const int nfl = sh[1], n_cslots = sh[6], n_cact = sh[7];
  int flush_t0 = sh[5];
  const int cbase = SA_NT - n_cslots;
  int npout = 0, ncout = 0;
  uint16_t* thr_of = P.thr_of + (size_t)strip * SA_NT;
  if (ok) {
    // logical slots: pairs (layer major), the flush warp, the camera threads at the top; lw[] = load of every logical warp
    // (steps of its fullest lane per strip; a camera observation costs about 1.3 pair products)
    float lw[SA_NT / 32];
    for (int w = 0; w < SA_NT / 32; ++w) lw[w] = 0.f;
    for (int l = 0; l < SA_NT; ++l) { sort_ab[l] = 0; sort_cnt[l] = 0; }   // logical slot tables (idle unless set below)
    int max_m = 0;
    for (int r = 0; r < npp; ++r) max_m = max(max_m, (int)pcopies[r]);
    for (int j = 0; j < max_m; ++j)
      for (int r = 0; r < npp; ++r)
        if (pcopies[r] > j) {
          const int t = j * npp + r;
          sort_ab[t] = pdest[r];                                  // logical slot -> destination (sort_ab / sort_cnt are free now)
          sort_cnt[t] = (SA_TYPE_PAIR << 30) | npout++;
          lw[t >> 5] = fmaxf(lw[t >> 5], (float)item_w(r));
        }
    if (flush) {
      for (int u = 0; u < 32; ++u) { sort_ab[flush_t0 + u] = 0; sort_cnt[flush_t0 + u] = (SA_TYPE_FLUSH << 30) | u; }
      lw[flush_t0 >> 5] = 1.5f * (float)sh[8] / 32.f + 4.f * ((nfl + 31) / 32);
    }
    int t = cbase;
    for (int j = 0; j < SA_CM_MAX; ++j)
      for (int s = 0; s < ncs; ++s)
        if (cm[s] > j) {
          sort_ab[t] = (uint16_t)s;
          sort_cnt[t] = (SA_TYPE_CAM << 30) | ncout++;
          lw[t >> 5] = fmaxf(lw[t >> 5], 1.3f * (float)camobs[s] / (float)cm[s]);
          ++t;
        }
    // warps -> sub-partitions (warp w runs on sub-partition w % 4): heaviest first into the lightest bin with room
    int phys[SA_NT / 32], fill[4] = {0, 0, 0, 0};
    float bin[4] = {0.f, 0.f, 0.f, 0.f};
    bool done[SA_NT / 32];
    for (int w = 0; w < SA_NT / 32; ++w) done[w] = false;
    for (int it = 0; it < SA_NT / 32; ++it) {
      int best = -1;
      for (int w = 0; w < SA_NT / 32; ++w)
        if (!done[w] && (best < 0 || lw[w] > lw[best])) best = w;
      int b = -1;
      for (int k = 0; k < 4; ++k)
        if (fill[k] < SA_NT / 128 && (b < 0 || bin[k] < bin[b])) b = k;
      done[best] = true;
      phys[best] = P.balance ? b + 4 * fill[b] : best;
      ++fill[b]; bin[b] += lw[best];
    }
    for (int l = 0; l < SA_NT; ++l) {
      const int ph = 32 * phys[l >> 5] + (l & 31);
      thr_of[l] = (uint16_t)ph;
      sout[ph] = (uint32_t)sort_cnt[l];
      sdest[ph] = sort_ab[l];
    }
    if (flush) flush_t0 = 32 * phys[flush_t0 >> 5];
    uint16_t* cthr = P.cthr + (size_t)strip * P.ncs_cap * SA_CM_MAX;
    t = cbase;
    for (int j = 0; j < SA_CM_MAX; ++j)
      for (int s = 0; s < ncs; ++s)
        if (cm[s] > j) { cthr[s * SA_CM_MAX + j] = thr_of[t]; ++t; }
    for (int s = 0; s < ncs; ++s) cslot[s] = cm[s];
  }
  int32_t* out = P.counts + 8 * (size_t)strip;
  out[0] = npout; out[1] = ncout; out[2] = nfl; out[3] = flush ? flush_t0 : -1; out[4] = npp; out[5] = n_cact; out[6] = cbase;
  out[7] = ok ? 1 : 0;
}

__global__ void k_sa_strip_desc(int n_strips, int L, int n_tiles, const int64_t* __restrict__ strip_cam_ptr, const int32_t* __restrict__ counts,
                                const int64_t* __restrict__ pout0, const int64_t* __restrict__ cout0, SaStrip* __restrict__ strips,
                                int* __restrict__ stat /* 0: all ok (min), 1: max nflush */) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_strips) return;
  const int32_t* c = counts + 8 * (size_t)s;
  SaStrip S;
  S.cam0 = strip_cam_ptr[s]; S.pout0 = pout0[s]; S.cout0 = cout0[s];
  S.tile0 = s * L; S.ntiles = min(L, n_tiles - s * L); S.ncs = (int32_t)(strip_cam_ptr[s + 1] - strip_cam_ptr[s]); S.nflush = c[2];
  S.flush_t0 = c[3]; S.npp = c[4]; S.ncact = c[5]; S.cbase = c[6];
  strips[s] = S;
  if (!c[7]) atomicMin(stat + 0, 0);
  atomicMax(stat + 1, c[2]);
}
__global__ void k_sa_widen3(int n, const int32_t* __restrict__ counts, int64_t* __restrict__ a, int64_t* __restrict__ b) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n) return;
  a[i] = i < n ? counts[8 * (size_t)i] : 0;
  b[i] = i < n ? counts[8 * (size_t)i + 1] : 0;
}

struct SaEntParams {
  int L, ncs_cap, segw, stage_cap;
  const SaTile* tiles; const SaStrip* strips;
  const int64_t* e_ptr; const int32_t* ob_e; const uint8_t* ob_slot; const uint16_t* pidx;
  const uint32_t* dslot; const uint32_t* cslot; const uint16_t* cthr; const uint16_t* thr_of;
  int32_t* ent; uint16_t* seg; int64_t* tile_nfl;
};
// owner slot and entry of the pair (l, l2) / of observation l; returns false when there is none
__device__ __forceinline__ int sa_pair_owner(const SaEntParams& P, const SaStrip& S, const uint32_t* dslot, const uint16_t* thr_of, int sa, int sb,
                                             int lp) {
  const uint32_t ds = dslot[sa * P.ncs_cap + sb];
  if (ds & 0x80000000u) return SA_NT + (int)(ds & 0xffffu);
  const int m = (int)((ds >> 12) & 0xffu);
  return thr_of[(int)(ds & 0xfffu) + (lp % m) * S.npp];
}
// One CTA per tile: counting sort of the tile's entries by owner slot (counts and offsets are exact integers; the
// order inside a segment is then made canonical by sorting the segment), segment table, flush outputs of the tile.
__global__ void __launch_bounds__(512) k_sa_tile_entries(SaEntParams P) {
  extern __shared__ int sm_i[];
  int* count = sm_i;                 // [segw]
  int* start = count + P.segw;       // [segw + 1]
  int* stage = start + P.segw + 1;   // [stage_cap]
  __shared__ int nfl_s;
  __shared__ int wtot[32];
  const int t = blockIdx.x, tid = threadIdx.x, nthr = blockDim.x;
  const SaTile T = P.tiles[t];
  const SaStrip S = P.strips[t / P.L];
  const uint32_t* dslot = P.dslot + (size_t)(t / P.L) * P.ncs_cap * P.ncs_cap;
  const uint32_t* cslot = P.cslot + (size_t)(t / P.L) * P.ncs_cap;
  const uint16_t* cthr = P.cthr + (size_t)(t / P.L) * P.ncs_cap * SA_CM_MAX;
  const uint16_t* thr_of = P.thr_of + (size_t)(t / P.L) * SA_NT;
  const int nv = SA_NT + S.nflush;
  for (int i = tid; i < P.segw; i += nthr) count[i] = 0;
  if (tid == 0) nfl_s = 0;
  __syncthreads();
  const bool staged = T.nent <= P.stage_cap;
  int32_t* dst = staged ? stage : P.ent + T.ent0;
  for (int pass = 0; pass < 2; ++pass) {
    for (int l = tid; l < T.nobs; l += nthr) {
      const int64_t o = T.ob0 + l;
      const int e = P.ob_e[o];
      const int lp = (int)(e - T.pt0);
      const int s = P.ob_slot[o], pos = P.pidx[T.pidx0 + l];
      {
        const int owner = cthr[s * SA_CM_MAX + lp % (int)cslot[s]];
        if (pass == 0) atomicAdd(&count[owner], 1);
        else dst[start[owner] + atomicAdd(&count[owner], 1)] = pos;
      }
      const int64_t end = P.e_ptr[e + 1];
      for (int64_t o2 = o + 1; o2 < end; ++o2) {
        const int s2 = P.ob_slot[o2], pos2 = P.pidx[T.pidx0 + (int)(o2 - T.ob0)];
        if (s2 == s) continue;
        const bool fwd = s < s2;
        const int owner = sa_pair_owner(P, S, dslot, thr_of, fwd ? s : s2, fwd ? s2 : s, lp);
        if (pass == 0) atomicAdd(&count[owner], 1);
        else dst[start[owner] + atomicAdd(&count[owner], 1)] = fwd ? (pos | (pos2 << 12)) : (pos2 | (pos << 12));
      }
    }
    __syncthreads();
    if (pass == 0) {
      {   // exclusive scan over <= 1536 + 1 owner slots: a run of consecutive slots per thread, warp scans, the warp totals by warp 0
        const int per = (P.segw + nthr - 1) / nthr;
        const int v0 = tid * per, v1 = min(v0 + per, P.segw);
        int mine = 0;
        for (int v = v0; v < v1; ++v) mine += count[v];
        int incl = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int y = __shfl_up_sync(0xffffffffu, incl, o);
          if ((tid & 31) >= o) incl += y;
        }
        if ((tid & 31) == 31) wtot[tid >> 5] = incl;
        __syncthreads();
        if (tid < 32) {
          const int nw = nthr >> 5;
          int t = tid < nw ? wtot[tid] : 0;
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, t, o);
            if (tid >= o) t += y;
          }
          if (tid < nw) wtot[tid] = t;   // inclusive totals of the warps
        }
        __syncthreads();
        int a = incl - mine + ((tid >> 5) > 0 ? wtot[(tid >> 5) - 1] : 0);
        for (int v = v0; v < v1; ++v) { start[v] = a; a += count[v]; }
        if (tid == nthr - 1) start[P.segw] = wtot[(nthr >> 5) - 1];
      }
      __syncthreads();
      for (int v = tid; v < P.segw; v += nthr) {
        P.seg[(size_t)t * P.segw + v] = (uint16_t)start[v];
        if (v >= SA_NT && v < nv && count[v] > 0) atomicAdd(&nfl_s, 1);
        count[v] = 0;
      }
      __syncthreads();
    }
  }
  // canonical order inside every segment
  for (int v = tid; v < nv; v += nthr) {
    const int b = start[v], n = start[v + 1];
    for (int i = b + 1; i < n; ++i) {
      const int32_t x = dst[i];
      int j = i - 1;
      while (j >= b && dst[j] > x) { dst[j + 1] = dst[j]; --j; }
      dst[j + 1] = x;
    }
  }
  __syncthreads();
  if (staged)
    for (int i = tid; i < T.nent; i += nthr) P.ent[T.ent0 + i] = i < start[P.segw] ? stage[i] : 0;
  if (tid == 0) P.tile_nfl[t] = nfl_s;
}
__global__ void k_sa_set_fout(int n_tiles, const int64_t* __restrict__ fout0, SaTile* __restrict__ tiles) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n_tiles) tiles[t].fout0 = fout0[t];
}
// targets of the persistent outputs: one thread per (strip, owner slot)
__global__ void k_sa_targets_persist(int n_strips, const SaStrip* __restrict__ strips, const uint32_t* __restrict__ slot_out,
                                     const uint16_t* __restrict__ slot_dest, const int32_t* __restrict__ strip_cams, int64_t nf,
                                     const uint64_t* __restrict__ dh_keys, const int32_t* __restrict__ dh_val, uint64_t dh_mask, int dh_shift,
                                     int32_t* __restrict__ ptarget, int32_t* __restrict__ ctarget) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= (int64_t)n_strips * SA_NT) return;
  const int s = (int)(i / SA_NT);
  const uint32_t so = slot_out[i];
  const int type = (int)(so >> 30), rank = (int)(so & 0x3fffffffu);
  const SaStrip S = strips[s];
  const uint16_t d = slot_dest[i];
  if (type == SA_TYPE_PAIR) {
    const uint64_t ca = (uint64_t)strip_cams[S.cam0 + (d >> 8)], cb = (uint64_t)strip_cams[S.cam0 + (d & 0xff)];
    ptarget[S.pout0 + rank] = dh_find(dh_keys, dh_val, dh_mask, dh_shift, ca * (uint64_t)nf + cb);
  } else if (type == SA_TYPE_CAM) {
    ctarget[S.cout0 + rank] = strip_cams[S.cam0 + d];
  }
}
// targets of the flush outputs: one warp per tile, the same ballot ranks the flush warp of pass 1 computes
__global__ void k_sa_targets_flush(int n_tiles, int L, int segw, int nf_cap, const SaTile* __restrict__ tiles, const SaStrip* __restrict__ strips,
                                   const uint16_t* __restrict__ seg, const uint16_t* __restrict__ fl_dest, const int32_t* __restrict__ strip_cams,
                                   int64_t nf, const uint64_t* __restrict__ dh_keys, const int32_t* __restrict__ dh_val, uint64_t dh_mask,
                                   int dh_shift, int64_t n_pout, int32_t* __restrict__ ptarget) {
  const int t = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (t >= n_tiles) return;
  const int strip = t / L;
  const SaStrip S = strips[strip];
  const uint16_t* sg = seg + (size_t)t * segw + SA_NT;
  int64_t base = n_pout + tiles[t].fout0;
  for (int f0 = 0; f0 < S.nflush; f0 += 32) {
    const int f = f0 + lane;
    const bool on = f < S.nflush && sg[f + 1] > sg[f];
    const unsigned m = __ballot_sync(0xffffffffu, on);
    if (on) {
      const uint16_t d = fl_dest[(size_t)strip * nf_cap + f];
      const uint64_t ca = (uint64_t)strip_cams[S.cam0 + (d >> 8)], cb = (uint64_t)strip_cams[S.cam0 + (d & 0xff)];
      ptarget[base + __popc(m & ((1u << lane) - 1u))] = dh_find(dh_keys, dh_val, dh_mask, dh_shift, ca * (uint64_t)nf + cb);
    }
    base += __popc(m);
  }
}
// FaTile descriptors for pass 2 / k_fa_jac on the same tiles (camera list = the strip's)
__global__ void k_sa_fa_tiles(int n_tiles, int L, const SaTile* __restrict__ tiles, const SaStrip* __restrict__ strips, FaTile* __restrict__ out) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_tiles) return;
  const SaTile T = tiles[t];
  const SaStrip S = strips[t / L];
  FaTile F;
  F.pt0 = T.pt0; F.ob0 = T.ob0; F.cam0 = S.cam0; F.pe0 = 0; F.ce0 = 0; F.pitem0 = 0; F.citem0 = 0;
  F.npts = T.npts; F.nobs = T.nobs; F.ncam = S.ncs; F.npe = 0; F.nce = 0; F.npitem = 0; F.ncitem = 0;
  F.pad_[0] = F.pad_[1] = F.pad_[2] = 0;
  out[t] = F;
}

inline int sa_exclusive_scan(const DVec<int64_t>& in, DVec<int64_t>& out, int n_plus_1, cudaStream_t st) {
  BA_TRY(out.alloc((size_t)n_plus_1));
  return cub_call([&](void* t, size_t& b) { return cub::DeviceScan::ExclusiveSum(t, b, in.p, out.p, n_plus_1, st); });
}

// Builds the strip structure of a Model A problem, and fills the tile structure of `F` (descriptors, per-observation
// words, geometry) that pass 2 and k_fa_jac run on.  BA_ERR_UNSUPPORTED: the problem does not fit (a strip with more
// than SA_NCS_MAX cameras even at one tile per strip, a point seen twice by one camera, a point with more than FA_KMAX
// observations ...); the caller then uses the first-generation fused path.
inline int build_strip_a_geom(StripA& A, FusedA& F, const Structure& S, const double2* uv, cudaStream_t st, int tobs, int L);

inline int build_strip_a(StripA& A, FusedA& F, const Structure& S, const double2* uv, cudaStream_t st) {
  A.ready = false;
  if (S.ne == 0 || S.nb == 0 || S.nslots != 1 || S.dh_keys.n == 0) return BA_ERR_UNSUPPORTED;
  // BA_SA: 0 = never, 2 = whenever the problem fits, 1 (default) = when it fits and pays: measured on B200, strips win
  // on problems with many pair products per observation (30 M observations, 4.8 pairs each: 5.5 vs 6.9 ms for pass 1 +
  // reduction; 8-camera rig, 4.5: 0.44 vs 1.2 ms) and lose on sparse ones (5 M observations, 3 pairs each: 1.02 vs 0.66 ms)
  const int mode = env_int("BA_SA", 0, 2, 1);
  if (mode == 0) return BA_ERR_UNSUPPORTED;
  if (mode == 1 && (double)(S.npairs - S.nf) < 4.0 * (double)S.nb) return BA_ERR_UNSUPPORTED;
  int tobs = env_int("BA_SA_TOBS", 64, 2048, 832);   // measured on the 30 M-observation problem: 576 .. 896 within 8 %, 832 best
  int L = env_int("BA_SA_L", 1, 64, 8);
  for (int attempt = 0; attempt < 8; ++attempt) {
    const int rc = build_strip_a_geom(A, F, S, uv, st, tobs, L);
    if (rc != BA_ERR_UNSUPPORTED) return rc;
    if (A.kmax > FA_KMAX) return rc;
    // too many cameras in a strip: shorter strips first; shared memory does not fit: smaller tiles
    if (A.ncs_cap > SA_NCS_MAX && L > 1) L = L / 2;
    else if (tobs > 128) tobs = tobs * 3 / 4 / 32 * 32;
    else return rc;
  }
  return BA_ERR_UNSUPPORTED;
}

inline int build_strip_a_geom(StripA& A, FusedA& F, const Structure& S, const double2* uv, cudaStream_t st, int tobs, int L) {
  A.ready = false; F.ready = false;
  const int64_t ne = S.ne, nb = S.nb, nf = S.nf;
  A.tobs = tobs; A.L = L;
  FaLap Lp(st);
  // 1. tiles of consecutive points
  DVec<int32_t> flag, tile_of_pt;
  DVec<int> kmax;
  BA_TRY(flag.alloc(ne)); BA_TRY(tile_of_pt.alloc(ne)); BA_TRY(kmax.alloc_zero(1, st));
  k_fa_tile_flags<<<grid_for(ne, 256), 256, 0, st>>>(S.e_ptr.p, ne, tobs, flag.p, kmax.p);
  BA_TRY(cub_call([&](void* t, size_t& b) { return cub::DeviceScan::InclusiveSum(t, b, flag.p, tile_of_pt.p, (int)ne, st); }));
  int last_tile = 0;
  BA_CUDA_TRY(cudaMemcpyAsync(&A.kmax, kmax.p, sizeof(int), cudaMemcpyDeviceToHost, st));
  BA_CUDA_TRY(cudaMemcpyAsync(&last_tile, tile_of_pt.p + (ne - 1), sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  BA_CUDA_TRY(cudaStreamSynchronize(st));
  if (A.kmax > FA_KMAX) return BA_ERR_UNSUPPORTED;
  const int nt = last_tile + 1;
  A.n_tiles = nt;
  A.n_strips = (nt + L - 1) / L;
  const int ns = A.n_strips;
  BA_TRY(A.tile_pt_ptr.alloc((size_t)nt + 1));
  k_seg_ptr<int32_t><<<grid_for(ne > nt + 1 ? ne : nt + 1, 256), 256, 0, st>>>(tile_of_pt.p, ne, nt, A.tile_pt_ptr.p);
  // 2. camera list of every strip (sorted), camera slot of every observation
  int ng = 0;
  {
    DVec<uint64_t> keys, sorted, uniq;
    DVec<int> nu;
    DVec<int32_t> gstrip;
    BA_TRY(keys.alloc(nb)); BA_TRY(sorted.alloc(nb)); BA_TRY(uniq.alloc(nb)); BA_TRY(nu.alloc(1));
    k_sa_strip_keys<<<grid_for(nb, 256), 256, 0, st>>>(nb, S.ob_e.p, S.ob_f0.p, tile_of_pt.p, L, nf, keys.p);
    const int bits = bits_for((uint64_t)ns * (uint64_t)nf);
    BA_TRY(cub_call([&](void* t, size_t& b) { return cub::DeviceRadixSort::SortKeys(t, b, keys.p, sorted.p, (int)nb, 0, bits, st); }));
    BA_TRY(cub_call([&](void* t, size_t& b) { return cub::DeviceSelect::Unique(t, b, sorted.p, uniq.p, nu.p, (int)nb, st); }));
    BA_CUDA_TRY(cudaMemcpyAsync(&ng, nu.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    BA_CUDA_TRY(cudaStreamSynchronize(st));
    BA_TRY(gstrip.alloc(ng)); BA_TRY(A.strip_cams.alloc(ng)); BA_TRY(A.strip_cam_ptr.alloc((size_t)ns + 1));
    k_sa_split_keys<<<grid_for(ng, 256), 256, 0, st>>>(ng, uniq.p, nf, gstrip.p, A.strip_cams.p);
    k_seg_ptr<int32_t><<<grid_for(ng > ns + 1 ? ng : ns + 1, 256), 256, 0, st>>>(gstrip.p, ng, ns, A.strip_cam_ptr.p);
    DVec<int> mx;
    BA_TRY(mx.alloc_zero(1, st));
    k_fa_max_diff<<<grid_for(ns, 256), 256, 0, st>>>(ns, A.strip_cam_ptr.p, mx.p);
    BA_CUDA_TRY(cudaMemcpyAsync(&A.ncs_cap, mx.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    BA_CUDA_TRY(cudaStreamSynchronize(st));
  }
  if (A.ncs_cap > SA_NCS_MAX) return BA_ERR_UNSUPPORTED;
  A.ncs_cap = std::max(A.ncs_cap, 1);
  Lp.lap("strip: tiles, cameras");
  DVec<uint8_t> ob_slot;
  BA_TRY(ob_slot.alloc(nb)); BA_TRY(A.ob_meta.alloc(nb));
  k_sa_obs_slot<<<grid_for(nb, 256), 256, 0, st>>>(nb, S.ob_e.p, S.ob_f0.p, tile_of_pt.p, A.tile_pt_ptr.p, L, A.strip_cam_ptr.p, A.strip_cams.p,
                                                   ob_slot.p, A.ob_meta.p);
  // 3. per tile sizes, bases of the per-tile slices
  DVec<int64_t> t_npos, t_nent, t_npidx, pos0, ent0, pidx0;
  DVec<int> stat;
  BA_TRY(t_npos.alloc_zero((size_t)nt + 1, st)); BA_TRY(t_nent.alloc_zero((size_t)nt + 1, st)); BA_TRY(t_npidx.alloc_zero((size_t)nt + 1, st));
  BA_TRY(stat.alloc_zero(8, st));
  k_sa_tile_sizes<<<nt, 256, 0, st>>>(nt, L, A.tile_pt_ptr.p, S.e_ptr.p, ob_slot.p, A.strip_cam_ptr.p, t_npos.p, t_nent.p, t_npidx.p, stat.p);
  BA_TRY(sa_exclusive_scan(t_npos, pos0, nt + 1, st)); BA_TRY(sa_exclusive_scan(t_nent, ent0, nt + 1, st));
  BA_TRY(sa_exclusive_scan(t_npidx, pidx0, nt + 1, st));
  int h[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  int64_t tot[3] = {0, 0, 0};
  BA_CUDA_TRY(cudaMemcpyAsync(h, stat.p, sizeof(h), cudaMemcpyDeviceToHost, st));
  BA_CUDA_TRY(cudaMemcpyAsync(&tot[0], pos0.p + nt, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  BA_CUDA_TRY(cudaMemcpyAsync(&tot[1], ent0.p + nt, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  BA_CUDA_TRY(cudaMemcpyAsync(&tot[2], pidx0.p + nt, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  BA_CUDA_TRY(cudaStreamSynchronize(st));
  if (h[4] != 0 || h[0] > SA_POS_MAX || h[2] > 65532) return BA_ERR_UNSUPPORTED;
  A.cap_pos = std::max(8, h[0]); A.pts_cap = std::max(1, h[1]); A.nobs_cap = h[3]; A.pidx_cap = std::max(16, h[5]);
  A.tcs = A.ncs_cap | 1;
  const int max_nent = h[2];
  // 4. positions, position-ordered inputs, descriptors
  BA_TRY(A.tiles.alloc((size_t)nt)); BA_TRY(A.pm.alloc_zero((size_t)tot[0] + 8, st)); BA_TRY(A.puv.alloc((size_t)tot[0] + 8));
  BA_TRY(A.pidx.alloc_zero((size_t)tot[2] + 16, st));
  k_sa_tile_fill<<<nt, 256, 0, st>>>(nt, L, A.tile_pt_ptr.p, S.e_ptr.p, S.ob_e.p, ob_slot.p, uv, A.strip_cam_ptr.p, pos0.p, ent0.p, pidx0.p,
                                    t_npos.p, t_nent.p, A.tiles.p, A.pm.p, A.puv.p, A.pidx.p);
  Lp.lap("strip: positions");
  // 5. owner slots per strip
  const int nf_cap = std::min(SA_NF_CAP, std::max(8, A.ncs_cap * A.ncs_cap / 2));
  DVec<uint32_t> dslot, cslot;
  DVec<uint16_t> slot_dest, fl_dest, cthr, thr_of;
  DVec<int32_t> counts;
  BA_TRY(dslot.alloc((size_t)ns * A.ncs_cap * A.ncs_cap)); BA_TRY(cslot.alloc((size_t)ns * A.ncs_cap));
  BA_TRY(A.slot_out.alloc((size_t)ns * SA_NT)); BA_TRY(slot_dest.alloc((size_t)ns * SA_NT)); BA_TRY(fl_dest.alloc((size_t)ns * nf_cap));
  BA_TRY(counts.alloc((size_t)ns * 8)); BA_TRY(cthr.alloc((size_t)ns * A.ncs_cap * SA_CM_MAX)); BA_TRY(thr_of.alloc((size_t)ns * SA_NT));
  {
    SaPlanParams P;
    P.n_strips = ns; P.L = L; P.n_tiles = nt; P.ncs_cap = A.ncs_cap; P.nf_cap = nf_cap;
    P.cam_budget = env_int("BA_SA_NCAM", 32, 256, 64) / 32 * 32;
    P.by_count = env_int("BA_SA_ORDER", 0, 1, 0);
    P.balance = env_int("BA_SA_BALANCE", 0, 1, 1);
    P.arrange = env_int("BA_SA_ARRANGE", 0, 1, P.by_count);   // measured: no gain in (diagonal, camera) order
    P.tile_pt_ptr = A.tile_pt_ptr.p; P.e_ptr = S.e_ptr.p; P.ob_slot = ob_slot.p; P.strip_cam_ptr = A.strip_cam_ptr.p;
    P.dslot = dslot.p; P.cslot = cslot.p; P.cthr = cthr.p; P.slot_out = A.slot_out.p; P.slot_dest = slot_dest.p; P.fl_dest = fl_dest.p;
    P.thr_of = thr_of.p;
    P.counts = counts.p;
    k_sa_strip_plan<<<ns, 256, 0, st>>>(P);
  }
  DVec<int64_t> c_p, c_c, pout0, cout0;
  BA_TRY(c_p.alloc((size_t)ns + 1)); BA_TRY(c_c.alloc((size_t)ns + 1));
  k_sa_widen3<<<grid_for(ns + 1, 256), 256, 0, st>>>(ns, counts.p, c_p.p, c_c.p);
  BA_TRY(sa_exclusive_scan(c_p, pout0, ns + 1, st)); BA_TRY(sa_exclusive_scan(c_c, cout0, ns + 1, st));
  BA_TRY(A.strips.alloc((size_t)ns));
  {
    const int init[2] = {1, 0};
    BA_CUDA_TRY(cudaMemcpyAsync(stat.p, init, sizeof(init), cudaMemcpyHostToDevice, st));
    k_sa_strip_desc<<<grid_for(ns, 256), 256, 0, st>>>(ns, L, nt, A.strip_cam_ptr.p, counts.p, pout0.p, cout0.p, A.strips.p, stat.p);
    BA_CUDA_TRY(cudaMemcpyAsync(h, stat.p, sizeof(int) * 2, cudaMemcpyDeviceToHost, st));
    BA_CUDA_TRY(cudaMemcpyAsync(&A.n_pout, pout0.p + ns, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    BA_CUDA_TRY(cudaMemcpyAsync(&A.n_cout, cout0.p + ns, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    BA_CUDA_TRY(cudaStreamSynchronize(st));
  }
  if (h[0] != 1) return BA_ERR_UNSUPPORTED;
  A.segw = (SA_NT + h[1] + 1 + 7) & ~7;
  Lp.lap("strip: owner plan");
  // shared-memory geometry of pass 1: stage as many entries as fit
  A.ent_cap = max_nent;
  if (A.smem() > FA_SMEM_MAX) {
    const size_t excess = (A.smem() - FA_SMEM_MAX + 15) / 16 * 4;
    if ((size_t)A.ent_cap <= excess) return BA_ERR_UNSUPPORTED;
    A.ent_cap = (int)(A.ent_cap - excess) & ~3;
    if (A.ent_cap < max_nent / 2) return BA_ERR_UNSUPPORTED;   // retried with smaller tiles
  }
  // 6. entries by owner slot
  BA_TRY(A.ent.alloc((size_t)tot[1] + 8)); BA_TRY(A.seg.alloc((size_t)nt * A.segw + 8));
  DVec<int64_t> t_nfl, fout0;
  BA_TRY(t_nfl.alloc_zero((size_t)nt + 1, st));
  {
    SaEntParams P;
    P.L = L; P.ncs_cap = A.ncs_cap; P.segw = A.segw; P.stage_cap = 12288;
    P.tiles = A.tiles.p; P.strips = A.strips.p; P.e_ptr = S.e_ptr.p; P.ob_e = S.ob_e.p; P.ob_slot = ob_slot.p; P.pidx = A.pidx.p;
    P.dslot = dslot.p; P.cslot = cslot.p; P.cthr = cthr.p; P.thr_of = thr_of.p; P.ent = A.ent.p; P.seg = A.seg.p; P.tile_nfl = t_nfl.p;
    const size_t sm = ((size_t)2 * A.segw + 1 + P.stage_cap) * sizeof(int);
    BA_CUDA_TRY(cudaFuncSetAttribute(k_sa_tile_entries, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    k_sa_tile_entries<<<nt, 512, sm, st>>>(P);
  }
  BA_TRY(sa_exclusive_scan(t_nfl, fout0, nt + 1, st));
  k_sa_set_fout<<<grid_for(nt, 256), 256, 0, st>>>(nt, fout0.p, A.tiles.p);
  BA_CUDA_TRY(cudaMemcpyAsync(&A.n_fout, fout0.p + nt, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  BA_CUDA_TRY(cudaStreamSynchronize(st));
  BA_CUDA_TRY(cudaGetLastError());
  Lp.lap("strip: entries");
  // 7. reduction lists over the partial blocks
  const int64_t n_pblocks = A.n_pout + A.n_fout;
  if (n_pblocks >= (int64_t)INT32_MAX / 64 || A.n_cout >= (int64_t)INT32_MAX / 64) return BA_ERR_UNSUPPORTED;
  {
    DVec<int32_t> ptarget, ctarget, iota;
    BA_TRY(ptarget.alloc((size_t)n_pblocks)); BA_TRY(ctarget.alloc((size_t)A.n_cout));
    k_sa_targets_persist<<<grid_for((int64_t)ns * SA_NT, 256), 256, 0, st>>>(ns, A.strips.p, A.slot_out.p, slot_dest.p, A.strip_cams.p, nf,
                                                                            S.dh_keys.p, S.dh_val.p, S.dh_mask, S.dh_shift, ptarget.p, ctarget.p);
    k_sa_targets_flush<<<grid_for(nt, 4), 128, 0, st>>>(nt, L, A.segw, nf_cap, A.tiles.p, A.strips.p, A.seg.p, fl_dest.p, A.strip_cams.p, nf,
                                                       S.dh_keys.p, S.dh_val.p, S.dh_mask, S.dh_shift, A.n_pout, ptarget.p);
    const int64_t nmax = std::max(n_pblocks, A.n_cout);
    BA_TRY(iota.alloc((size_t)nmax));
    k_iota<<<grid_for(nmax, 256), 256, 0, st>>>(iota.p, nmax, 0);
    BA_TRY(sort_to_csr(ptarget.p, iota.p, n_pblocks, S.ndest, A.red_pairs.tgt_ptr, A.red_pairs.items, st));
    BA_TRY(build_chunks(A.red_pairs.ch, A.red_pairs.tgt_ptr.p, S.ndest, FA_CH_RED, st));
    BA_TRY(sort_to_csr(ctarget.p, iota.p, A.n_cout, nf, A.red_cams.tgt_ptr, A.red_cams.items, st));
    BA_TRY(build_chunks(A.red_cams.ch, A.red_cams.tgt_ptr.p, (int)nf, FA_CH_RED, st));
    BA_CUDA_TRY(cudaStreamSynchronize(st));
  }
  Lp.lap("strip: reduction lists");
  BA_TRY(A.red_pairs.part.alloc((size_t)n_pblocks * 36)); BA_TRY(A.red_cams.part.alloc((size_t)A.n_cout * SA_NVC));
  BA_TRY(A.red_pairs.red1.alloc((size_t)A.red_pairs.ch.n * 36)); BA_TRY(A.red_cams.red1.alloc((size_t)A.red_cams.ch.n * SA_NVC));
  // 8. the tile structure pass 2 and k_fa_jac run on
  F.n_tiles = nt; F.tobs = tobs; F.kmax = A.kmax; F.cap = std::max(A.nobs_cap, 1);
  F.threads = SA_NT; F.threads2 = env_int("BA_FA_THREADS2", 32, FA_MAX_THREADS, tobs >= 640 ? 256 : 128) / 32 * 32;
  F.pts_cap = A.pts_cap; F.tcam = std::min(A.ncs_cap, FA_TCAM); F.tcs = F.tcam | 1; F.pent_cap = 0;
  if (F.smem2() > FA_SMEM_MAX || F.smemj(FA_JAC_THREADS) > FA_SMEM_MAX) return BA_ERR_UNSUPPORTED;
  BA_TRY(F.tiles.alloc((size_t)nt));
  k_sa_fa_tiles<<<grid_for(nt, 256), 256, 0, st>>>(nt, L, A.tiles.p, A.strips.p, F.tiles.p);
  BA_TRY(F.camacc.alloc((size_t)nf * SA_NVC + 2 + 64));
  BA_TRY(F.Lz.alloc((size_t)ne * 9));
  BA_CUDA_TRY(cudaStreamSynchronize(st));
  BA_CUDA_TRY(cudaGetLastError());
  if (Lp.on)
    std::fprintf(stderr, "[ba_cuda timing]   strip geometry: tobs %d L %d tiles %d strips %d | positions %d points %d cameras %d entries staged %d of %d "
                         "owner slots %d | smem %zu B | blocks: %lld per strip + %lld flushed, %lld camera\n", tobs, L, nt, ns, A.cap_pos, A.pts_cap,
                 A.ncs_cap, A.ent_cap, max_nent, A.segw, A.smem(), (long long)A.n_pout, (long long)A.n_fout, (long long)A.n_cout);
  A.ready = true; F.ready = true;
  return BA_OK;
}

// ---------------------------------------------------------------------------------------
// pass 1
// ---------------------------------------------------------------------------------------
struct SaParams {
  const SaStrip* strips; const SaTile* tiles; const int32_t* strip_cams; const uint32_t* slot_out;
  const uint32_t* pm; const double2* puv; const uint16_t* pidx; const int32_t* ent; const uint16_t* seg;
  int segw, cap_pos, pts_cap, tcs, ent_cap, pidx_cap;
  const double* xe; const double* se; const double* tab_f; const double* radius;
  double min_diag, max_diag;
  double* partP; double* partC; int64_t n_pout;
  double* Lz; double* se_out; double* cost_partial; double* g2_partial; double* gmax_partial; int* status;
  int dbg;   // BA_SA_DBG (timing experiments only, results are wrong): 1 skips the pair products, 2 the camera sums, 4 the point phases
  unsigned long long* clocks;   // BA_SA_CLOCKS: [8] cycles per phase, summed over the CTAs by thread 0 of each (nullptr: off)
  LossSpec loss;                // robust loss on every observation (type 0 = none, the reference)
};

__device__ __forceinline__ uint32_t sa_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void sa_mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(sa_smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void sa_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(sa_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void sa_mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok = 0;
  const uint32_t a = sa_smem_u32(bar);
  do {
    asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
                 : "=r"(ok) : "r"(a), "r"(parity) : "memory");
  } while (!ok);
}
// contiguous global -> shared copy by the TMA engine; both addresses 16-byte aligned, bytes a multiple of 16
__device__ __forceinline__ void sa_bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(sa_smem_u32(dst)), "l"(src), "r"(bytes), "r"(sa_smem_u32(bar)) : "memory");
}

template <int MODE>
__global__ void __launch_bounds__(SA_NT, 1) k_sa_pass1(SaParams P) {
  constexpr bool FIRST = MODE == SA_FIRST, FULL = MODE == SA_FULL || FIRST, UNIT = FIRST;
  extern __shared__ __align__(128) double smem[];
  double* rec = smem;                                          // [cap_pos][SA_REC]
  double* tabs = rec + (size_t)P.cap_pos * SA_REC;             // table planes [2 TAB][tcs] x 32 bit
  double* xs = tabs + (size_t)P.tcs * TAB;                     // [3 pts_cap + 4] points of the tile (16-byte aligned slice)
  double* ss = xs + sa_xs_len(P.pts_cap);                      // [3 pts_cap + 4] their Jacobi scaling
  double2* puv_s = reinterpret_cast<double2*>(ss + sa_xs_len(P.pts_cap));   // [cap_pos]
  uint32_t* pm_s = reinterpret_cast<uint32_t*>(puv_s + P.cap_pos);       // [cap_pos]
  uint16_t* pidx_s = reinterpret_cast<uint16_t*>(pm_s + P.cap_pos);      // [pidx_cap]
  int32_t* ent_s = reinterpret_cast<int32_t*>(pidx_s + P.pidx_cap);      // [ent_cap]
  uint16_t* seg_s = reinterpret_cast<uint16_t*>(ent_s + P.ent_cap);      // [segw]
  uint64_t* bars = reinterpret_cast<uint64_t*>(seg_s + P.segw);          // [2]
  __shared__ double red[96];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const SaStrip S = P.strips[blockIdx.x];
  const uint32_t so = P.slot_out[(size_t)blockIdx.x * SA_NT + tid];
  const int ttype = (int)(so >> 30);
  const int orank = (int)(so & 0x3fffffffu);
  // the thread that issues the bulk copies (each costs it a few hundred cycles): lane 0 of the flush warp -- or of the
  // last warp --, which has one round of A1 at most and little to do in B, so the copies are off the critical path
  const bool producer = tid == (S.flush_t0 >= 0 ? S.flush_t0 : SA_NT - 32);

  // one thread issues the bulk copies of a tile's inputs; group 1: what A1 / A2a read, group 2: what B reads
  auto issue_g1 = [&](const SaTile& T) {
    const uint32_t b_uv = (uint32_t)T.npos * 16u, b_pm = (uint32_t)T.npos * 4u;
    const uint32_t n_idx = (uint32_t)(((T.nobs + 7) & ~7) + ((T.npts + 1 + 7) & ~7));
    const uint32_t b_idx = n_idx * 2u;
    const int64_t x0 = (3 * T.pt0) & ~(int64_t)1;
    const uint32_t b_x = (uint32_t)((3 * T.pt0 + 3 * T.npts - x0 + 1) & ~(int64_t)1) * 8u;
    sa_mbar_expect_tx(bars + 0, b_uv + b_pm + b_idx + (UNIT ? b_x : 2 * b_x));
    sa_bulk_g2s(puv_s, P.puv + T.pos0, b_uv, bars + 0);
    sa_bulk_g2s(pm_s, P.pm + T.pos0, b_pm, bars + 0);
    sa_bulk_g2s(pidx_s, P.pidx + T.pidx0, b_idx, bars + 0);
    sa_bulk_g2s(xs, P.xe + x0, b_x, bars + 0);
    if (!UNIT) sa_bulk_g2s(ss, P.se + x0, b_x, bars + 0);
  };
  auto issue_g2 = [&](const SaTile& T, int tile) {
    const uint32_t b_ent = (uint32_t)min(T.nent, P.ent_cap) * 4u, b_seg = (uint32_t)P.segw * 2u;
    sa_mbar_expect_tx(bars + 1, b_ent + b_seg);
    if (b_ent) sa_bulk_g2s(ent_s, P.ent + T.ent0, b_ent, bars + 1);
    sa_bulk_g2s(seg_s, P.seg + (size_t)tile * P.segw, b_seg, bars + 1);
  };

  if (tid == 0) {
    sa_mbar_init(bars + 0, 1);
    sa_mbar_init(bars + 1, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  {  // the strip's camera tables -> 32-bit planes (as fa_stage_tables_async)
    const int nw = SA_NT >> 5;
    uint32_t* planes = reinterpret_cast<uint32_t*>(tabs);
    for (int s = warp; s < S.ncs; s += nw) {
      const int32_t cam = __ldg(P.strip_cams + S.cam0 + s);
      const uint32_t* src = reinterpret_cast<const uint32_t*>(P.tab_f + (int64_t)TAB * cam + lane);
      uint32_t* dst = planes + (size_t)(2 * lane) * P.tcs + s;
      __pipeline_memcpy_async(dst, src, 4);
      __pipeline_memcpy_async(dst + P.tcs, src + 1, 4);
    }
    __pipeline_commit();
    __pipeline_wait_prior(0);
  }
  __syncthreads();
  if (producer) {
    const SaTile T0 = P.tiles[S.tile0];
    issue_g1(T0);
    issue_g2(T0, S.tile0);
  }
  double acc[SA_NVC];
#pragma unroll
  for (int k = 0; k < SA_NVC; ++k) acc[k] = 0.0;
  double sq = 0.0, gmx = 0.0, g2 = 0.0;
  const double inv_radius = 1.0 / *P.radius;
  uint32_t ph1 = 0, ph2 = 0;
  long long ck[7] = {0, 0, 0, 0, 0, 0, 0}, c_last = clock64();
  auto tick = [&](int k) { if (P.clocks && tid == 0) { const long long c = clock64(); ck[k] += c - c_last; c_last = c; } };

  // the descriptor of a tile is fetched one tile ahead (a dependent global load at the top of every tile would stall
  // the whole CTA for its latency)
  SaTile Tn;
  auto load_desc = [&](int tile) {
    const int4* s4 = reinterpret_cast<const int4*>(P.tiles + tile);
    int4* d4 = reinterpret_cast<int4*>(&Tn);
#pragma unroll
    for (int k = 0; k < 4; ++k) d4[k] = __ldg(s4 + k);
  };
  load_desc(S.tile0);
  for (int ti = 0; ti < S.ntiles; ++ti) {
    const int tile = S.tile0 + ti;
    const SaTile T = Tn;
    if (ti + 1 < S.ntiles) load_desc(tile + 1);
    const int npos = T.npos, npts = T.npts;
    const int xoff = (int)((3 * T.pt0) & 1);
    const uint16_t* pbeg = pidx_s + ((T.nobs + 7) & ~7);
    tick(0);
    sa_mbar_wait(bars + 0, ph1); ph1 ^= 1u;
    tick(1);
    // ---- A1: one thread per record position ----
    for (int pos = tid; pos < npos; pos += SA_NT) {
      const uint32_t m = pm_s[pos];
      double2* R2 = reinterpret_cast<double2*>(rec + (size_t)pos * SA_REC);
      if (!(m >> 31)) continue;
      const int lp = (int)(m & 0xfffu), slot = (int)((m >> 12) & 0x3fu);
      const double2 ob = puv_s[pos];
      const double X[3] = {xs[xoff + 3 * lp], xs[xoff + 3 * lp + 1], xs[xoff + 3 * lp + 2]};
      double s[3] = {1.0, 1.0, 1.0};
      if (!UNIT) { s[0] = ss[xoff + 3 * lp]; s[1] = ss[xoff + 3 * lp + 1]; s[2] = ss[xoff + 3 * lp + 2]; }
      // the table fields are read from the staged planes where they are used (the accumulators of phase B stay in
      // registers across this phase: a 32-double table in registers would push them out)
      auto tf = [&](int f) { return fa_table_field(tabs, P.tcs, f, slot); };
      double r[2], je[6], jf[12];
      {
        const double q0 = tf(0) * X[0] + tf(1) * X[1] + tf(2) * X[2];
        const double q1 = tf(3) * X[0] + tf(4) * X[1] + tf(5) * X[2];
        const double q2 = tf(6) * X[0] + tf(7) * X[1] + tf(8) * X[2];
        const double p0 = q0 + tf(18), p1 = q1 + tf(19), p2 = q2 + tf(20);
        const double fx = tf(21), fy = tf(22);
        const double iz = 1.0 / p2;   // the one division of the observation: p / p2 as p * (1 / p2) differs from Ceres' quotient by an ulp
        r[0] = fx * p0 * iz + tf(23) - ob.x;
        r[1] = fy * p1 * iz + tf(24) - ob.y;
        const double a = fx * iz, bb = -fx * p0 * iz * iz, cc = fy * iz, dd = -fy * p1 * iz * iz;
        const bool small = tf(25) != 0.0;
        const double b0 = small ? X[0] : q0, b1 = small ? X[1] : q1, b2 = small ? X[2] : q2;
#pragma unroll
        for (int k = 0; k < 3; ++k) {   // D[:,k] = A[:,k] x b
          const double a0 = tf(9 + k), a1 = tf(12 + k), a2 = tf(15 + k);
          const double d0 = a1 * b2 - a2 * b1, d1 = a2 * b0 - a0 * b2, d2 = a0 * b1 - a1 * b0;
          const double sk = tf(26 + k);
          jf[k] = (a * d0 + bb * d2) * sk;
          jf[6 + k] = (cc * d1 + dd * d2) * sk;
        }
        jf[3] = a * tf(29); jf[4] = 0.0;         jf[5] = bb * tf(31);
        jf[9] = 0.0;        jf[10] = cc * tf(30); jf[11] = dd * tf(31);
        je[0] = (a * tf(0) + bb * tf(6)) * s[0]; je[1] = (a * tf(1) + bb * tf(7)) * s[1]; je[2] = (a * tf(2) + bb * tf(8)) * s[2];
        je[3] = (cc * tf(3) + dd * tf(6)) * s[0]; je[4] = (cc * tf(4) + dd * tf(7)) * s[1]; je[5] = (cc * tf(5) + dd * tf(8)) * s[2];
      }
      sq += fa_apply_loss(P.loss, r, je, jf);
#pragma unroll
      for (int k = 0; k < 3; ++k) R2[k] = make_double2(je[2 * k], je[2 * k + 1]);
#pragma unroll
      for (int k = 0; k < 6; ++k) R2[3 + k] = make_double2(jf[2 * k], jf[2 * k + 1]);
      R2[9] = make_double2(r[0], r[1]);
    }
    __syncthreads();
    tick(2);
    // ---- A2: four lanes per point.  E^T E, E^T r (fixed butterfly over the four lanes), LM diagonal, 3x3 Cholesky and
    // z in every lane of the group; then every lane takes its observations of the point again: U = L^-1 J_e^T (rows),
    // w = U^T z.  L | z leave for pass 2 straight from the registers. ----
    for (int base = 0; base < ((P.dbg & 4) ? 0 : npts); base += SA_NT / 4) {
      const int lp = base + (tid >> 2), q = tid & 3;
      const bool on = lp < npts;
      int l0 = 0, l1 = 0;
      if (on) { l0 = pbeg[lp]; l1 = pbeg[lp + 1]; }
      double M[6] = {0, 0, 0, 0, 0, 0}, g[3] = {0, 0, 0};
      for (int l = l0 + q; l < l1; l += 4) {
        const double* R = rec + (size_t)pidx_s[l] * SA_REC;
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) {
          const double j0 = R[3 * rr], j1 = R[3 * rr + 1], j2 = R[3 * rr + 2], rv = R[18 + rr];
          M[0] += j0 * j0; M[1] += j0 * j1; M[2] += j0 * j2; M[3] += j1 * j1; M[4] += j1 * j2; M[5] += j2 * j2;
          g[0] += j0 * rv; g[1] += j1 * rv; g[2] += j2 * rv;
        }
      }
#pragma unroll
      for (int k = 0; k < 6; ++k) { M[k] += __shfl_xor_sync(0xffffffffu, M[k], 1); M[k] += __shfl_xor_sync(0xffffffffu, M[k], 2); }
#pragma unroll
      for (int k = 0; k < 3; ++k) { g[k] += __shfl_xor_sync(0xffffffffu, g[k], 1); g[k] += __shfl_xor_sync(0xffffffffu, g[k], 2); }
      if (!on) continue;
      const int64_t e = T.pt0 + lp;
      double sc[3] = {1.0, 1.0, 1.0}, isc[3] = {1.0, 1.0, 1.0};   // Jacobi scaling of the point and its reciprocal
      if (FIRST) {  // Jacobi scaling of this point from the unscaled column norms; E^T E, E^T r in scaled columns
        isc[0] = 1.0 + sqrt(M[0]); isc[1] = 1.0 + sqrt(M[3]); isc[2] = 1.0 + sqrt(M[5]);
        sc[0] = 1.0 / isc[0]; sc[1] = 1.0 / isc[1]; sc[2] = 1.0 / isc[2];
        M[0] *= sc[0] * sc[0]; M[1] *= sc[0] * sc[1]; M[2] *= sc[0] * sc[2]; M[3] *= sc[1] * sc[1]; M[4] *= sc[1] * sc[2]; M[5] *= sc[2] * sc[2];
        g[0] *= sc[0]; g[1] *= sc[1]; g[2] *= sc[2];
        if (q == 0) { P.se_out[3 * e] = sc[0]; P.se_out[3 * e + 1] = sc[1]; P.se_out[3 * e + 2] = sc[2]; }
      } else {
        sc[0] = ss[xoff + 3 * lp]; sc[1] = ss[xoff + 3 * lp + 1]; sc[2] = ss[xoff + 3 * lp + 2];
        if (q == 0) { isc[0] = 1.0 / sc[0]; isc[1] = 1.0 / sc[1]; isc[2] = 1.0 / sc[2]; }
      }
      if (q == 0 && l1 > l0) {  // |x - Plus(x, -g)| of the unscaled gradient (TrustRegionMinimizer::EvaluateGradientAndJacobian)
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          const double xv = xs[xoff + 3 * lp + k];
          const double d = xv - (xv + (-(g[k] * isc[k])));
          gmx = fmax(gmx, fabs(d)); g2 += d * d;
        }
      }
      if (!FULL) continue;
      // LM diagonal D^2 = clamp(diag) / radius (Ceres squares sqrt(clamp(diag) / radius): the same to an ulp, without
      // three square roots and three divisions in the most serial part of the tile)
      M[0] += fmin(fmax(M[0], P.min_diag), P.max_diag) * inv_radius;
      M[3] += fmin(fmax(M[3], P.min_diag), P.max_diag) * inv_radius;
      M[5] += fmin(fmax(M[5], P.min_diag), P.max_diag) * inv_radius;
      double Lp[6];
      if (!fa_chol3(M, Lp)) {
        if (q == 0) atomicOr(P.status, 1);
        Lp[0] = Lp[1] = Lp[2] = 0.0; Lp[3] = Lp[4] = Lp[5] = 1.0;
      }
      fa_fwd3(Lp, g);  // z
      {  // L | z of the point -> HBM (9 doubles, dealt over the four lanes)
        double* out = P.Lz + 9 * e;
#pragma unroll
        for (int k = 0; k < 9; ++k)
          if ((k & 3) == q) out[k] = k < 6 ? Lp[k] : g[k - 6];
      }
      for (int l = l0 + q; l < l1; l += 4) {
        double* R = rec + (size_t)pidx_s[l] * SA_REC;
        double w2[2];
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) {
          double u[3] = {R[3 * rr] * (FIRST ? sc[0] : 1.0), R[3 * rr + 1] * (FIRST ? sc[1] : 1.0), R[3 * rr + 2] * (FIRST ? sc[2] : 1.0)};
          fa_fwd3(Lp, u);
          R[3 * rr] = u[0]; R[3 * rr + 1] = u[1]; R[3 * rr + 2] = u[2];
          w2[rr] = u[0] * g[0] + u[1] * g[1] + u[2] * g[2];
        }
        R[20] = w2[0]; R[21] = w2[1];
      }
    }
    tick(3);
    sa_mbar_wait(bars + 1, ph2); ph2 ^= 1u;
    __syncthreads();
    tick(4);
    if (producer && ti + 1 < S.ntiles) issue_g1(Tn);   // group 1 is free: the next tile's inputs travel during B
    // ---- B: every thread works through the entries of ITS destination / camera in this tile ----
    const int nstaged = min(T.nent, P.ent_cap);
    if ((ttype == SA_TYPE_PAIR || ttype == SA_TYPE_FLUSH) && !(P.dbg & 1)) {
      if (FULL) {
        const int nrounds = ttype == SA_TYPE_PAIR ? 1 : (S.nflush + 31) >> 5;
        int64_t fbase = P.n_pout + T.fout0;
        for (int c = 0; c < nrounds; ++c) {
          const int v = ttype == SA_TYPE_PAIR ? tid : SA_NT + 32 * c + orank;
          int q = 0, q1 = 0;
          if (ttype == SA_TYPE_PAIR || 32 * c + orank < S.nflush) { q = seg_s[v]; q1 = seg_s[v + 1]; }
          unsigned fm = 0;
          if (ttype == SA_TYPE_FLUSH) {   // warp-uniform branch: the whole warp is the flush warp
            fm = __ballot_sync(0xffffffffu, q1 > q);
#pragma unroll
            for (int k = 0; k < 36; ++k) acc[k] = 0.0;
          }
          for (; q < q1; ++q) {
            const int32_t cur = q < nstaged ? ent_s[q] : __ldg(P.ent + T.ent0 + q);
            const double2* Ri = reinterpret_cast<const double2*>(rec + (size_t)(cur & 0xfff) * SA_REC);
            const double2* Rj = reinterpret_cast<const double2*>(rec + (size_t)((cur >> 12) & 0xfff) * SA_REC);
            double ui[6], uj[6];
#pragma unroll
            for (int k = 0; k < 3; ++k) { const double2 a = Ri[k], b = Rj[k]; ui[2 * k] = a.x; ui[2 * k + 1] = a.y; uj[2 * k] = b.x; uj[2 * k + 1] = b.y; }
            const double g00 = ui[0] * uj[0] + ui[1] * uj[1] + ui[2] * uj[2], g01 = ui[0] * uj[3] + ui[1] * uj[4] + ui[2] * uj[5];
            const double g10 = ui[3] * uj[0] + ui[4] * uj[1] + ui[5] * uj[2], g11 = ui[3] * uj[3] + ui[4] * uj[4] + ui[5] * uj[5];
            double fj[12];
#pragma unroll
            for (int k = 0; k < 6; ++k) { const double2 b = Rj[3 + k]; fj[2 * k] = b.x; fj[2 * k + 1] = b.y; }
            // J_f = [* * * a 0 b ; * * * 0 c d]: entries 4 and 9 are structural zeros
            double t0[6], t1[6];
#pragma unroll
            for (int b = 0; b < 6; ++b) {
              if (b == 3) { t0[b] = g00 * fj[3]; t1[b] = g10 * fj[3]; }
              else if (b == 4) { t0[b] = g01 * fj[10]; t1[b] = g11 * fj[10]; }
              else { t0[b] = g00 * fj[b] + g01 * fj[6 + b]; t1[b] = g10 * fj[b] + g11 * fj[6 + b]; }
            }
#pragma unroll
            for (int k = 0; k < 3; ++k) {
              const double2 f0 = Ri[3 + k], f1 = Ri[6 + k];   // J_f,i rows 0 / 1, columns 2k, 2k+1
#pragma unroll
              for (int b = 0; b < 6; ++b) {
                // one FMA per product, straight into the accumulator (a sum of two products added afterwards costs a
                // DMUL + DFMA + DADD where two DFMAs do)
                if (k == 1) {        // column 3: row 1 is zero
                  acc[(2 * k) * 6 + b] = fma(f0.x, t0[b], fma(f1.x, t1[b], acc[(2 * k) * 6 + b]));
                  acc[(2 * k + 1) * 6 + b] = fma(f0.y, t0[b], acc[(2 * k + 1) * 6 + b]);
                } else if (k == 2) { // column 4: row 0 is zero
                  acc[(2 * k) * 6 + b] = fma(f1.x, t1[b], acc[(2 * k) * 6 + b]);
                  acc[(2 * k + 1) * 6 + b] = fma(f0.y, t0[b], fma(f1.y, t1[b], acc[(2 * k + 1) * 6 + b]));
                } else {
                  acc[(2 * k) * 6 + b] = fma(f0.x, t0[b], fma(f1.x, t1[b], acc[(2 * k) * 6 + b]));
                  acc[(2 * k + 1) * 6 + b] = fma(f0.y, t0[b], fma(f1.y, t1[b], acc[(2 * k + 1) * 6 + b]));
                }
              }
            }
          }
          if (ttype == SA_TYPE_FLUSH) {
            if ((fm >> lane) & 1u) {
              double2* out = reinterpret_cast<double2*>(P.partP + (size_t)(fbase + __popc(fm & ((1u << lane) - 1u))) * 36);
#pragma unroll
              for (int k = 0; k < 18; ++k) out[k] = make_double2(acc[2 * k], acc[2 * k + 1]);
            }
            fbase += __popc(fm);
          }
        }
      }
    } else if (ttype == SA_TYPE_CAM && !(P.dbg & 2)) {
      int q = seg_s[tid];
      const int q1 = seg_s[tid + 1];
      for (; q < q1; ++q) {
        const int32_t cur = q < nstaged ? ent_s[q] : __ldg(P.ent + T.ent0 + q);
        const double2* R2 = reinterpret_cast<const double2*>(rec + (size_t)(cur & 0xfff) * SA_REC);
        double jf[12];
#pragma unroll
        for (int k = 0; k < 6; ++k) { const double2 v = R2[3 + k]; jf[2 * k] = v.x; jf[2 * k + 1] = v.y; }
        const double2 rv = R2[9];
#pragma unroll
        for (int a = 0; a < 6; ++a) acc[21 + a] = fma(jf[a], rv.x, fma(jf[6 + a], rv.y, acc[21 + a]));
        if (FULL) {
          const double2 wv = R2[10];
          const double2 ua = R2[0], ub = R2[1], uc = R2[2];   // u_0 = (ua.x ua.y ub.x), u_1 = (ub.y uc.x uc.y)
          const double h00 = 1.0 - (ua.x * ua.x + ua.y * ua.y + ub.x * ub.x);
          const double h01 = -(ua.x * ub.y + ua.y * uc.x + ub.x * uc.y);
          const double h11 = 1.0 - (ub.y * ub.y + uc.x * uc.x + uc.y * uc.y);
          double t0[6], t1[6];
#pragma unroll
          for (int b = 0; b < 6; ++b) { t0[b] = h00 * jf[b] + h01 * jf[6 + b]; t1[b] = h01 * jf[b] + h11 * jf[6 + b]; }
          int c = 0;
#pragma unroll
          for (int a = 0; a < 6; ++a)
#pragma unroll
            for (int b = a; b < 6; ++b) { acc[c] = fma(jf[a], t0[b], fma(jf[6 + a], t1[b], acc[c])); ++c; }
#pragma unroll
          for (int a = 0; a < 6; ++a) {
            acc[27 + a] = fma(jf[a], wv.x, fma(jf[6 + a], wv.y, acc[27 + a]));
            acc[33 + a] = fma(jf[a], jf[a], fma(jf[6 + a], jf[6 + a], acc[33 + a]));
          }
        }
      }
    }
    tick(5);
    __syncthreads();
    tick(6);
    if (producer && ti + 1 < S.ntiles) issue_g2(Tn, tile + 1);
  }
  if (P.clocks && tid == 0)
    for (int k = 0; k < 7; ++k) atomicAdd(P.clocks + k, (unsigned long long)ck[k]);
  // ---- the strip's partial blocks ----
  if (ttype == SA_TYPE_PAIR && FULL) {
    double2* out = reinterpret_cast<double2*>(P.partP + (size_t)(S.pout0 + orank) * 36);
#pragma unroll
    for (int k = 0; k < 18; ++k) out[k] = make_double2(acc[2 * k], acc[2 * k + 1]);
  } else if (ttype == SA_TYPE_CAM) {
    double* out = P.partC + (size_t)(S.cout0 + orank) * SA_NVC;
#pragma unroll
    for (int k = 0; k < SA_NVC; ++k) out[k] = acc[k];
  }
  {
    double v[3] = {sq, g2, gmx};
    const bool mx[3] = {false, false, true};
    fa_block_reduce(v, mx, 3, red);
    if (tid == 0) { P.cost_partial[blockIdx.x] = v[0]; P.g2_partial[blockIdx.x] = v[1]; P.gmax_partial[blockIdx.x] = v[2]; }
  }
}

}  // namespace ba
