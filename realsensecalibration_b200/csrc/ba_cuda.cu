// ba_cuda.cu -- the ba_cuda_* C ABI (include/ba_cuda.h) and the Levenberg-Marquardt driver.
//
// The driver restates Ceres 1.14's TrustRegionMinimizer + LevenbergMarquardtStrategy (the code
// behind ceres::Solve at Main_Calibration/bundle_adjustment_manager.cpp:94,
// Test1_BundleAdjustment/main.cpp:86, Test2_BundleAdjustment/main.cpp:103; spec in SURVEY.md 5.9)
// with every numeric step running as CUDA kernels on one B200; the host only reads back a
// handful of scalars per iteration to take the accept / reject / terminate decision.
// There is no CPU fallback: without a CUDA device ba_cuda_create() fails.
#include <dlfcn.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstddef>
#include <string>

#include "ba_dense.cuh"
#include "ba_dense_blocked.cuh"
#include "ba_kernels.cuh"
#include "ba_structure.cuh"
#include "ba_rcs.cuh"
#include "ba_fused_a.cuh"
#include "ba_strip_a.cuh"
#include "ba_exchange.cuh"
#include "ba_rig.cuh"
#include "ba_cov.cuh"

using namespace ba;

// ---- minimal NCCL surface, bound at run time (the process usually has torch's libnccl loaded) ----
namespace {
typedef struct ncclComm* ncclComm_t;
struct NcclUniqueId { char internal[128]; };
struct Nccl {
  void* handle = nullptr;
  int (*GetUniqueId)(NcclUniqueId*) = nullptr;
  int (*CommInitRank)(ncclComm_t*, int, NcclUniqueId, int) = nullptr;
  int (*CommDestroy)(ncclComm_t) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  bool ok() const { return handle != nullptr; }
};
constexpr int kNcclFloat64 = 8, kNcclInt32 = 2, kNcclInt64 = 4, kNcclUint64 = 5, kNcclSum = 0, kNcclMax = 2;
Nccl& nccl() {
  static Nccl n;
  static bool tried = false;
  if (!tried) {
    tried = true;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* nm : names) {
      n.handle = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
      if (n.handle) break;
    }
    if (n.handle) {
      n.GetUniqueId = (int (*)(NcclUniqueId*))dlsym(n.handle, "ncclGetUniqueId");
      n.CommInitRank = (int (*)(ncclComm_t*, int, NcclUniqueId, int))dlsym(n.handle, "ncclCommInitRank");
      n.CommDestroy = (int (*)(ncclComm_t))dlsym(n.handle, "ncclCommDestroy");
      n.AllReduce = (int (*)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t))dlsym(n.handle, "ncclAllReduce");
      n.GetErrorString = (const char* (*)(int))dlsym(n.handle, "ncclGetErrorString");
      n.AllGather = (int (*)(const void*, void*, size_t, int, ncclComm_t, cudaStream_t))dlsym(n.handle, "ncclAllGather");
      if (!n.GetUniqueId || !n.CommInitRank || !n.CommDestroy || !n.AllReduce) n.handle = nullptr;
    }
  }
  return n;
}
double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

// S_CAND .. S_STATUSD are contiguous: the shard-local values one ncclAllReduce sums after a step
enum Scal { S_COST = 0, S_G2E, S_GMAXE, S_CAND, S_MCC, S_XE2, S_DE2, S_STATUSD, S_XF2, S_DF2, S_GMAXF, S_G2F, S_RADIUS, S_COUNT = 16 };
constexpr int kMaxWorld = 64;  // ranks whose gradient maxima ride in the tail of one sum-allreduce
enum Family { F_JAC = 0, F_SCHUR, F_SOLVE, F_UPDATE, F_COST, F_COLL, F_COUNT };
// one entry per kernel (family member) of the solve path; names are what ba_cuda_get_kernel_stats() reports
enum KT {
  KT_TABLES = 0, KT_JAC, KT_COST, KT_FOBS, KT_EM, KT_INCW, KT_DOBS, KT_ECHOL, KT_INCY, KT_FINC, KT_PAIRS, KT_SEGFIN,
  KT_ASSEMBLE, KT_RCS, KT_BACKSUB, KT_MODELCOST, KT_CANDIDATE, KT_GRADNORM, KT_FOLD, KT_MISC, KT_FA_P1, KT_FA_RED, KT_FA_P2, KT_FA_P1L, KT_RIG,
  KT_COV_LINV, KT_COV_INV, KT_COV_FRAMES, KT_RIG_BATCH, KT_COUNT
};
const char* const kKtName[KT_COUNT] = {
  "k1_tables", "k1_residual_jacobian", "k5_cost", "k2_fobs_partial", "k2_e_normal", "k2_inc_w", "k2_dobs_partial",
  "k2_e_cholesky", "k2_inc_y", "k2_finc_partial", "k2_pairs_partial", "k2_seg_final", "k2_assemble", "k3_rcs_solve",
  "k4_backsub", "k4_model_cost", "k4_candidate", "k4_gradient_norm", "fold_partials", "misc",
  "k1k2_fused_pass1", "k2_reduce_items", "k4k5_fused_pass2", "k1_fused_pass1_light", "rig_lm_whole_loop",
  "cov_l_inverse", "cov_inverse_kept", "cov_frames", "rig_lm_batch"};
}  // namespace

struct LmState {  // TrustRegionMinimizer's loop variables, kept between ba_cuda_solve_iterate() calls
  ba_cuda_options opt;
  ba_cuda_summary Z;
  double radius = 0.0, decrease_factor = 2.0, x_cost = 0.0, gmax = 0.0, gnorm = 0.0, t_start = 0.0;
  int num_invalid = 0;
  bool began = false, go = false;
  bool need_linearize = false;  // fused Model A path: the Schur system must be re-formed (new radius after a rejection)
  bool rig = false;             // the whole loop runs in k_rig_lm (ba_rig.cuh)
  bool rig_begin_pending = false;   // ba_cuda_solve: iteration zero rides in the first (only) launch
};

struct ba_cuda_problem {
  int device = 0;
  cudaStream_t st = nullptr, own_st = nullptr;
  cudaStream_t copy_st = nullptr;             // H2D of the observations runs here, beside the structure build
  cudaEvent_t copy_go = nullptr, copy_done = nullptr;
  int model = -1;  // 0 = A, 1 = B
  int32_t n_cam = 0, n_time = 0, n_marker = 0;
  int64_t n_pt = 0, n_params = 0;
  double half_side = 0.0;
  Structure S;
  std::vector<int32_t> h_perm;
  // model data in sorted observation order
  DVec<double2> uv;
  DVec<double> obs8, intr_f;
  DVec<int32_t> ob_cam, ob_marker;
  // parameters (x), candidate (xc), Jacobi scaling, block tables
  DVec<double> xf, xe, xf_c, xe_c, xf_s, xe_s, sf, se, tab_f, tab_e, tabc_f, tabc_e;  // _s: saved snapshot
  // Jacobian and Schur workspace
  DVec<double> RES, JE, JF0, JF1, ME, HG, Wt, Lb, zb, Yt, vb, Pacc, Qacc, Sd, rhs, yf, ye;
  DVec<double> part_fobs, part_finc, part_pairs, part_dobs, bp0, bp1, scal;
  DVec<int> status;
  DVec<int64_t> f_act_ptr;   // exclusive scan of the kept blocks' GLOBAL activity: active iff ptr[f + 1] > ptr[f]
  int64_t n_active_e_global = 0, n_active_f_global = 0, nb_global = 0;
  // reduced camera system: block-sparse pattern (shared by all ranks), values, PCG workspace
  RcsPattern R;
  PcgWork pcg;
  CholBlockedWork cholb;
  DVec<double> Sb;           // R.nd * 36 block values | nf * 6 rhs correction (one collective covers both)
  int solver = 0;            // ba_rcs_solver resolved for the current solve
  FusedA FA;                 // Model A: tile structure of the fused two-pass pipeline
  StripA SA;                 // Model A: strip structure of pass 1 (ba_strip_a.cuh); FA then only carries the tiles of pass 2 / k_fa_jac
  bool use_fused = false, use_strip = false, generic_ws = false;
  bool smem_attr_set = false;   // the opt-in shared-memory sizes are per device: set once per problem
  bool rig_attr_set = false;
  bool one_shot = false;        // inside ba_cuda_solve: nobody looks at row 0 before the loop runs
  bool building = false;        // inside ba_cuda_set_model_*: a failure from here on leaves no half-built model behind
  DVec<unsigned char> rig_buf;  // RigState | rows of one launch
  unsigned char* h_rig = nullptr;   // pinned mirror
  SparseExchange SX;            // multi-GPU, fused Model A + PCG: all-gather of the ranks' own blocks instead of an all-reduce of all
  LossSpec loss{0, 1.0};        // robust loss of the current solve (options.loss_function / loss_scale); 0 outside a solve
  DVec<double> fa_part;      // 7 per-tile partial arrays (cost, g2, gmax, mcc, x2, d2, cand)
  int h_pcg_iters = 0;
  double* h_scal = nullptr;  // pinned
  int* h_status = nullptr;   // pinned
  bool params_set = false;
  std::vector<ba_cuda_iteration> rows;
  LmState lm;
  // multi-GPU
  ncclComm_t comm = nullptr;
  int rank = 0, world = 1;
  // timing
  cudaEvent_t ev[F_COUNT][2] = {};
  double fam_ms[F_COUNT] = {};
  bool fam_open[F_COUNT] = {};
  cudaEvent_t k0 = nullptr, k1 = nullptr;
  float last_kernel_ms = 0.f;
  // per-kernel accounting
  bool profile = false;
  int64_t kt_launches[KT_COUNT] = {};
  double kt_ms[KT_COUNT] = {};
  std::vector<cudaEvent_t> ev_pool;
  size_t ev_next = 0;
  struct Pending { int kt; size_t e0, e1; };
  std::vector<Pending> pending;
  int64_t n_rcs() const { return 6 * S.nf; }
  // rhs correction (sum of v_i per camera) lives at the tail of the RCS value buffer: one collective covers both
  double* vsum() { return solver == BA_RCS_PCG ? Sb.p + (int64_t)R.nd * 36 : Sd.p + n_rcs() * n_rcs(); }
};

namespace {

int use_device(ba_cuda_problem* p) {
  BA_CUDA_TRY(cudaSetDevice(p->device));
  DevCache::current_stream() = p->st;  // device buffers freed from here on are reused in this stream's order
  return BA_OK;
}
std::atomic<int> g_live_problems{0};
struct PhaseTimer {  // BA_CUDA_TIMING=1: host wall clock of the phases of ba_cuda_set_model_* on stderr
  const bool on = std::getenv("BA_CUDA_TIMING") != nullptr;
  double t = now_s();
  void lap(const char* what) {
    if (!on) return;
    const double n = now_s();
    std::fprintf(stderr, "[ba_cuda timing] %-28s %9.3f ms\n", what, 1e3 * (n - t));
    t = n;
  }
};

// ---- per-kernel accounting -------------------------------------------------------------
cudaEvent_t pool_event(ba_cuda_problem* p, size_t* idx) {
  if (p->ev_next == p->ev_pool.size()) {
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    p->ev_pool.push_back(e);
  }
  *idx = p->ev_next++;
  return p->ev_pool[*idx];
}
struct LaunchScope {  // counts the launch; with profiling on, brackets it with two pooled events
  ba_cuda_problem* p; int kt; size_t e0 = 0, e1 = 0;
  LaunchScope(ba_cuda_problem* p_, int kt_) : p(p_), kt(kt_) {
    ++p->kt_launches[kt];
    if (p->profile) cudaEventRecord(pool_event(p, &e0), p->st);
  }
  ~LaunchScope() {
    if (p->profile) { cudaEventRecord(pool_event(p, &e1), p->st); p->pending.push_back({kt, e0, e1}); }
  }
};
// BA_LAUNCH(p, KT_X, (kernel<T...>), grid, block, smem, args...)
#define BA_LAUNCH(p, kt, kern, grid, block, smem, ...)            \
  do {                                                            \
    LaunchScope scope__((p), (kt));                               \
    kern<<<(grid), (block), (smem), (p)->st>>>(__VA_ARGS__);      \
  } while (0)

void kt_collect(ba_cuda_problem* p) {  // call after a stream synchronize
  for (const auto& q : p->pending) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, p->ev_pool[q.e0], p->ev_pool[q.e1]) == cudaSuccess) p->kt_ms[q.kt] += ms;
  }
  p->pending.clear();
  p->ev_next = 0;
}

// ---- family timers: one event pair per family, accumulated at the iteration's host sync ----
void fam_begin(ba_cuda_problem* p, int f) { cudaEventRecord(p->ev[f][0], p->st); p->fam_open[f] = true; }
void fam_end(ba_cuda_problem* p, int f) { cudaEventRecord(p->ev[f][1], p->st); }
void fam_collect(ba_cuda_problem* p) {  // call after a stream synchronize
  for (int f = 0; f < F_COUNT; ++f)
    if (p->fam_open[f]) {
      float ms = 0.f;
      if (cudaEventElapsedTime(&ms, p->ev[f][0], p->ev[f][1]) == cudaSuccess) p->fam_ms[f] += ms;
      p->fam_open[f] = false;
    }
  kt_collect(p);
}

int fold(ba_cuda_problem* p, const double* partial, int n, int slot, bool is_max = false) {
  BA_LAUNCH(p, KT_FOLD, k_fold_partials, 1, 1024, 0, partial, n, p->scal.p, slot, is_max ? 1 : 0);
  BA_CUDA_TRY(cudaGetLastError());
  return BA_OK;
}

int allreduce(ba_cuda_problem* p, void* buf, size_t count, int op, int dtype = kNcclFloat64) {
  if (p->world <= 1) return BA_OK;
  const int rc = nccl().AllReduce(buf, buf, count, dtype, op, p->comm, p->st);
  if (rc != 0) return fail(BA_ERR_NCCL, "ncclAllReduce failed: %s", nccl().GetErrorString ? nccl().GetErrorString(rc) : "?");
  return BA_OK;
}

// Shard-local scalars ride on collectives that are needed anyway (every separate ncclAllReduce costs ~25 us of latency):
// tail = [cost, |g_e|^2, gmax_e of rank 0 .. world-1]; a SUM all-reduce then carries the maximum too.
__global__ void k_pack_grad_tail(const double* __restrict__ scal, int rank, int world, double* __restrict__ tail) {
  const int i = threadIdx.x;
  if (i == 0) tail[0] = scal[S_COST];
  if (i == 1) tail[1] = scal[S_G2E];
  if (i < world) tail[2 + i] = i == rank ? scal[S_GMAXE] : 0.0;
}
__global__ void k_unpack_grad_tail(const double* __restrict__ tail, int world, double* __restrict__ scal) {
  if (threadIdx.x != 0) return;
  scal[S_COST] = tail[0];
  scal[S_G2E] = tail[1];
  double m = 0.0;
  for (int r = 0; r < world; ++r) m = fmax(m, tail[2 + r]);
  scal[S_GMAXE] = m;
}
__global__ void k_status_to_scal(const int* __restrict__ status, double* __restrict__ scal) { scal[S_STATUSD] = *status != 0 ? 1.0 : 0.0; }

// after a step: candidate cost, model cost change, |x_e|^2, |delta_e|^2 and the "a block factorisation failed" flag of
// all shards in one collective
int allreduce_step_scalars(ba_cuda_problem* p) {
  if (p->world <= 1) return BA_OK;
  k_status_to_scal<<<1, 1, 0, p->st>>>(p->status.p, p->scal.p);
  return allreduce(p, p->scal.p + S_CAND, S_STATUSD - S_CAND + 1, kNcclSum);
}
// after a linearisation: cost, |g_e|^2 (sums) and max |g_e| through `tail` (2 + world doubles at the end of `buf`)
int allreduce_with_grad_tail(ba_cuda_problem* p, double* buf, size_t n) {
  if (p->world <= 1) return BA_OK;
  k_pack_grad_tail<<<1, kMaxWorld, 0, p->st>>>(p->scal.p, p->rank, p->world, buf + n);
  BA_TRY(allreduce(p, buf, n + 2 + p->world, kNcclSum));
  k_unpack_grad_tail<<<1, 32, 0, p->st>>>(buf + n, p->world, p->scal.p);
  BA_CUDA_TRY(cudaGetLastError());
  return BA_OK;
}

// dense RCS solve: whole matrix in one CTA's shared memory while it fits, blocked DMMA Cholesky over the GPU above
int dense_solve(ba_cuda_problem* p, int64_t n) {
  // measured on B200: n = 132 (cfg2) 0.18 ms blocked vs 0.24 ms single CTA; below ~96 the single CTA wins (one launch, no grid barrier)
  static const int smem_max_n = env_int("BA_DENSE_SMEM_MAX_N", 0, CHOL_SMEM_MAX_N, 96);
  static const bool ldlt = env_int("BA_DENSE_LDLT", 0, 1, 1) != 0;
  if (ldlt && n <= RIG_MAX_N) {   // the panel LDL^T of the rig kernel, one CTA, matrix in shared memory (ba_rig.cuh)
    const size_t smem = rig_smem_bytes((int)n);
    if (smem > 48 * 1024) BA_CUDA_TRY(cudaFuncSetAttribute(k_ldlt_small, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rig_smem_bytes(RIG_MAX_N)));
    k_ldlt_small<<<1, RIG_THREADS, smem, p->st>>>((int)n, p->Sd.p, p->rhs.p, p->yf.p, p->status.p);
    BA_CUDA_TRY(cudaGetLastError());
    return BA_OK;
  }
  if (n <= smem_max_n) return launch_chol_solve((int)n, p->Sd.p, p->rhs.p, p->yf.p, p->status.p, p->st);
  return launch_chol_blocked(p->cholb, (int)n, p->Sd.p, p->rhs.p, p->yf.p, p->status.p, p->device, p->st);
}

// Multi-GPU: every rank only knows the destination blocks its own shard couples; the stored pattern has to be
// the union, identical on all ranks, so that one ncclAllReduce sums the block values in place.
int build_global_pattern(ba_cuda_problem* p) {
  const Structure& S = p->S;
  if (!nccl().AllGather) return fail(BA_ERR_NCCL, "ncclAllGather is not available");
  // 1. counts
  DVec<int64_t> cnt;
  BA_TRY(cnt.alloc(p->world));
  const int64_t mine = S.ndest;
  BA_CUDA_TRY(cudaMemcpyAsync(cnt.p + p->rank, &mine, sizeof(int64_t), cudaMemcpyHostToDevice, p->st));
  int rc = nccl().AllGather(cnt.p + p->rank, cnt.p, 1, kNcclInt64, p->comm, p->st);
  if (rc != 0) return fail(BA_ERR_NCCL, "ncclAllGather failed (%d)", rc);
  std::vector<int64_t> h(p->world);
  BA_CUDA_TRY(cudaMemcpyAsync(h.data(), cnt.p, sizeof(int64_t) * p->world, cudaMemcpyDeviceToHost, p->st));
  BA_CUDA_TRY(cudaStreamSynchronize(p->st));
  int64_t mx = 0;
  for (int64_t v : h) mx = std::max(mx, v);
  if (mx * p->world >= (int64_t)INT32_MAX) return fail(BA_ERR_UNSUPPORTED, "reduced camera system pattern too large");
  // 2. keys, padded with ~0 to the largest count
  DVec<uint64_t> all, sorted, uniq;
  DVec<int> nuniq;
  BA_TRY(all.alloc((size_t)mx * p->world)); BA_TRY(sorted.alloc((size_t)mx * p->world)); BA_TRY(uniq.alloc((size_t)mx * p->world));
  BA_TRY(nuniq.alloc(1));
  uint64_t* my = all.p + (size_t)mx * p->rank;
  BA_CUDA_TRY(cudaMemsetAsync(my, 0xff, sizeof(uint64_t) * mx, p->st));
  BA_CUDA_TRY(cudaMemcpyAsync(my, S.dest_keys.p, sizeof(uint64_t) * S.ndest, cudaMemcpyDeviceToDevice, p->st));
  rc = nccl().AllGather(my, all.p, (size_t)mx, kNcclUint64, p->comm, p->st);
  if (rc != 0) return fail(BA_ERR_NCCL, "ncclAllGather failed (%d)", rc);
  const int total = (int)(mx * p->world);
  BA_TRY(cub_call([&](void* t, size_t& b) { return cub::DeviceRadixSort::SortKeys(t, b, all.p, sorted.p, total, 0, 64, p->st); }));
  BA_TRY(cub_call([&](void* t, size_t& b) { return cub::DeviceSelect::Unique(t, b, sorted.p, uniq.p, nuniq.p, total, p->st); }));
  int nu = 0;
  uint64_t last = 0;
  BA_CUDA_TRY(cudaMemcpyAsync(&nu, nuniq.p, sizeof(int), cudaMemcpyDeviceToHost, p->st));
  BA_CUDA_TRY(cudaStreamSynchronize(p->st));
  BA_CUDA_TRY(cudaMemcpyAsync(&last, uniq.p + (nu - 1), sizeof(uint64_t), cudaMemcpyDeviceToHost, p->st));
  BA_CUDA_TRY(cudaStreamSynchronize(p->st));
  if (last == ~0ull) --nu;
  return build_rcs_pattern(p->R, uniq.p, nu, S.nf, p->st);
}

int build_tables(ba_cuda_problem* p, bool candidate) {
  const Structure& S = p->S;
  const double* xf = candidate ? p->xf_c.p : p->xf.p;
  double* tf = candidate ? p->tabc_f.p : p->tab_f.p;
  BA_LAUNCH(p, KT_TABLES, k_tables, grid_for(S.nf, 128), 128, 0, xf, p->intr_f.p, p->sf.p, S.nf, tf);
  if (p->model == 1) {
    const double* xe = candidate ? p->xe_c.p : p->xe.p;
    double* te = candidate ? p->tabc_e.p : p->tab_e.p;
    BA_LAUNCH(p, KT_TABLES, k_tables, grid_for(S.ne, 128), 128, 0, xe, nullptr, p->se.p, S.ne, te);
  }
  BA_CUDA_TRY(cudaGetLastError());
  return BA_OK;
}

FaParams fa_params(ba_cuda_problem* p, const ba_cuda_options& opt);
int fa_set_smem_attr(ba_cuda_problem* p);
int sx_exchange(ba_cuda_problem* p, double* camacc, bool with_blocks);
bool sx_active(const ba_cuda_problem* p);

// K1 at the current parameters: residuals, scaled Jacobian, sum of squares -> scal[S_COST]
int run_jacobian(ba_cuda_problem* p) {
  const Structure& S = p->S;
  BA_TRY(build_tables(p, false));
  int grid;
  if (p->model == 0 && p->use_fused) {  // the tile structure exists: tables staged in shared memory, J leaves as full lines
    BA_TRY(fa_set_smem_attr(p));
    ba_cuda_options o;
    ba_cuda_options_init(&o);
    const FaParams P = fa_params(p, o);
    grid = p->FA.n_tiles;
    BA_LAUNCH(p, KT_JAC, k_fa_jac, grid, FA_JAC_THREADS, p->FA.smemj(FA_JAC_THREADS), P);
    BA_CUDA_TRY(cudaGetLastError());
    return fold(p, p->fa_part.p, grid, S_COST);
  }
  if (p->model == 0) {
    grid = (int)grid_for(S.nb, 256);
    BA_LAUNCH(p, KT_JAC, k_jac_a, grid, 256, 0, S.nb, S.ob_e.p, S.ob_f0.p, p->uv.p, p->tab_f.p, p->xe.p, p->se.p, p->RES.p,
              p->JE.p, p->JF0.p, p->bp0.p, p->loss);
  } else {
    grid = (int)grid_for(S.nb * 4, 128);
    BA_LAUNCH(p, KT_JAC, k_jac_b, grid, 128, 0, S.nb, S.ob_e.p, S.ob_f0.p, S.ob_f1.p, p->ob_cam.p, p->obs8.p, p->tab_f.p,
              p->tab_e.p, p->half_side, p->RES.p, p->JE.p, p->JF0.p, p->JF1.p, p->bp0.p, p->loss);
  }
  BA_CUDA_TRY(cudaGetLastError());
  return fold(p, p->bp0.p, grid, S_COST);
}

// cost-only evaluation at the candidate -> scal[S_CAND]
int run_cost_candidate(ba_cuda_problem* p) {
  const Structure& S = p->S;
  BA_TRY(build_tables(p, true));
  int grid;
  if (p->model == 0) {
    grid = (int)grid_for(S.nb, 256);
    BA_LAUNCH(p, KT_COST, k_cost_a, grid, 256, 0, S.nb, S.ob_e.p, S.ob_f0.p, p->uv.p, p->tabc_f.p, p->xe_c.p, p->bp0.p, p->loss);
  } else {
    grid = (int)grid_for(S.nb * 4, 128);
    BA_LAUNCH(p, KT_COST, k_cost_b, grid, 128, 0, S.nb, S.ob_e.p, S.ob_f0.p, S.ob_f1.p, p->ob_cam.p, p->obs8.p, p->tabc_f.p,
              p->tabc_e.p, p->half_side, p->bp0.p, p->loss);
  }
  BA_CUDA_TRY(cudaGetLastError());
  return fold(p, p->bp0.p, grid, S_CAND);
}

// Everything of the normal equations that depends only on J: F^T F / F^T r per f-block, E^T E / E^T r per
// e-block, Model B: W_i per incidence and the off-diagonal F^T F blocks.
template <int RD, int DE, int GE>
int run_normal_parts(ba_cuda_problem* p) {
  const Structure& S = p->S;
  if (S.ch_fobs.n > 0)
    BA_LAUNCH(p, KT_FOBS, (k_fobs_partial<RD>), grid_for(S.ch_fobs.n, 4), 128, 0, S.ch_fobs.n, S.ch_fobs.ch, S.ch_fobs.seg.p,
              S.ch_fobs.begin.p, S.fobs_ptr.p, S.fobs.p, p->RES.p, p->JF0.p, p->JF1.p, p->part_fobs.p);
  BA_LAUNCH(p, KT_SEGFIN, (k_seg_final<NV_F>), grid_for(S.nf, 4), 128, 0, (int)S.nf, S.ch_fobs.seg_first.p, p->part_fobs.p, p->HG.p);
  BA_LAUNCH(p, KT_EM, (k_e_M<RD, DE, GE>), grid_for(S.ne * GE, 128), 128, 0, S.ne, S.e_ptr.p, p->RES.p, p->JE.p, p->ME.p);
  if (p->model == 1) {
    BA_LAUNCH(p, KT_INCW, (k_inc_W<RD>), grid_for(S.ninc * RD, 128), 128, 0, S.ninc, S.incobs_ptr.p, S.incobs.p, p->JE.p, p->JF0.p,
              p->JF1.p, p->Wt.p);
    if (S.ch_dobs.n > 0)
      BA_LAUNCH(p, KT_DOBS, (k_dobs_partial<RD>), grid_for(S.ch_dobs.n, 4), 128, 0, S.ch_dobs.n, S.ch_dobs.ch, S.ch_dobs.seg.p,
                S.ch_dobs.begin.p, S.dobs_ptr.p, S.dobs.p, p->JF0.p, p->JF1.p, p->part_dobs.p);
    BA_LAUNCH(p, KT_SEGFIN, (k_seg_final<36>), grid_for(S.ndest, 4), 128, 0, S.ndest, S.ch_dobs.seg_first.p, p->part_dobs.p, p->Qacc.p);
  }
  BA_CUDA_TRY(cudaGetLastError());
  return BA_OK;
}

template <int DE>
int run_gradient_norms_e(ba_cuda_problem* p) {  // eliminated blocks: shard local
  const Structure& S = p->S;
  constexpr int NU = DE * (DE + 1) / 2;
  const int ge = (int)grid_for(S.ne * DE, 256);
  BA_LAUNCH(p, KT_GRADNORM, (k_gradient_norm<DE, NU + DE, NU>), ge, 256, 0, S.ne, S.e_ptr.p, p->xe.p, p->se.p, p->ME.p, p->bp0.p, p->bp1.p);
  {
    FoldJob J = {{p->bp0.p, p->bp1.p, nullptr, nullptr}, {S_GMAXE, S_G2E, 0, 0}, {1, 0, 0, 0}};
    BA_LAUNCH(p, KT_FOLD, k_fold_multi, 2, 1024, 0, J, ge, p->scal.p);
  }
  BA_CUDA_TRY(cudaGetLastError());
  return BA_OK;
}
int run_gradient_norms_f(ba_cuda_problem* p) {  // kept blocks: from the (globally summed) F^T r
  const Structure& S = p->S;
  const int gf = (int)grid_for(S.nf * 6, 256);
  BA_LAUNCH(p, KT_GRADNORM, (k_gradient_norm<6, NV_F, 21>), gf, 256, 0, S.nf, p->f_act_ptr.p, p->xf.p, p->sf.p, p->HG.p, p->bp0.p, p->bp1.p);
  {
    FoldJob J = {{p->bp0.p, p->bp1.p, nullptr, nullptr}, {S_GMAXF, S_G2F, 0, 0}, {1, 0, 0, 0}};
    BA_LAUNCH(p, KT_FOLD, k_fold_multi, 2, 1024, 0, J, gf, p->scal.p);
  }
  BA_CUDA_TRY(cudaGetLastError());
  return BA_OK;
}

// TrustRegionMinimizer::EvaluateGradientAndJacobian: r, J, cost, gradient norms at x; on the first call also
// the Jacobi scaling (computed once, from the unscaled J).
template <int RD, int DE, int GE>
int eval_gradient_and_jacobian(ba_cuda_problem* p, bool first, bool jacobi_scaling) {
  const Structure& S = p->S;
  fam_begin(p, F_JAC);
  if (first) {
    BA_LAUNCH(p, KT_MISC, k_fill, grid_for(S.ne * DE, 256), 256, 0, p->se.p, S.ne * DE, 1.0);
    BA_LAUNCH(p, KT_MISC, k_fill, grid_for(S.nf * 6, 256), 256, 0, p->sf.p, S.nf * 6, 1.0);
  }
  BA_TRY(run_jacobian(p));
  fam_end(p, F_JAC);
  fam_begin(p, F_SCHUR);
  BA_TRY((run_normal_parts<RD, DE, GE>(p)));
  if (first && jacobi_scaling) {
    BA_TRY(allreduce(p, p->HG.p, S.nf * NV_F, kNcclSum));  // column norms of the kept blocks are global sums
    constexpr int NU = DE * (DE + 1) / 2;
    BA_LAUNCH(p, KT_MISC, (k_jacobi_scale<DE, NU + DE>), grid_for(S.ne * DE, 256), 256, 0, S.ne, p->ME.p, p->se.p);
    BA_LAUNCH(p, KT_MISC, (k_jacobi_scale<6, NV_F>), grid_for(S.nf * 6, 256), 256, 0, S.nf, p->HG.p, p->sf.p);
    BA_TRY(run_jacobian(p));  // same residuals, Jacobian now column scaled
    BA_TRY((run_normal_parts<RD, DE, GE>(p)));
  }
  fam_end(p, F_SCHUR);
  BA_TRY(run_gradient_norms_e<DE>(p));
  if (p->world > 1) {  // F^T F | F^T r of the kept blocks and the shard-local gradient scalars in one collective
    fam_begin(p, F_COLL);
    BA_TRY(allreduce_with_grad_tail(p, p->HG.p, S.nf * NV_F));
    fam_end(p, F_COLL);
  }
  return run_gradient_norms_f(p);
}

// SchurEliminator for the LM diagonal of the radius in scal[S_RADIUS]: frame / point blocks factored (Lb, zb), Yt, and
// the reduced camera system with its rhs (Sd | rhs, or Sb | rhs for PCG).  Leaves the F_SOLVE family open: the caller's
// solve of the system belongs to it.  The covariance runs it with radius = +inf, i.e. without LM diagonal.
template <int RD, int DE>
int schur_complement(ba_cuda_problem* p, const ba_cuda_options& opt) {
  const Structure& S = p->S;
  const int64_t n = p->n_rcs();
  const double* radius = p->scal.p + S_RADIUS;
  fam_begin(p, F_SCHUR);
  BA_CUDA_TRY(cudaMemsetAsync(p->status.p, 0, sizeof(int), p->st));
  BA_LAUNCH(p, KT_ECHOL, (k_e_chol<DE>), grid_for(S.ne, 256), 256, 0, S.ne, p->ME.p, radius, opt.min_lm_diagonal, opt.max_lm_diagonal,
            p->Lb.p, p->zb.p, p->status.p);
  if (p->model == 0)
    BA_LAUNCH(p, KT_INCY, (k_inc_Y<RD, DE, true>), grid_for(S.ninc, 128), 128, 0, S.ninc, S.inc_e, p->JE.p, p->JF0.p, nullptr, p->Lb.p,
              p->zb.p, p->Yt.p, p->vb.p);
  else
    BA_LAUNCH(p, KT_INCY, (k_inc_Y<RD, DE, false>), grid_for(S.ninc, 128), 128, 0, S.ninc, S.inc_e, nullptr, nullptr, p->Wt.p, p->Lb.p,
              p->zb.p, p->Yt.p, p->vb.p);
  const bool pcg = p->solver == BA_RCS_PCG;
  if (pcg) { if (p->world > 1) BA_CUDA_TRY(cudaMemsetAsync(p->Sb.p, 0, p->Sb.bytes(), p->st)); }
  else BA_CUDA_TRY(cudaMemsetAsync(p->Sd.p, 0, sizeof(double) * (n * n + n), p->st));
  if (S.ch_finc.n > 0)
    BA_LAUNCH(p, KT_FINC, k_finc_partial, grid_for(S.ch_finc.n, 4), 128, 0, S.ch_finc.n, S.ch_finc.ch, S.ch_finc.seg.p, S.ch_finc.begin.p,
              S.finc_ptr.p, S.finc.p, p->vb.p, p->part_finc.p);
  BA_LAUNCH(p, KT_SEGFIN, (k_seg_final<6>), grid_for(S.nf, 4), 128, 0, (int)S.nf, S.ch_finc.seg_first.p, p->part_finc.p, p->vsum());
  BA_LAUNCH(p, KT_PAIRS, (k_pairs_partial<DE>), grid_for(S.ch_pairs.n, 4), 128, 0, S.ch_pairs.n, S.ch_pairs.ch, S.ch_pairs.seg.p,
            S.ch_pairs.begin.p, S.dpair_ptr.p, S.pairs.p, p->Yt.p, p->part_pairs.p);
  BA_LAUNCH(p, KT_SEGFIN, (k_seg_final<36>), grid_for(S.ndest, 4), 128, 0, S.ndest, S.ch_pairs.seg_first.p, p->part_pairs.p, p->Pacc.p);
  if (pcg)
    BA_LAUNCH(p, KT_ASSEMBLE, k_assemble_bsr, grid_for((int64_t)S.ndest * 36, 256), 256, 0, S.ndest, p->R.l2g.p, p->Pacc.p,
              p->model == 1 ? p->Qacc.p : nullptr, p->Sb.p);
  else
    BA_LAUNCH(p, KT_ASSEMBLE, k_assemble_dense, grid_for((int64_t)S.ndest * 36, 256), 256, 0, S.ndest, S.dest_fa.p, S.dest_fb.p, p->Pacc.p,
              p->model == 1 ? p->Qacc.p : nullptr, n, p->Sd.p);
  BA_CUDA_TRY(cudaGetLastError());
  fam_end(p, F_SCHUR);
  if (p->world > 1) {
    fam_begin(p, F_COLL);
    // partial RCS and the partial rhs correction in one call
    if (pcg) BA_TRY(allreduce(p, p->Sb.p, p->Sb.n, kNcclSum));
    else BA_TRY(allreduce(p, p->Sd.p, n * n + n, kNcclSum));
    fam_end(p, F_COLL);
  }
  fam_begin(p, F_SOLVE);
  if (pcg)
    BA_LAUNCH(p, KT_ASSEMBLE, k_diag_rhs_bsr<>, grid_for(S.nf * 6, 128), 128, 0, S.nf, p->R.diag.p, p->HG.p, NV_F, p->vsum(), 6, radius,
              opt.min_lm_diagonal, opt.max_lm_diagonal, p->Sb.p, p->rhs.p);
  else
    BA_LAUNCH(p, KT_ASSEMBLE, k_diag_rhs_dense<>, grid_for(S.nf * 6, 128), 128, 0, S.nf, p->HG.p, NV_F, p->vsum(), 6, radius, opt.min_lm_diagonal,
              opt.max_lm_diagonal, n, p->Sd.p, p->rhs.p);
  return BA_OK;
}

// LevenbergMarquardtStrategy::ComputeStep + SchurEliminator + dense Cholesky + BackSubstitute + the model cost
// change and the candidate point.  scal[S_RADIUS] must hold the trust-region radius.
template <int RD, int DE, int GE, int NSLOT>
int compute_step(ba_cuda_problem* p, const ba_cuda_options& opt) {
  const Structure& S = p->S;
  const int64_t n = p->n_rcs();
  BA_TRY((schur_complement<RD, DE>(p, opt)));
  if (p->solver == BA_RCS_PCG) {
    {
      LaunchScope scope(p, KT_RCS);
      BA_TRY(launch_pcg(p->pcg, p->R, p->Sb.p, p->rhs.p, p->yf.p, p->status.p, opt, p->st));
    }
    BA_CUDA_TRY(cudaMemcpyAsync(&p->h_pcg_iters, p->pcg.iters.p, sizeof(int), cudaMemcpyDeviceToHost, p->st));
  } else {
    LaunchScope scope(p, KT_RCS);
    BA_TRY(dense_solve(p, n));
  }
  fam_end(p, F_SOLVE);
  fam_begin(p, F_UPDATE);
  BA_LAUNCH(p, KT_BACKSUB, (k_e_backsub<DE, GE>), grid_for(S.ne * GE, 128), 128, 0, S.ne, S.einc_ptr, S.inc_f, p->Yt.p, p->Lb.p, p->zb.p,
            p->yf.p, p->ye.p);
  const int gm = (int)grid_for(S.nb * RD, 256);   // one thread per residual row
  BA_LAUNCH(p, KT_MODELCOST, (k_model_cost<RD, DE, NSLOT>), gm, 256, 0, S.nb, S.ob_e.p, S.ob_f0.p, S.ob_f1.p, p->RES.p, p->JE.p, p->JF0.p,
            p->JF1.p, p->ye.p, p->yf.p, p->bp0.p);
  BA_TRY(fold(p, p->bp0.p, gm, S_MCC));
  const int gce = (int)grid_for(S.ne * DE, 256), gcf = (int)grid_for(S.nf * 6, 256);
  BA_LAUNCH(p, KT_CANDIDATE, (k_candidate<DE>), gce, 256, 0, S.ne, S.e_ptr.p, p->xe.p, p->se.p, p->ye.p, p->xe_c.p, p->bp0.p, p->bp1.p);
  {
    FoldJob J = {{p->bp0.p, p->bp1.p, nullptr, nullptr}, {S_XE2, S_DE2, 0, 0}, {0, 0, 0, 0}};
    BA_LAUNCH(p, KT_FOLD, k_fold_multi, 2, 1024, 0, J, gce, p->scal.p);
  }
  BA_LAUNCH(p, KT_CANDIDATE, (k_candidate<6>), gcf, 256, 0, S.nf, p->f_act_ptr.p, p->xf.p, p->sf.p, p->yf.p, p->xf_c.p, p->bp0.p, p->bp1.p);
  {
    FoldJob J = {{p->bp0.p, p->bp1.p, nullptr, nullptr}, {S_XF2, S_DF2, 0, 0}, {0, 0, 0, 0}};
    BA_LAUNCH(p, KT_FOLD, k_fold_multi, 2, 1024, 0, J, gcf, p->scal.p);
  }
  BA_CUDA_TRY(cudaGetLastError());
  fam_end(p, F_UPDATE);
  fam_begin(p, F_COST);
  BA_TRY(run_cost_candidate(p));
  fam_end(p, F_COST);
  return allreduce_step_scalars(p);
}

// ---- fused Model A path (ba_fused_a.cuh) -------------------------------------------------------------
FaParams fa_params(ba_cuda_problem* p, const ba_cuda_options& opt) {
  const Structure& S = p->S;
  FusedA& F = p->FA;
  const size_t nt = (size_t)F.n_tiles;
  FaParams P;
  P.tiles = F.tiles.p; P.e_ptr = S.e_ptr.p; P.ob_f = S.ob_f0.p; P.uv = p->uv.p;
  P.ob_meta = p->use_strip ? p->SA.ob_meta.p : F.ob_meta.p;
  P.tile_cams = p->use_strip ? p->SA.strip_cams.p : F.cams.group_target.p; P.cap = F.cap;
  P.pts_cap = F.pts_cap; P.tcam = F.tcam; P.tcs = F.tcs; P.pent_cap = F.pent_cap;
  P.pitem_begin = F.pairs.item_begin.p; P.pitem_end = F.pairs.item_end.p; P.pent = F.pairs.ent.p;
  P.citem_begin = F.cams.item_begin.p; P.citem_end = F.cams.item_end.p; P.cent = F.cams.ent.p;
  P.xe = p->xe.p; P.se = p->se.p; P.tab_f = p->tab_f.p; P.radius = p->scal.p + S_RADIUS;
  P.min_diag = opt.min_lm_diagonal; P.max_diag = opt.max_lm_diagonal;
  P.partP = F.red_pairs.part.p; P.partC = F.red_cams.part.p; P.Lz = F.Lz.p; P.se_out = p->se.p;
  P.cost_partial = p->fa_part.p; P.g2_partial = p->fa_part.p + nt; P.gmax_partial = p->fa_part.p + 2 * nt;
  P.yf = p->yf.p; P.tabc_f = p->tabc_f.p; P.xe_c = p->xe_c.p;
  P.mcc_partial = p->fa_part.p + 3 * nt; P.x2_partial = p->fa_part.p + 4 * nt; P.d2_partial = p->fa_part.p + 5 * nt;
  P.cand_partial = p->fa_part.p + 6 * nt;
  P.RES = p->RES.p; P.JE = p->JE.p; P.JF = p->JF0.p;
  P.status = p->status.p;
  P.loss = p->loss;
  return P;
}

int fa_set_smem_attr(ba_cuda_problem* p) {
  if (!p->smem_attr_set) {   // per device (the attribute lives in the context of the device this problem runs on)
    const int kMax = (int)FA_SMEM_MAX;  // dynamic part; the kernels also hold a little static shared memory
    BA_CUDA_TRY(cudaFuncSetAttribute(k_fa_pass1<FA_FULL>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMax));
    BA_CUDA_TRY(cudaFuncSetAttribute(k_fa_pass1<FA_NORMS>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMax));
    BA_CUDA_TRY(cudaFuncSetAttribute(k_fa_pass1<FA_GRAD>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMax));
    BA_CUDA_TRY(cudaFuncSetAttribute(k_fa_pass1<FA_FIRST>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMax));
    BA_CUDA_TRY(cudaFuncSetAttribute(k_fa_pass2, cudaFuncAttributeMaxDynamicSharedMemorySize, kMax));
    BA_CUDA_TRY(cudaFuncSetAttribute(k_fa_jac, cudaFuncAttributeMaxDynamicSharedMemorySize, kMax));
    BA_CUDA_TRY(cudaFuncSetAttribute(k_sa_pass1<SA_FULL>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMax));
    BA_CUDA_TRY(cudaFuncSetAttribute(k_sa_pass1<SA_GRAD>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMax));
    BA_CUDA_TRY(cudaFuncSetAttribute(k_sa_pass1<SA_FIRST>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMax));
    p->smem_attr_set = true;
  }
  return BA_OK;
}

// Sums the partial blocks of one reduction list per target into out (n_targets blocks of NV doubles), in a fixed order.
template <int NV>
int reduce_partials(ba_cuda_problem* p, const ReduceList& R, int n_targets, double* out) {
  if (R.ch.n > 0)
    BA_LAUNCH(p, KT_FA_RED, (k_reduce_items<NV>), grid_for(R.ch.n, 4), 128, 0, R.ch.n, R.ch.ch, R.ch.seg.p, R.ch.begin.p, R.tgt_ptr.p,
              R.items.p, R.part.p, R.red1.p);
  BA_LAUNCH(p, KT_FA_RED, (k_reduce_final<NV>), grid_for(n_targets, 4), 128, 0, n_targets, R.ch.seg_first.p, R.red1.p, out);
  return BA_OK;
}

// Pass 1 on single tiles (ba_fused_a.cuh); n_cta: the number of CTAs, each leaving its cost / gradient partials in fa_part.
int fa_pass1(ba_cuda_problem* p, const ba_cuda_options& opt, bool grad_only, bool first, int& n_cta) {
  const FusedA& F = p->FA;
  const FaParams P = fa_params(p, opt);
  n_cta = F.n_tiles;
  if (grad_only) BA_LAUNCH(p, KT_FA_P1L, (k_fa_pass1<FA_GRAD>), n_cta, F.threads, F.smem1(), P);
  else if (first) BA_LAUNCH(p, KT_FA_P1, (k_fa_pass1<FA_FIRST>), n_cta, F.threads, F.smem1(), P);
  else BA_LAUNCH(p, KT_FA_P1, (k_fa_pass1<FA_FULL>), n_cta, F.threads, F.smem1(), P);
  return BA_OK;
}

// Pass 1 on strips (ba_strip_a.cuh): one CTA linearises, eliminates and accumulates the Schur products of a strip.
int sa_pass1(ba_cuda_problem* p, const ba_cuda_options& opt, bool grad_only, bool first, int& n_cta) {
  const StripA& A = p->SA;
  const size_t ns = (size_t)A.n_strips;
  SaParams P;
  P.strips = A.strips.p; P.tiles = A.tiles.p; P.strip_cams = A.strip_cams.p; P.slot_out = A.slot_out.p;
  P.pm = A.pm.p; P.puv = A.puv.p; P.pidx = A.pidx.p; P.ent = A.ent.p; P.seg = A.seg.p;
  P.segw = A.segw; P.cap_pos = A.cap_pos; P.pts_cap = A.pts_cap; P.tcs = A.tcs; P.ent_cap = A.ent_cap; P.pidx_cap = A.pidx_cap;
  P.xe = p->xe.p; P.se = p->se.p; P.tab_f = p->tab_f.p; P.radius = p->scal.p + S_RADIUS;
  P.min_diag = opt.min_lm_diagonal; P.max_diag = opt.max_lm_diagonal;
  P.partP = A.red_pairs.part.p; P.partC = A.red_cams.part.p; P.n_pout = A.n_pout;
  P.Lz = p->FA.Lz.p; P.se_out = p->se.p;
  P.cost_partial = p->fa_part.p; P.g2_partial = p->fa_part.p + ns; P.gmax_partial = p->fa_part.p + 2 * ns;
  P.status = p->status.p;
  P.dbg = env_int("BA_SA_DBG", 0, 7, 0);
  P.loss = p->loss;
  static DVec<unsigned long long>* clk = nullptr;   // BA_SA_CLOCKS=1: cycles of thread 0 per phase of pass 1, printed per launch (tuning aid)
  P.clocks = nullptr;
  if (env_int("BA_SA_CLOCKS", 0, 1, 0)) {
    if (!clk) { clk = new DVec<unsigned long long>(); BA_TRY(clk->alloc(8)); }
    BA_CUDA_TRY(cudaMemsetAsync(clk->p, 0, 8 * sizeof(unsigned long long), p->st));
    P.clocks = clk->p;
  }
  n_cta = A.n_strips;
  if (first) BA_LAUNCH(p, KT_FA_P1, (k_sa_pass1<SA_FIRST>), n_cta, SA_NT, A.smem(), P);
  else if (grad_only) BA_LAUNCH(p, KT_FA_P1L, (k_sa_pass1<SA_GRAD>), n_cta, SA_NT, A.smem(), P);
  else BA_LAUNCH(p, KT_FA_P1, (k_sa_pass1<SA_FULL>), n_cta, SA_NT, A.smem(), P);
  if (P.clocks) {
    unsigned long long h[8];
    BA_CUDA_TRY(cudaMemcpyAsync(h, P.clocks, sizeof(h), cudaMemcpyDeviceToHost, p->st));
    BA_CUDA_TRY(cudaStreamSynchronize(p->st));
    const double n = (double)A.n_tiles;
    std::fprintf(stderr, "[ba_cuda clocks] pass 1, cycles per tile as thread 0 sees them: top %.0f | wait inputs %.0f | A1 + barrier %.0f | A2 (own) %.0f | "
                         "wait entries + barrier %.0f | B (own) %.0f | barrier after B %.0f | sum %.0f\n", h[0] / n, h[1] / n, h[2] / n, h[3] / n, h[4] / n,
                 h[5] / n, h[6] / n, (h[0] + h[1] + h[2] + h[3] + h[4] + h[5] + h[6]) / n);
  }
  return BA_OK;
}

// Width of the per-camera record of the fused path: strips keep diag F^T F in a slot of its own (SA_NVC), single tiles
// read it from the packed F^T F (FA_NVC).
int fa_nvc(const ba_cuda_problem* p) { return p->use_strip ? SA_NVC : FA_NVC; }

// r, J, cost, gradient norms at x AND the eliminated Schur system for the radius in scal[S_RADIUS]
// (TrustRegionMinimizer::EvaluateGradientAndJacobian + SchurEliminator::Eliminate in one pass).
// norms = true (single tiles only): iteration 0, computes the Jacobi scaling only.  grad_only = true: no further step can
// follow (the iteration limit is reached), so only what the row of the progress table needs is computed: cost and
// gradient.  first = true: iteration 0 with Jacobi scaling in one pass (FA_FIRST / SA_FIRST): the point scaling is applied
// inside the pass, the camera scaling to the reduced results.  NVC: the camera record of the geometry (fa_nvc).
template <int NVC>
int fused_linearize(ba_cuda_problem* p, const ba_cuda_options& opt, bool norms, bool grad_only, bool first) {
  constexpr bool strip = NVC == SA_NVC;
  constexpr int DIAG = strip ? 33 : -1;   // where diag F^T F sits in the record (-1: the packed diagonal)
  const Structure& S = p->S;
  FusedA& F = p->FA;
  const ReduceList& red_cams = strip ? p->SA.red_cams : F.red_cams;
  const ReduceList& red_pairs = strip ? p->SA.red_pairs : F.red_pairs;
  BA_TRY(fa_set_smem_attr(p));
  fam_begin(p, F_JAC);
  if (norms || first) {
    BA_LAUNCH(p, KT_MISC, k_fill, grid_for(S.nf * 6, 256), 256, 0, p->sf.p, S.nf * 6, 1.0);
    BA_LAUNCH(p, KT_MISC, k_fill, grid_for(S.ne * 3, 256), 256, 0, p->se.p, S.ne * 3, 1.0);
  }
  BA_TRY(build_tables(p, false));
  if (norms) {
    BA_LAUNCH(p, KT_FA_P1L, (k_fa_pass1<FA_NORMS>), F.n_tiles, F.threads, F.smem1(), fa_params(p, opt));
    BA_TRY(reduce_partials<NVC>(p, red_cams, (int)S.nf, F.camacc.p));
    BA_CUDA_TRY(cudaGetLastError());
    BA_TRY(allreduce(p, F.camacc.p, (size_t)S.nf * NVC, kNcclSum));
    BA_LAUNCH(p, KT_MISC, (k_jacobi_scale<6, NVC, DIAG>), grid_for(S.nf * 6, 256), 256, 0, S.nf, F.camacc.p, p->sf.p);
    BA_CUDA_TRY(cudaGetLastError());
    fam_end(p, F_JAC);
    return BA_OK;
  }
  BA_CUDA_TRY(cudaMemsetAsync(p->status.p, 0, sizeof(int), p->st));
  int n_cta = 0;
  BA_TRY(strip ? sa_pass1(p, opt, grad_only, first, n_cta) : fa_pass1(p, opt, grad_only, first, n_cta));
  {
    const double* part = p->fa_part.p;
    FoldJob J = {{part, part + n_cta, part + 2 * (size_t)n_cta, nullptr}, {S_COST, S_G2E, S_GMAXE, 0}, {0, 0, 1, 0}};
    BA_LAUNCH(p, KT_FOLD, k_fold_multi, 3, 1024, 0, J, n_cta, p->scal.p);
  }
  fam_end(p, F_JAC);
  // the pair blocks are needed for a step, and on strips also for the scaling of iteration 0
  const bool pairs = !grad_only || (strip && first);
  fam_begin(p, F_SCHUR);
  BA_TRY(reduce_partials<NVC>(p, red_cams, (int)S.nf, F.camacc.p));
  if (pairs) BA_TRY(reduce_partials<36>(p, red_pairs, S.ndest, p->Pacc.p));
  BA_CUDA_TRY(cudaGetLastError());
  fam_end(p, F_SCHUR);
  const bool sx = sx_active(p);
  if (p->world > 1) {  // camera sums and the shard-local gradient scalars in one collective; the partial blocks too when they travel sparse
    fam_begin(p, F_COLL);
    if (sx) BA_TRY(sx_exchange(p, F.camacc.p, pairs));
    else BA_TRY(allreduce_with_grad_tail(p, F.camacc.p, (size_t)S.nf * NVC));
    fam_end(p, F_COLL);
  }
  if (first) {  // camera scaling from the (global) unscaled column norms, then everything reduced so far into scaled columns
    BA_LAUNCH(p, KT_MISC, (k_jacobi_scale<6, NVC, DIAG>), grid_for(S.nf * 6, 256), 256, 0, S.nf, F.camacc.p, p->sf.p);
    BA_LAUNCH(p, KT_MISC, (k_fa_scale_cams<NVC>), grid_for(S.nf * NVC, 256), 256, 0, S.nf, p->sf.p, F.camacc.p);
    if (sx) BA_LAUNCH(p, KT_MISC, k_sx_scale_blocks, grid_for((int64_t)p->R.nd * 36, 256), 256, 0, p->R.nd, p->R.fa.p, p->R.fb.p, p->sf.p, p->Sb.p);
    else
    BA_LAUNCH(p, KT_MISC, k_fa_scale_pairs, grid_for((int64_t)S.ndest * 36, 256), 256, 0, S.ndest, S.dest_fa.p, S.dest_fb.p, p->sf.p, p->Pacc.p);
    BA_TRY(build_tables(p, false));   // pass 2 linearises with the scaled camera columns
  }
  const int gf = (int)grid_for(S.nf * 6, 256);
  BA_LAUNCH(p, KT_GRADNORM, (k_gradient_norm<6, NVC, 21>), gf, 256, 0, S.nf, p->f_act_ptr.p, p->xf.p, p->sf.p, F.camacc.p, p->bp0.p, p->bp1.p);
  {
    FoldJob J = {{p->bp0.p, p->bp1.p, nullptr, nullptr}, {S_GMAXF, S_G2F, 0, 0}, {1, 0, 0, 0}};
    BA_LAUNCH(p, KT_FOLD, k_fold_multi, 2, 1024, 0, J, gf, p->scal.p);
  }
  BA_CUDA_TRY(cudaGetLastError());
  return BA_OK;
}

// Strips never take the separate scaling pass (norms): they always scale in one pass.
int fa_linearize(ba_cuda_problem* p, const ba_cuda_options& opt, bool norms, bool grad_only = false, bool first = false) {
  if (fa_nvc(p) == SA_NVC) return fused_linearize<SA_NVC>(p, opt, false, grad_only, first);
  return fused_linearize<FA_NVC>(p, opt, norms, grad_only, first);
}

// RCS assembly + solve + (pass 2) back-substitution, model cost change, candidate and its cost
template <int NVC>
int fused_step(ba_cuda_problem* p, const ba_cuda_options& opt) {
  constexpr int DIAG = NVC == SA_NVC ? 33 : -1;   // as in fused_linearize
  const Structure& S = p->S;
  FusedA& F = p->FA;
  const int64_t n = p->n_rcs();
  const double* radius = p->scal.p + S_RADIUS;
  const bool pcg = p->solver == BA_RCS_PCG;
  const bool sx = sx_active(p);   // the block values were exchanged and assembled with the linearisation (sx_exchange)
  fam_begin(p, F_SCHUR);
  if (pcg && sx) {
  } else if (pcg) {
    if (p->world > 1) BA_CUDA_TRY(cudaMemsetAsync(p->Sb.p, 0, p->Sb.bytes(), p->st));
    BA_LAUNCH(p, KT_ASSEMBLE, k_assemble_bsr, grid_for((int64_t)S.ndest * 36, 256), 256, 0, S.ndest, p->R.l2g.p, p->Pacc.p, nullptr, p->Sb.p);
  } else {
    BA_CUDA_TRY(cudaMemsetAsync(p->Sd.p, 0, sizeof(double) * n * n, p->st));
    BA_LAUNCH(p, KT_ASSEMBLE, k_assemble_dense, grid_for((int64_t)S.ndest * 36, 256), 256, 0, S.ndest, S.dest_fa.p, S.dest_fb.p, p->Pacc.p,
              nullptr, n, p->Sd.p);
  }
  fam_end(p, F_SCHUR);
  if (p->world > 1 && !(pcg && sx)) {
    fam_begin(p, F_COLL);
    if (pcg) BA_TRY(allreduce(p, p->Sb.p, (size_t)p->R.nd * 36, kNcclSum));
    else BA_TRY(allreduce(p, p->Sd.p, n * n, kNcclSum));
    fam_end(p, F_COLL);
  }
  fam_begin(p, F_SOLVE);
  if (pcg) {
    BA_LAUNCH(p, KT_ASSEMBLE, k_diag_rhs_bsr<DIAG>, grid_for(S.nf * 6, 128), 128, 0, S.nf, p->R.diag.p, F.camacc.p, NVC, F.camacc.p + 27, NVC,
              radius, opt.min_lm_diagonal, opt.max_lm_diagonal, p->Sb.p, p->rhs.p);
    {
      LaunchScope scope(p, KT_RCS);
      BA_TRY(launch_pcg(p->pcg, p->R, p->Sb.p, p->rhs.p, p->yf.p, p->status.p, opt, p->st));
    }
    BA_CUDA_TRY(cudaMemcpyAsync(&p->h_pcg_iters, p->pcg.iters.p, sizeof(int), cudaMemcpyDeviceToHost, p->st));
  } else {
    BA_LAUNCH(p, KT_ASSEMBLE, k_diag_rhs_dense<DIAG>, grid_for(S.nf * 6, 128), 128, 0, S.nf, F.camacc.p, NVC, F.camacc.p + 27, NVC, radius,
              opt.min_lm_diagonal, opt.max_lm_diagonal, n, p->Sd.p, p->rhs.p);
    LaunchScope scope(p, KT_RCS);
    BA_TRY(dense_solve(p, n));
  }
  fam_end(p, F_SOLVE);
  fam_begin(p, F_UPDATE);
  const int gcf = (int)grid_for(S.nf * 6, 256);
  BA_LAUNCH(p, KT_CANDIDATE, (k_candidate<6>), gcf, 256, 0, S.nf, p->f_act_ptr.p, p->xf.p, p->sf.p, p->yf.p, p->xf_c.p, p->bp0.p, p->bp1.p);
  {
    FoldJob J = {{p->bp0.p, p->bp1.p, nullptr, nullptr}, {S_XF2, S_DF2, 0, 0}, {0, 0, 0, 0}};
    BA_LAUNCH(p, KT_FOLD, k_fold_multi, 2, 1024, 0, J, gcf, p->scal.p);
  }
  BA_TRY(build_tables(p, true));
  const FaParams P = fa_params(p, opt);
  BA_LAUNCH(p, KT_FA_P2, k_fa_pass2, F.n_tiles, F.threads2, F.smem2(), P);
  {
    FoldJob J = {{P.mcc_partial, P.x2_partial, P.d2_partial, P.cand_partial}, {S_MCC, S_XE2, S_DE2, S_CAND}, {0, 0, 0, 0}};
    BA_LAUNCH(p, KT_FOLD, k_fold_multi, 4, 1024, 0, J, F.n_tiles, p->scal.p);
  }
  BA_CUDA_TRY(cudaGetLastError());
  fam_end(p, F_UPDATE);
  return allreduce_step_scalars(p);
}
int fa_step(ba_cuda_problem* p, const ba_cuda_options& opt) {
  return fa_nvc(p) == SA_NVC ? fused_step<SA_NVC>(p, opt) : fused_step<FA_NVC>(p, opt);
}

bool lm_fused(const ba_cuda_problem* p) { return p->model == 0 && p->use_fused && !p->lm.opt.force_generic_path; }

// Sparse exchange (ba_exchange.cuh): which of my blocks / cameras travel, every rank's lists, the inverse maps.
int sx_prepare(ba_cuda_problem* p) {
  const Structure& S = p->S;
  SparseExchange& X = p->SX;
  X.on = false; X.world = p->world; X.nvc = fa_nvc(p);
  if (!nccl().AllGather || !env_int("BA_SX", 0, 1, 1)) return BA_OK;
  cudaStream_t st = p->st;
  const int64_t nf = S.nf, nd = p->R.nd;
  // my cameras, my sent blocks
  DVec<int32_t> cflag, cpos, dflag, dpos;
  BA_TRY(cflag.alloc(nf + 1)); BA_TRY(cpos.alloc(nf + 1)); BA_TRY(dflag.alloc((size_t)S.ndest + 1)); BA_TRY(dpos.alloc((size_t)S.ndest + 1));
  BA_CUDA_TRY(cudaMemsetAsync(cflag.p, 0, sizeof(int32_t) * (nf + 1), st));
  BA_CUDA_TRY(cudaMemsetAsync(dflag.p, 0, sizeof(int32_t) * ((size_t)S.ndest + 1), st));
  k_sx_flags<<<grid_for(nf, 256), 256, 0, st>>>(S.fobs_ptr.p, nf, cflag.p);
  k_sx_send_flags<<<grid_for(S.ndest, 256), 256, 0, st>>>(S.ndest, S.dest_fa.p, S.dest_fb.p, cflag.p, dflag.p);
  BA_TRY(cub_call([&](void* t, size_t& b) { return cub::DeviceScan::ExclusiveSum(t, b, cflag.p, cpos.p, (int)(nf + 1), st); }));
  BA_TRY(cub_call([&](void* t, size_t& b) { return cub::DeviceScan::ExclusiveSum(t, b, dflag.p, dpos.p, S.ndest + 1, st); }));
  int32_t h2[2] = {0, 0};
  BA_CUDA_TRY(cudaMemcpyAsync(&h2[0], cpos.p + nf, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  BA_CUDA_TRY(cudaMemcpyAsync(&h2[1], dpos.p + S.ndest, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  BA_CUDA_TRY(cudaStreamSynchronize(st));
  X.nc_local = h2[0]; X.n_send = h2[1];
  BA_TRY(X.my_cams.alloc((size_t)X.nc_local)); BA_TRY(X.send_d.alloc((size_t)X.n_send));
  k_sx_compact<<<grid_for(nf, 256), 256, 0, st>>>(cflag.p, cpos.p, nf, X.my_cams.p);
  k_sx_compact<<<grid_for(S.ndest, 256), 256, 0, st>>>(dflag.p, dpos.p, S.ndest, X.send_d.p);
  // every rank's counts
  DVec<int64_t> cnt;
  BA_TRY(cnt.alloc(2 * (size_t)p->world));
  const int64_t mine[2] = {X.n_send, X.nc_local};
  BA_CUDA_TRY(cudaMemcpyAsync(cnt.p + 2 * p->rank, mine, sizeof(mine), cudaMemcpyHostToDevice, st));
  int rc = nccl().AllGather(cnt.p + 2 * p->rank, cnt.p, 2, kNcclInt64, p->comm, st);
  if (rc != 0) return fail(BA_ERR_NCCL, "ncclAllGather failed (%d)", rc);
  std::vector<int64_t> h(2 * (size_t)p->world);
  BA_CUDA_TRY(cudaMemcpyAsync(h.data(), cnt.p, sizeof(int64_t) * h.size(), cudaMemcpyDeviceToHost, st));
  BA_CUDA_TRY(cudaStreamSynchronize(st));
  int64_t sum_nd = 0, max_nd = 1, max_nc = 1;
  for (int r = 0; r < p->world; ++r) { sum_nd += h[2 * r]; max_nd = std::max(max_nd, h[2 * r]); max_nc = std::max(max_nc, h[2 * r + 1]); }
  // worth it only while the shards' lists are (nearly) disjoint: the all-reduce moves ~2 nd blocks per rank, the all-gather sum_nd
  if ((double)max_nd * p->world > 1.5 * (double)nd) return BA_OK;
  X.max_nd = (int)max_nd; X.max_nc = (int)max_nc;
  X.slot = (size_t)max_nd * 36 + (size_t)max_nc * X.nvc + 4;
  // every rank's lists -> inverse maps
  DVec<int32_t> lists_d, lists_c;
  BA_TRY(lists_d.alloc((size_t)max_nd * p->world)); BA_TRY(lists_c.alloc((size_t)max_nc * p->world));
  BA_CUDA_TRY(cudaMemsetAsync(lists_d.p, 0xff, sizeof(int32_t) * (size_t)max_nd * p->world, st));
  BA_CUDA_TRY(cudaMemsetAsync(lists_c.p, 0xff, sizeof(int32_t) * (size_t)max_nc * p->world, st));
  k_sx_gather_l2g<<<grid_for(X.n_send, 256), 256, 0, st>>>(X.n_send, X.send_d.p, p->R.l2g.p, lists_d.p + (size_t)max_nd * p->rank);
  BA_CUDA_TRY(cudaMemcpyAsync(lists_c.p + (size_t)max_nc * p->rank, X.my_cams.p, sizeof(int32_t) * X.nc_local, cudaMemcpyDeviceToDevice, st));
  rc = nccl().AllGather(lists_d.p + (size_t)max_nd * p->rank, lists_d.p, (size_t)max_nd, kNcclInt32, p->comm, st);
  if (rc == 0) rc = nccl().AllGather(lists_c.p + (size_t)max_nc * p->rank, lists_c.p, (size_t)max_nc, kNcclInt32, p->comm, st);
  if (rc != 0) return fail(BA_ERR_NCCL, "ncclAllGather failed (%d)", rc);
  BA_TRY(X.inv_d.alloc((size_t)nd * p->world)); BA_TRY(X.inv_c.alloc((size_t)nf * p->world));
  BA_CUDA_TRY(cudaMemsetAsync(X.inv_d.p, 0xff, sizeof(int32_t) * (size_t)nd * p->world, st));
  BA_CUDA_TRY(cudaMemsetAsync(X.inv_c.p, 0xff, sizeof(int32_t) * (size_t)nf * p->world, st));
  k_sx_invert<<<grid_for((int64_t)max_nd * p->world, 256), 256, 0, st>>>(p->world, (int)max_nd, lists_d.p, nd, X.inv_d.p);
  k_sx_invert<<<grid_for((int64_t)max_nc * p->world, 256), 256, 0, st>>>(p->world, (int)max_nc, lists_c.p, nf, X.inv_c.p);
  BA_TRY(X.buf.alloc(X.slot * p->world));
  BA_CUDA_TRY(cudaStreamSynchronize(st));
  BA_CUDA_TRY(cudaGetLastError());
  X.on = true;
  return BA_OK;
}

// After a linearisation: my blocks, my cameras' sums and my scalars to every rank in one all-gather; the pieces are then
// added in rank order: the global camera sums, the shard scalars and (with_blocks) the block values of the reduced system.
int sx_exchange(ba_cuda_problem* p, double* camacc, bool with_blocks) {
  const Structure& S = p->S;
  SparseExchange& X = p->SX;
  double* slot = X.buf.p + X.slot * p->rank;
  const int64_t n = (int64_t)X.slot;
  k_sx_pack<<<grid_for(n, 256), 256, 0, p->st>>>(X.n_send, X.send_d.p, p->Pacc.p, X.nc_local, X.my_cams.p, X.nvc, camacc, p->scal.p, S_COST, S_G2E,
                                              S_GMAXE, X.max_nd, X.max_nc, slot);
  const int rc = nccl().AllGather(slot, X.buf.p, X.slot, kNcclFloat64, p->comm, p->st);
  if (rc != 0) return fail(BA_ERR_NCCL, "ncclAllGather failed: %s", nccl().GetErrorString ? nccl().GetErrorString(rc) : "?");
  const size_t cam_off = (size_t)X.max_nd * 36;
  k_sx_unpack_cams<<<grid_for(S.nf * X.nvc, 256), 256, 0, p->st>>>(p->world, S.nf, X.nvc, X.slot, cam_off, X.buf.p, X.inv_c.p, camacc);
  k_sx_unpack_scalars<<<1, 32, 0, p->st>>>(p->world, X.slot, cam_off + (size_t)X.max_nc * X.nvc, X.buf.p, p->scal.p, S_COST, S_G2E, S_GMAXE);
  if (with_blocks)
    k_sx_unpack_blocks<<<grid_for((int64_t)p->R.nd * 36, 256), 256, 0, p->st>>>(p->world, p->R.nd, X.slot, X.buf.p, X.inv_d.p, p->Sb.p);
  BA_CUDA_TRY(cudaGetLastError());
  return BA_OK;
}
bool sx_active(const ba_cuda_problem* p) { return p->world > 1 && p->SX.on && p->solver == BA_RCS_PCG; }

// Resolves options.rcs_solver for this problem and makes sure the matching RCS storage exists.
// BA_RCS_AUTO: dense Cholesky while the system is rig sized (Ceres DENSE_SCHUR, what the reference asks for),
// block-sparse PCG above.
constexpr int64_t kDenseAutoMaxN = 1536;   // rigs (cameras + markers); BAL-scale camera counts go to PCG
constexpr int64_t kDenseMaxN = 16384;      // 2 GiB of fp64
int prepare_solver(ba_cuda_problem* p, const ba_cuda_options& opt) {
  const Structure& S = p->S;
  const int64_t n = p->n_rcs();
  int want = opt.rcs_solver;
  if (want == BA_RCS_AUTO) want = n <= kDenseAutoMaxN ? BA_RCS_DENSE_CHOLESKY : BA_RCS_PCG;
  if (want != BA_RCS_DENSE_CHOLESKY && want != BA_RCS_PCG) return fail(BA_ERR_INVALID_ARGUMENT, "unknown rcs_solver %d", opt.rcs_solver);
  if (want == BA_RCS_DENSE_CHOLESKY) {
    if (n > kDenseMaxN)
      return fail(BA_ERR_UNSUPPORTED, "dense RCS of dimension %lld is too large; use BA_RCS_PCG", (long long)n);
    if (p->Sd.n != (size_t)(n * n + n)) BA_TRY(p->Sd.alloc(n * n + n));
  } else {
    if (p->R.nd == 0 || p->R.nf != S.nf) {
      if (p->world > 1) BA_TRY(build_global_pattern(p));
      else BA_TRY(build_rcs_pattern(p->R, S.dest_keys.p, S.ndest, S.nf, p->st));
      BA_TRY(p->R.l2g.alloc(S.ndest));
      k_map_keys<<<grid_for(S.ndest, 256), 256, 0, p->st>>>(S.dest_keys.p, S.ndest, p->R.keys.p, p->R.nd, p->R.l2g.p);
      BA_CUDA_TRY(cudaGetLastError());
      BA_TRY(p->Sb.alloc((size_t)p->R.nd * 36 + (size_t)S.nf * 6));
      BA_TRY(pcg_prepare(p->pcg, S.nf, p->device));
      if (p->world > 1 && p->model == 0 && p->use_fused) BA_TRY(sx_prepare(p));
      BA_CUDA_TRY(cudaStreamSynchronize(p->st));
    }
  }
  p->solver = want;
  return BA_OK;
}

int fetch_scalars(ba_cuda_problem* p) {
  BA_CUDA_TRY(cudaMemcpyAsync(p->h_scal, p->scal.p, sizeof(double) * S_COUNT, cudaMemcpyDeviceToHost, p->st));
  BA_CUDA_TRY(cudaMemcpyAsync(p->h_status, p->status.p, sizeof(int), cudaMemcpyDeviceToHost, p->st));
  BA_CUDA_TRY(cudaStreamSynchronize(p->st));
  fam_collect(p);
  return BA_OK;
}

// FinalizeIterationAndCheckIfMinimizerCanContinue
bool lm_finalize(ba_cuda_problem* p, ba_cuda_iteration row, double iter_t0) {
  LmState& L = p->lm;
  const ba_cuda_options& opt = L.opt;
  ba_cuda_summary& Z = L.Z;
  if (row.step_is_successful) Z.num_successful_steps++; else Z.num_unsuccessful_steps++;
  row.trust_region_radius = L.radius;
  row.iteration_time_s = now_s() - iter_t0;
  p->rows.push_back(row);
  if (opt.minimizer_progress_to_stdout && p->rank == 0) {
    if (row.iteration == 0) std::printf("iter      cost      cost_change  |gradient|   |step|    tr_ratio  tr_radius\n");
    std::printf("%4d % 14.6e % 10.2e % 10.2e % 10.2e % 10.2e % 10.2e\n", row.iteration, row.cost, row.cost_change,
                row.gradient_max_norm, row.step_norm, row.relative_decrease, row.trust_region_radius);
  }
  if (row.iteration >= opt.max_num_iterations) { Z.termination_type = BA_NO_CONVERGENCE; Z.termination_reason = BA_REASON_MAX_ITERATIONS; return false; }
  if (row.step_is_successful && row.gradient_max_norm <= opt.gradient_tolerance) { Z.termination_type = BA_CONVERGENCE; Z.termination_reason = BA_REASON_GRADIENT_TOLERANCE; return false; }
  if (row.trust_region_radius <= opt.min_trust_region_radius) { Z.termination_type = BA_CONVERGENCE; Z.termination_reason = BA_REASON_MIN_TRUST_REGION_RADIUS; return false; }
  return true;
}

void lm_read_gradient(ba_cuda_problem* p) {
  LmState& L = p->lm;
  L.x_cost = 0.5 * p->h_scal[S_COST];
  L.gmax = std::max(p->h_scal[S_GMAXE], p->h_scal[S_GMAXF]);
  L.gnorm = std::sqrt(p->h_scal[S_G2E] + p->h_scal[S_G2F]);
}

// ---- the rig-size path (ba_rig.cuh): one CTA runs the whole loop ---------------------------------------------
int ensure_generic_workspace(ba_cuda_problem* p);
// the size and configuration test of the one-CTA path (ba_cuda_solve and ba_cuda_solve_batch); `solver` is the resolved
// rcs_solver, `max_rows` the residual-row limit
bool rig_fits(const ba_cuda_problem* p, int solver, bool force_generic_path, int64_t max_rows) {
  const int64_t rows = p->S.nb * (p->model == 0 ? 2 : 8);
  return p->world == 1 && !force_generic_path && solver == BA_RCS_DENSE_CHOLESKY && p->n_rcs() <= RIG_MAX_N && rows <= max_rows;
}
bool rig_eligible(const ba_cuda_problem* p, const ba_cuda_options& opt) {
  const bool on = env_int("BA_RIG", 0, 1, 1) != 0;   // read per solve: tests run both machines in one process
  const int64_t max_rows = env_int("BA_RIG_MAX_ROWS", 0, 1 << 30, (int)RIG_MAX_ROWS);   // tuning aid (profiles/tools/rig_crossover.py)
  return on && rig_fits(p, p->solver, opt.force_generic_path != 0, max_rows);
}

template <int RD, int DE, int GE, int NSLOT>
int rig_run(ba_cuda_problem* p, bool begin, int32_t max_new) {
  LmState& L = p->lm;
  const Structure& S = p->S;
  const size_t buf_bytes = sizeof(RigState) + sizeof(ba_cuda_iteration) * RIG_ROWS_CAP;
  if (p->rig_buf.n != buf_bytes) BA_TRY(p->rig_buf.alloc(buf_bytes));
  if (!p->h_rig) BA_CUDA_TRY(cudaMallocHost((void**)&p->h_rig, buf_bytes));
  const int n = (int)p->n_rcs();
  const size_t smem = rig_smem_bytes(n);
  if (!p->rig_attr_set) {
    BA_CUDA_TRY(cudaFuncSetAttribute(k_rig_lm<RD, DE, GE, NSLOT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rig_smem_bytes(RIG_MAX_N)));
    p->rig_attr_set = true;
  }
  RigParams P;
  std::memset(&P, 0, sizeof(P));
  P.nb = S.nb; P.ne = S.ne; P.nf = S.nf; P.ninc = S.ninc; P.ndest = S.ndest; P.n = n; P.ld = n | 1;
  P.ob_e = S.ob_e.p; P.ob_f0 = S.ob_f0.p; P.ob_f1 = S.ob_f1.p; P.ob_cam = p->ob_cam.p; P.e_ptr = S.e_ptr.p;
  P.inc_e = S.inc_e; P.inc_f = S.inc_f; P.einc_ptr = S.einc_ptr; P.incobs_ptr = S.incobs_ptr.p; P.incobs = S.incobs.p;
  P.finc_ptr = S.finc_ptr.p; P.fobs_ptr = S.fobs_ptr.p; P.finc = S.finc.p; P.fobs = S.fobs.p;
  P.dest_fa = S.dest_fa.p; P.dest_fb = S.dest_fb.p; P.dpair_ptr = S.dpair_ptr.p; P.pairs = S.pairs.p;
  P.dobs_ptr = S.dobs_ptr.p; P.dobs = S.dobs.p; P.f_act_ptr = p->f_act_ptr.p;
  P.uv = p->uv.p; P.obs8 = p->obs8.p; P.intr_f = p->intr_f.p; P.half_side = p->half_side;
  P.xe = p->xe.p; P.xf = p->xf.p; P.xe_c = p->xe_c.p; P.xf_c = p->xf_c.p; P.se = p->se.p; P.sf = p->sf.p;
  P.tab_f = p->tab_f.p; P.tab_e = p->tab_e.p; P.tabc_f = p->tabc_f.p; P.tabc_e = p->tabc_e.p;
  P.RES = p->RES.p; P.JE = p->JE.p; P.JF0 = p->JF0.p; P.JF1 = p->JF1.p; P.ME = p->ME.p; P.HG = p->HG.p; P.Wt = p->Wt.p;
  P.Qacc = p->Qacc.p; P.Lb = p->Lb.p; P.zb = p->zb.p; P.Yt = p->Yt.p; P.vb = p->vb.p; P.Pacc = p->Pacc.p; P.vsum = p->vsum();
  P.yf = p->yf.p; P.ye = p->ye.p;
  P.state = reinterpret_cast<RigState*>(p->rig_buf.p);
  P.rows = reinterpret_cast<ba_cuda_iteration*>(p->rig_buf.p + sizeof(RigState));
  P.opt = L.opt; P.loss = p->loss;
  static const bool clocks = env_int("BA_RIG_CLOCKS", 0, 1, 0) != 0;
  DVec<long long> clk;
  if (clocks) { BA_TRY(clk.alloc_zero(16, p->st)); P.clk = clk.p; }
  int64_t left = max_new;
  bool first = begin;
  while (first || (L.go && left > 0)) {
    P.begin = first ? 1 : 0;
    P.max_new = (int32_t)std::min<int64_t>(left, RIG_ROWS_CAP - P.begin);
    P.rows_base = (int32_t)p->rows.size();
    if (first) {
      std::memset(&P.init, 0, sizeof(P.init));
      P.init.radius = L.radius; P.init.decrease_factor = L.decrease_factor; P.init.go = 1;
    }
    BA_LAUNCH(p, KT_RIG, (k_rig_lm<RD, DE, GE, NSLOT>), 1, RIG_THREADS, smem, P);
    BA_CUDA_TRY(cudaGetLastError());
    BA_CUDA_TRY(cudaMemcpyAsync(p->h_rig, p->rig_buf.p, buf_bytes, cudaMemcpyDeviceToHost, p->st));
    BA_CUDA_TRY(cudaStreamSynchronize(p->st));
    fam_collect(p);
    const RigState& st = *reinterpret_cast<const RigState*>(p->h_rig);
    const ba_cuda_iteration* rows = reinterpret_cast<const ba_cuda_iteration*>(p->h_rig + sizeof(RigState));
    const int fresh = st.n_rows - P.rows_base;
    for (int r = 0; r < fresh && r < RIG_ROWS_CAP; ++r) {
      p->rows.push_back(rows[r]);
      if (L.opt.minimizer_progress_to_stdout) {
        const ba_cuda_iteration& row = rows[r];
        if (row.iteration == 0) std::printf("iter      cost      cost_change  |gradient|   |step|    tr_ratio  tr_radius\n");
        std::printf("%4d % 14.6e % 10.2e % 10.2e % 10.2e % 10.2e % 10.2e\n", row.iteration, row.cost, row.cost_change,
                    row.gradient_max_norm, row.step_norm, row.relative_decrease, row.trust_region_radius);
      }
    }
    L.radius = st.radius; L.decrease_factor = st.decrease_factor; L.x_cost = st.x_cost; L.gmax = st.gmax; L.gnorm = st.gnorm;
    L.num_invalid = st.num_invalid; L.go = st.go != 0;
    ba_cuda_summary& Z = L.Z;
    Z.num_jacobian_evaluations = st.n_jac; Z.num_linear_solves = st.n_solves; Z.num_cost_evaluations = st.n_solves;
    Z.num_successful_steps = st.n_success; Z.num_unsuccessful_steps = st.n_unsuccess;
    if (first) Z.initial_cost = st.n_rows > 0 ? p->rows.front().cost : st.x_cost;
    Z.final_cost = st.x_cost;
    if (!L.go) { Z.termination_type = st.term_type; Z.termination_reason = st.term_reason; }
    left -= P.max_new;
    first = false;
    if (clocks) {
      long long h[16];
      BA_CUDA_TRY(cudaMemcpy(h, clk.p, sizeof(h), cudaMemcpyDeviceToHost));
      static const char* const nm[16] = {"jacobian", "normal_parts", "gradient", "e_chol+inc_Y", "vsum+pairs", "assemble+diag", "ldlt+solve",
                                         "backsub+model_cost", "candidate", "cost_candidate", "decision", "other", "of_which_triangular_solves",
                                         "factor:(b)", "factor:barrier_after_b", "factor:diag_block"};
      std::fprintf(stderr, "[ba_cuda rig clocks] rows=%d", st.n_rows);
      for (int k = 0; k < 16; ++k) std::fprintf(stderr, " %s=%lld", nm[k], h[k]);
      std::fprintf(stderr, "\n");
    }
  }
  return BA_OK;
}

// TrustRegionMinimizer::IterationZero
template <int RD, int DE, int GE, int NSLOT>
int lm_begin(ba_cuda_problem* p, const ba_cuda_options& opt) {
  LmState& L = p->lm;
  L = LmState();
  L.opt = opt;
  L.t_start = now_s();
  std::memset(&L.Z, 0, sizeof(L.Z));
  p->rows.clear();
  p->profile = opt.profile_kernels != 0;
  for (int f = 0; f < F_COUNT; ++f) { p->fam_ms[f] = 0.0; p->fam_open[f] = false; }
  L.Z.num_residuals = p->nb_global * RD;
  L.Z.rcs_solver_used = p->solver;
  L.Z.path_used = lm_fused(p) ? (p->use_strip ? BA_PATH_FUSED_STRIPS : BA_PATH_FUSED_TILES) : BA_PATH_GENERIC;
  L.radius = opt.initial_trust_region_radius;
  L.decrease_factor = 2.0;
  L.began = true;
  if (rig_eligible(p, opt)) {   // the reference's own problem sizes: the whole loop in one CTA
    BA_TRY(ensure_generic_workspace(p));
    L.rig = true;
    L.Z.path_used = BA_PATH_RIG;
    if (p->one_shot) { L.rig_begin_pending = true; L.go = true; return BA_OK; }
    return rig_run<RD, DE, GE, NSLOT>(p, true, 0);
  }
  const double iter_t0 = now_s();
  if (lm_fused(p)) {
    static const bool one_pass = env_int("BA_FA_FIRST", 0, 1, 1) != 0;
    const bool first = opt.jacobi_scaling && (p->use_strip || (opt.max_num_iterations > 0 && one_pass));   // the strip path always scales in one pass
    if (!opt.jacobi_scaling) {  // a previous solve of this problem may have left its scaling behind
      BA_LAUNCH(p, KT_MISC, k_fill, grid_for(p->S.nf * 6, 256), 256, 0, p->sf.p, p->S.nf * 6, 1.0);
      BA_LAUNCH(p, KT_MISC, k_fill, grid_for(p->S.ne * 3, 256), 256, 0, p->se.p, p->S.ne * 3, 1.0);
    }
    if (opt.jacobi_scaling && !first) BA_TRY(fa_linearize(p, opt, true));
    BA_CUDA_TRY(cudaMemcpyAsync(p->scal.p + S_RADIUS, &L.radius, sizeof(double), cudaMemcpyHostToDevice, p->st));
    BA_TRY(fa_linearize(p, opt, false, opt.max_num_iterations <= 0, first));
  } else {
    BA_TRY((eval_gradient_and_jacobian<RD, DE, GE>(p, true, opt.jacobi_scaling != 0)));
  }
  L.Z.num_jacobian_evaluations++;
  BA_TRY(fetch_scalars(p));
  lm_read_gradient(p);
  ba_cuda_iteration row;
  std::memset(&row, 0, sizeof(row));
  L.Z.initial_cost = L.Z.final_cost = L.x_cost;
  if (!std::isfinite(L.x_cost)) {
    L.Z.termination_type = BA_FAILURE; L.Z.termination_reason = BA_REASON_INITIAL_EVALUATION_FAILED;
    L.go = false;
    return BA_OK;
  }
  row.iteration = 0; row.step_is_valid = 1; row.step_is_successful = 1; row.cost = L.x_cost;
  row.gradient_max_norm = L.gmax; row.gradient_norm = L.gnorm;
  L.go = lm_finalize(p, row, iter_t0);
  return BA_OK;
}

// the trust-region loop body, at most max_new more rows
template <int RD, int DE, int GE, int NSLOT>
int lm_iterate(ba_cuda_problem* p, int32_t max_new) {
  LmState& L = p->lm;
  const ba_cuda_options& opt = L.opt;
  ba_cuda_summary& Z = L.Z;
  ba_cuda_iteration row;
  if (L.rig) {
    const bool begin = L.rig_begin_pending;
    L.rig_begin_pending = false;
    return rig_run<RD, DE, GE, NSLOT>(p, begin, max_new);
  }
  for (int32_t it = 0; L.go && it < max_new; ++it) {
    const double iter_t0 = now_s();
    std::memset(&row, 0, sizeof(row));
    row.iteration = p->rows.back().iteration + 1;
    const bool fused = lm_fused(p);
    BA_CUDA_TRY(cudaMemcpyAsync(p->scal.p + S_RADIUS, &L.radius, sizeof(double), cudaMemcpyHostToDevice, p->st));
    if (fused) {
      if (L.need_linearize) { BA_TRY(fa_linearize(p, opt, false)); L.need_linearize = false; }  // same x, new radius
      BA_TRY(fa_step(p, opt));
    } else {
      BA_TRY((compute_step<RD, DE, GE, NSLOT>(p, opt)));
    }
    Z.num_linear_solves++;
    Z.num_cost_evaluations++;
    BA_TRY(fetch_scalars(p));
    row.linear_solver_iterations = p->solver == BA_RCS_PCG ? p->h_pcg_iters : 0;
    int status = *p->h_status;
    // a failed block factorisation on any rank invalidates the step everywhere (summed with the step scalars)
    if (p->world > 1) status = p->h_scal[S_STATUSD] != 0.0 ? 1 : 0;
    const double model_cost_change = -p->h_scal[S_MCC];
    const bool solve_ok = status == 0 && std::isfinite(model_cost_change);
    row.step_is_valid = solve_ok && model_cost_change > 0.0;
    if (!row.step_is_valid) {  // HandleInvalidStep
      if (++L.num_invalid >= opt.max_num_consecutive_invalid_steps) {
        Z.termination_type = BA_FAILURE; Z.termination_reason = BA_REASON_TOO_MANY_INVALID_STEPS;
        L.go = false;
        break;
      }
      L.radius = L.radius / L.decrease_factor; L.decrease_factor *= 2.0;
      L.need_linearize = true;
      row.cost = L.x_cost; row.cost_change = 0.0;
      row.gradient_max_norm = p->rows.back().gradient_max_norm; row.gradient_norm = p->rows.back().gradient_norm;
      L.go = lm_finalize(p, row, iter_t0);
      continue;
    }
    L.num_invalid = 0;
    const double cand_cost = 0.5 * p->h_scal[S_CAND];
    // ParameterToleranceReached
    const double x_norm = std::sqrt(p->h_scal[S_XE2] + p->h_scal[S_XF2]);
    row.step_norm = std::sqrt(p->h_scal[S_DE2] + p->h_scal[S_DF2]);
    if (row.step_norm <= opt.parameter_tolerance * (x_norm + opt.parameter_tolerance)) {
      Z.termination_type = BA_CONVERGENCE; Z.termination_reason = BA_REASON_PARAMETER_TOLERANCE;
      L.go = false;
      break;
    }
    // FunctionToleranceReached
    row.cost_change = L.x_cost - cand_cost;
    if (std::fabs(row.cost_change) <= opt.function_tolerance * L.x_cost) {
      Z.termination_type = BA_CONVERGENCE; Z.termination_reason = BA_REASON_FUNCTION_TOLERANCE;
      L.go = false;
      break;
    }
    row.relative_decrease = row.cost_change / model_cost_change;
    if (row.relative_decrease > opt.min_relative_decrease) {  // HandleSuccessfulStep
      p->xe.swap(p->xe_c);
      p->xf.swap(p->xf_c);
      L.radius = L.radius / std::max(1.0 / 3.0, 1.0 - std::pow(2.0 * row.relative_decrease - 1.0, 3));
      L.radius = std::min(opt.max_trust_region_radius, L.radius);
      L.decrease_factor = 2.0;
      if (fused) {  // the next step's radius is known: linearize and eliminate in the same pass
        BA_CUDA_TRY(cudaMemcpyAsync(p->scal.p + S_RADIUS, &L.radius, sizeof(double), cudaMemcpyHostToDevice, p->st));
        BA_TRY(fa_linearize(p, opt, false, row.iteration >= opt.max_num_iterations));   // the last row: nothing to eliminate for
      } else {
        BA_TRY((eval_gradient_and_jacobian<RD, DE, GE>(p, false, opt.jacobi_scaling != 0)));
      }
      Z.num_jacobian_evaluations++;
      BA_TRY(fetch_scalars(p));
      lm_read_gradient(p);
      row.step_is_successful = 1;
      row.cost = L.x_cost; row.gradient_max_norm = L.gmax; row.gradient_norm = L.gnorm;
    } else {  // HandleUnsuccessfulStep
      L.radius = L.radius / L.decrease_factor; L.decrease_factor *= 2.0;
      L.need_linearize = true;
      row.cost = cand_cost;
    }
    L.go = lm_finalize(p, row, iter_t0);
  }
  return BA_OK;
}

void lm_end(ba_cuda_problem* p, ba_cuda_summary* sum) {
  LmState& L = p->lm;
  ba_cuda_summary& Z = L.Z;
  Z.num_iterations = (int32_t)p->rows.size();
  Z.final_cost = L.x_cost;
  Z.total_time_s = now_s() - L.t_start;
  Z.ms_jacobian = p->fam_ms[F_JAC]; Z.ms_schur = p->fam_ms[F_SCHUR]; Z.ms_rcs_solve = p->fam_ms[F_SOLVE];
  Z.ms_update = p->fam_ms[F_UPDATE]; Z.ms_cost = p->fam_ms[F_COST]; Z.ms_collective = p->fam_ms[F_COLL];
  if (sum) *sum = Z;
}

// index validation on the device (a host loop over 30M observations costs more than the upload): first offender wins
__global__ void k_validate_a(int64_t n, const int32_t* __restrict__ cam, const int32_t* __restrict__ pt, int32_t n_cam, int64_t n_pt,
                             unsigned long long* __restrict__ first_bad) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (cam[i] < 0 || cam[i] >= n_cam || pt[i] < 0 || pt[i] >= n_pt) atomicMin(first_bad, (unsigned long long)i);
}
__global__ void k_count_active(const int64_t* __restrict__ ptr, int64_t n, unsigned long long* __restrict__ count) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int active = (i < n && ptr[i + 1] > ptr[i]) ? 1 : 0;
  const unsigned ballot = __ballot_sync(0xffffffffu, active);
  if ((threadIdx.x & 31) == 0 && ballot) atomicAdd(count, (unsigned long long)__popc(ballot));
}

// minimum of a flag over the ranks (no-op on one GPU)
int agree_min(ba_cuda_problem* p, int* flag) {
  if (p->world <= 1) return BA_OK;
  DVec<int32_t> d;
  const int32_t h = *flag;
  BA_TRY(d.upload(&h, 1, p->st));
  BA_TRY(allreduce(p, d.p, 1, 3 /* ncclMin */, kNcclInt32));
  int32_t out = 0;
  BA_CUDA_TRY(cudaMemcpyAsync(&out, d.p, sizeof(out), cudaMemcpyDeviceToHost, p->st));
  BA_CUDA_TRY(cudaStreamSynchronize(p->st));
  *flag = out;
  return BA_OK;
}

// number of active blocks (from the CSR pointers)
int count_active(ba_cuda_problem* p, const DVec<int64_t>& ptr, int64_t nblk, int64_t* out) {
  DVec<unsigned long long> cnt;
  BA_TRY(cnt.alloc_zero(1, p->st));
  k_count_active<<<grid_for(nblk, 256), 256, 0, p->st>>>(ptr.p, nblk, cnt.p);
  unsigned long long h = 0;
  BA_CUDA_TRY(cudaMemcpyAsync(&h, cnt.p, sizeof(h), cudaMemcpyDeviceToHost, p->st));
  BA_CUDA_TRY(cudaStreamSynchronize(p->st));
  *out = (int64_t)h;
  return BA_OK;
}

__global__ void k_active_flags(const int64_t* __restrict__ ptr, int64_t n, int32_t* __restrict__ flag) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i <= n) flag[i] = (i < n && ptr[i + 1] > ptr[i]) ? 1 : 0;
}
__global__ void k_widen(const int32_t* __restrict__ a, int64_t n, int64_t* __restrict__ b) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) b[i] = a[i];
}

// Which kept blocks take part in the problem is a GLOBAL property (a camera may have no observation in this
// rank's shard); the eliminated blocks are owned by exactly one rank, so only their count is summed.
int build_activity(ba_cuda_problem* p) {
  const Structure& S = p->S;
  if (S.host_f_act_ptr && p->world == 1) {   // host-built structure: the scan and the counts came with it
    p->f_act_ptr.borrow(const_cast<int64_t*>(S.host_f_act_ptr), S.nf + 1);
    p->n_active_f_global = S.host_n_active_f;
    p->n_active_e_global = S.host_n_active_e;
    p->nb_global = S.nb;
    return BA_OK;
  }
  DVec<int32_t> flag;
  DVec<int64_t> wide;
  BA_TRY(flag.alloc(S.nf + 1)); BA_TRY(wide.alloc(S.nf + 1)); BA_TRY(p->f_act_ptr.alloc(S.nf + 1));
  k_active_flags<<<grid_for(S.nf + 1, 256), 256, 0, p->st>>>(S.fobs_ptr.p, S.nf, flag.p);
  BA_TRY(allreduce(p, flag.p, S.nf + 1, kNcclMax, kNcclInt32));
  k_widen<<<grid_for(S.nf + 1, 256), 256, 0, p->st>>>(flag.p, S.nf + 1, wide.p);
  BA_TRY(cub_call([&](void* t, size_t& b) { return cub::DeviceScan::ExclusiveSum(t, b, wide.p, p->f_act_ptr.p, (int)(S.nf + 1), p->st); }));
  BA_CUDA_TRY(cudaMemcpyAsync(&p->n_active_f_global, p->f_act_ptr.p + S.nf, sizeof(int64_t), cudaMemcpyDeviceToHost, p->st));
  int64_t cnt[2] = {0, S.nb};
  BA_TRY(count_active(p, S.e_ptr, S.ne, &cnt[0]));  // synchronises
  if (p->world > 1) {
    DVec<int64_t> t;
    BA_TRY(t.upload(cnt, 2, p->st));
    BA_TRY(allreduce(p, t.p, 2, kNcclSum, kNcclInt64));
    BA_CUDA_TRY(cudaMemcpyAsync(cnt, t.p, sizeof(int64_t) * 2, cudaMemcpyDeviceToHost, p->st));
    BA_CUDA_TRY(cudaStreamSynchronize(p->st));
  }
  p->n_active_e_global = cnt[0];
  p->nb_global = cnt[1];
  return BA_OK;
}

// buffers every path needs
int alloc_workspace(ba_cuda_problem* p, int RD, int DE) {
  const Structure& S = p->S;
  const int64_t n = p->n_rcs();
  cudaStream_t st = p->st;
  BA_TRY(p->xf.alloc_zero(S.nf * 6, st)); BA_TRY(p->xf_c.alloc_zero(S.nf * 6, st));
  // + 2: the strip pass reads a tile's points as a 16-byte aligned slice (one double before / after the tile's own)
  BA_TRY(p->xe.alloc_zero(S.ne * DE + 2, st)); BA_TRY(p->xe_c.alloc_zero(S.ne * DE + 2, st));
  BA_TRY(p->sf.alloc(S.nf * 6)); BA_TRY(p->se.alloc(S.ne * DE + 2));
  k_fill<<<grid_for(S.nf * 6, 256), 256, 0, st>>>(p->sf.p, S.nf * 6, 1.0);
  k_fill<<<grid_for(S.ne * DE, 256), 256, 0, st>>>(p->se.p, S.ne * DE, 1.0);
  BA_TRY(p->tab_f.alloc(S.nf * TAB)); BA_TRY(p->tabc_f.alloc(S.nf * TAB));
  if (p->model == 1) { BA_TRY(p->tab_e.alloc(S.ne * TAB)); BA_TRY(p->tabc_e.alloc(S.ne * TAB)); }
  BA_TRY(p->Pacc.alloc((int64_t)S.ndest * 36)); BA_TRY(p->Qacc.alloc(p->model == 1 ? (int64_t)S.ndest * 36 : 0));
  p->Sd.release(); p->Sb.release(); p->solver = 0;
  BA_TRY(p->rhs.alloc(n)); BA_TRY(p->yf.alloc_zero(n, st)); BA_TRY(p->ye.alloc_zero(S.ne * DE, st));
  const int64_t maxgrid = std::max<int64_t>({(int64_t)grid_for(S.nb * 4, 128), (int64_t)grid_for(S.ne * DE, 256), (int64_t)grid_for(S.nf * 6, 256)}) + 1;
  BA_TRY(p->bp0.alloc(maxgrid)); BA_TRY(p->bp1.alloc(maxgrid));
  BA_TRY(p->scal.alloc_zero(S_COUNT, st)); BA_TRY(p->status.alloc_zero(1, st));
  p->generic_ws = false;
  BA_CUDA_TRY(cudaStreamSynchronize(st));
  BA_CUDA_TRY(cudaGetLastError());
  return BA_OK;
}

// the materialised residual / Jacobian / Schur buffers of the generic pipeline (Model B always; Model A only when the
// fused path is not used, and for the ba_cuda_eval test hook)
// the materialised residual / Jacobian arrays alone (what ba_cuda_eval fills)
int ensure_jacobian_buffers(ba_cuda_problem* p) {
  const Structure& S = p->S;
  const int RD = p->model == 0 ? 2 : 8, DE = p->model == 0 ? 3 : 6;
  if (p->RES.n == (size_t)(S.nb * RD) && p->JE.n == (size_t)(S.nb * RD * DE) && p->JF0.n == (size_t)(S.nb * RD * 6)) return BA_OK;
  BA_TRY(p->RES.alloc(S.nb * RD)); BA_TRY(p->JE.alloc(S.nb * RD * DE)); BA_TRY(p->JF0.alloc(S.nb * RD * 6));
  BA_TRY(p->JF1.alloc(p->model == 1 ? S.nb * RD * 6 : 0));
  return BA_OK;
}

int ensure_generic_workspace(ba_cuda_problem* p) {
  if (p->generic_ws) return BA_OK;
  BA_TRY(ensure_pair_lists(p->S, p->st));   // Model A builds only the destination set up front (ba_structure.cuh)
  const Structure& S = p->S;
  const int DE = p->model == 0 ? 3 : 6;
  BA_TRY(ensure_jacobian_buffers(p));
  BA_TRY(p->ME.alloc(S.ne * (DE * (DE + 1) / 2 + DE))); BA_TRY(p->HG.alloc(S.nf * NV_F + 2 + kMaxWorld));
  BA_TRY(p->Wt.alloc(p->model == 1 ? S.ninc * 36 : 0));
  BA_TRY(p->Lb.alloc(S.ne * DE * DE)); BA_TRY(p->zb.alloc(S.ne * DE));
  BA_TRY(p->Yt.alloc(S.ninc * DE * 6)); BA_TRY(p->vb.alloc(S.ninc * 6));
  BA_TRY(p->part_fobs.alloc((int64_t)S.ch_fobs.n * NV_F)); BA_TRY(p->part_finc.alloc((int64_t)S.ch_finc.n * 6));
  BA_TRY(p->part_pairs.alloc((int64_t)S.ch_pairs.n * 36));
  BA_TRY(p->part_dobs.alloc(p->model == 1 ? (int64_t)S.ch_dobs.n * 36 : 0));
  p->generic_ws = true;
  return BA_OK;
}

__global__ void k_gather_uv(const double* __restrict__ src, const int32_t* __restrict__ perm, int64_t n, int width, double* __restrict__ dst) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= n * width) return;
  dst[t] = src[(int64_t)perm[t / width] * width + t % width];
}


// ---- K5 / post-BA outputs ---------------------------------------------------------------
// cv::Rodrigues(rvec -> R) as used by BAManager::Write (bundle_adjustment_manager.cpp:121) and by
// cv::projectPoints inside ReprojectionCheck::Reproject (reprojection_check.cpp:69).
__global__ void k_rodrigues_cv(const double* __restrict__ rt6, int n, double* __restrict__ R9, double* __restrict__ inv12) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double rx = rt6[6 * i], ry = rt6[6 * i + 1], rz = rt6[6 * i + 2];
  const double theta = sqrt(rx * rx + ry * ry + rz * rz);
  double R[9];
  if (theta < DBL_EPSILON) {
#pragma unroll
    for (int q = 0; q < 9; ++q) R[q] = (q % 4 == 0) ? 1.0 : 0.0;
  } else {
    const double c = cos(theta), s = sin(theta), c1 = 1.0 - c, it = 1.0 / theta;
    const double k0 = rx * it, k1 = ry * it, k2 = rz * it;
    R[0] = c + c1 * k0 * k0;      R[1] = c1 * k0 * k1 - s * k2; R[2] = c1 * k0 * k2 + s * k1;
    R[3] = c1 * k0 * k1 + s * k2; R[4] = c + c1 * k1 * k1;      R[5] = c1 * k1 * k2 - s * k0;
    R[6] = c1 * k0 * k2 - s * k1; R[7] = c1 * k1 * k2 + s * k0; R[8] = c + c1 * k2 * k2;
  }
#pragma unroll
  for (int q = 0; q < 9; ++q) R9[9 * i + q] = R[q];
  if (inv12) {  // rows of [R^T | -R^T t], bundle_adjustment_manager.cpp:135-149
    const double t0 = rt6[6 * i + 3], t1 = rt6[6 * i + 4], t2 = rt6[6 * i + 5];
#pragma unroll
    for (int row = 0; row < 3; ++row) {
      double* o = inv12 + 12 * i + 4 * row;
      o[0] = R[row]; o[1] = R[3 + row]; o[2] = R[6 + row];
      o[3] = -(R[row] * t0 + R[3 + row] * t1 + R[6 + row] * t2);
    }
  }
}

// ---- the numeric part of the correspondence stage (SURVEY 8 f1, Main_Calibration/correspondencer.cpp) ----------------
__device__ __forceinline__ void rodrigues_cv_dev(const double* r, double* R) {   // cv::Rodrigues, vector -> matrix
  const double theta = sqrt(r[0] * r[0] + r[1] * r[1] + r[2] * r[2]);
  if (theta < DBL_EPSILON) {
#pragma unroll
    for (int q = 0; q < 9; ++q) R[q] = (q % 4 == 0) ? 1.0 : 0.0;
    return;
  }
  const double c = cos(theta), s = sin(theta), c1 = 1.0 - c, it = 1.0 / theta;
  const double k0 = r[0] * it, k1 = r[1] * it, k2 = r[2] * it;
  R[0] = c + c1 * k0 * k0;      R[1] = c1 * k0 * k1 - s * k2; R[2] = c1 * k0 * k2 + s * k1;
  R[3] = c1 * k0 * k1 + s * k2; R[4] = c + c1 * k1 * k1;      R[5] = c1 * k1 * k2 - s * k0;
  R[6] = c1 * k0 * k2 - s * k1; R[7] = c1 * k1 * k2 + s * k0; R[8] = c + c1 * k2 * k2;
}
__device__ __forceinline__ void rodrigues_inv_cv_dev(const double* R, double* r) {   // cv::Rodrigues, matrix -> vector
  double rx = R[7] - R[5], ry = R[2] - R[6], rz = R[3] - R[1];
  const double s = sqrt((rx * rx + ry * ry + rz * rz) * 0.25);
  const double c = fmin(fmax((R[0] + R[4] + R[8] - 1.0) * 0.5, -1.0), 1.0);
  double theta = acos(c);
  if (s < 1e-5) {
    if (c > 0.0) { r[0] = r[1] = r[2] = 0.0; return; }
    double t = (R[0] + 1.0) * 0.5;
    rx = sqrt(fmax(t, 0.0));
    t = (R[4] + 1.0) * 0.5;
    ry = sqrt(fmax(t, 0.0)) * (R[1] < 0.0 ? -1.0 : 1.0);
    t = (R[8] + 1.0) * 0.5;
    rz = sqrt(fmax(t, 0.0)) * (R[2] < 0.0 ? -1.0 : 1.0);
    if (fabs(rx) < fabs(ry) && fabs(rx) < fabs(rz) && (R[5] > 0.0) != (ry * rz > 0.0)) rz = -rz;
    theta /= sqrt(rx * rx + ry * ry + rz * rz);
    r[0] = rx * theta; r[1] = ry * theta; r[2] = rz * theta;
  } else {
    const double vth = theta / (2.0 * s);
    r[0] = rx * vth; r[1] = ry * vth; r[2] = rz * vth;
  }
}
// Correspondencer::GetCornersInCameraWorld (correspondencer.cpp:5-39): t -+ E +- F with E, F = half side x the first two columns of R
__global__ void k_marker_corners(int64_t n, const double* __restrict__ rt6, double half, double* __restrict__ out) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  double R[9];
  rodrigues_cv_dev(rt6 + 6 * i, R);
  const double E[3] = {R[0] * half, R[3] * half, R[6] * half}, F[3] = {R[1] * half, R[4] * half, R[7] * half};
  const double* t = rt6 + 6 * i + 3;
  double* o = out + 12 * i;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    o[k] = t[k] + (-E[k] + F[k]);       // top left
    o[3 + k] = t[k] + (E[k] + F[k]);    // top right
    o[6 + k] = t[k] + (E[k] - F[k]);    // bottom right
    o[9 + k] = t[k] + (-E[k] - F[k]);   // bottom left
  }
}
// pose composition of correspondencer.cpp:100-149: out = a o b (R = Ra Rb, t = Ra tb + ta; :141-146) or, invert_b,
// out = a o b^-1 (R = Ra Rb^T, t = Ra Rb^T (-tb) + ta; :118-121)
__global__ void k_compose_poses(int64_t n, const double* __restrict__ a6, const double* __restrict__ b6, int invert_b, double* __restrict__ out6) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  double Ra[9], Rb[9], R[9];
  rodrigues_cv_dev(a6 + 6 * i, Ra);
  rodrigues_cv_dev(b6 + 6 * i, Rb);
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      double v = 0.0;
#pragma unroll
      for (int k = 0; k < 3; ++k) v += Ra[3 * r + k] * (invert_b ? Rb[3 * c + k] : Rb[3 * k + c]);
      R[3 * r + c] = v;
    }
  const double* ta = a6 + 6 * i + 3;
  const double* tb = b6 + 6 * i + 3;
  double* o = out6 + 6 * i;
  rodrigues_inv_cv_dev(R, o);
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    double v = 0.0;
    if (invert_b) { for (int k = 0; k < 3; ++k) v += R[3 * r + k] * (-tb[k]); }
    else { for (int k = 0; k < 3; ++k) v += Ra[3 * r + k] * tb[k]; }
    o[3 + r] = v + ta[r];
  }
}

// cv::projectPoints with zero distortion, then ((x^ - x)^2 + (y^ - y)^2) / 2 (reprojection_check.cpp:81)
__global__ void __launch_bounds__(256)
k_project_error(int64_t n, const double* __restrict__ xyz, const int32_t* __restrict__ cam, const double* __restrict__ R9,
                const double* __restrict__ t3, const double* __restrict__ K4, const float* __restrict__ img,
                double* __restrict__ rep, double* __restrict__ partial) {
  __shared__ double sm[32];
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  double e = 0.0;
  if (i < n) {
    const int c = cam[i];
    const double* R = R9 + 9 * c;
    const double* t = t3 + 3 * c;
    const double X = xyz[3 * i], Y = xyz[3 * i + 1], Z = xyz[3 * i + 2];
    const double x = R[0] * X + R[1] * Y + R[2] * Z + t[0];
    const double y = R[3] * X + R[4] * Y + R[5] * Z + t[1];
    const double z = R[6] * X + R[7] * Y + R[8] * Z + t[2];
    const double iz = z != 0.0 ? 1.0 / z : 1.0;
    const double u = (x * iz) * K4[4 * c] + K4[4 * c + 2], v = (y * iz) * K4[4 * c + 1] + K4[4 * c + 3];
    if (rep) { rep[2 * i] = u; rep[2 * i + 1] = v; }
    const double dx = (double)img[2 * i] - u, dy = (double)img[2 * i + 1] - v;
    e = (dx * dx + dy * dy) / 2;
  }
  e = block_sum(e, sm);
  if (threadIdx.x == 0) partial[blockIdx.x] = e;
}

// BALProblem::getPoint3dCoordinates (bundle_adjustment.cpp:89-130): marker corner -> base-marker frame -> base camera
__global__ void k_corners_b(int64_t nb, const int32_t* __restrict__ perm, const int32_t* __restrict__ ob_e,
                            const int32_t* __restrict__ ob_marker, int32_t n_cam, const double* __restrict__ tab_f,
                            const double* __restrict__ tab_e, double half, double* __restrict__ corners) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= nb * 4) return;
  const int64_t b = t >> 2;
  const int corner = (int)(t & 3);
  const double* Tm = tab_f + TAB * (int64_t)(n_cam + ob_marker[b]);
  const double* Tt = tab_e + TAB * (int64_t)ob_e[b];
  const double q0[3] = {(corner == 0 || corner == 3) ? -half : half, (corner < 2) ? half : -half, 0.0};
  double r[3], p1[3];
  mat3_vec(Tm, q0, r);
  p1[0] = r[0] + Tm[18]; p1[1] = r[1] + Tm[19]; p1[2] = r[2] + Tm[20];
  mat3_vec(Tt, p1, r);
  double* o = corners + ((int64_t)perm[b] * 4 + corner) * 3;
  o[0] = r[0] + Tt[18]; o[1] = r[1] + Tt[19]; o[2] = r[2] + Tt[20];
}

// ---- ba_cuda_solve_batch: K solves of one structure in one launch, one CTA each (ba_rig.cuh, k_rig_lm_batch) ---------
// instance i's observation j (structure order) is row i * n + perm[j] of the caller's k x n rows: with this map one
// k_gather_uv launch over all k * n rows puts every instance into structure order
__global__ void k_batch_perm(const int32_t* __restrict__ perm, int64_t n, int64_t k, int32_t* __restrict__ out) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t < n * k) out[t] = (int32_t)((t / n) * n + perm[t % n]);
}

// the arrays of one instance's slice of the batch workspace
enum RigBatchArray {
  RB_XE = 0, RB_XF, RB_XE_C, RB_XF_C, RB_SE, RB_SF, RB_TAB_F, RB_TAB_E, RB_TABC_F, RB_TABC_E,
  RB_RES, RB_JE, RB_JF0, RB_JF1, RB_ME, RB_HG, RB_WT, RB_QACC, RB_LB, RB_ZB, RB_YT, RB_VB, RB_PACC, RB_VSUM, RB_YF, RB_YE, RB_COUNT
};
// caller parameter layout <-> the instance slices: (caller offset, slice array, slice offset, count) per segment
struct ParamSegment { int64_t src, dst_arr, dst, count; };
int param_segments(const ba_cuda_problem* p, ParamSegment seg[3]) {
  const int64_t C = p->n_cam;
  if (p->model == 0) {
    seg[0] = {0, RB_XF, 0, 6 * C};
    seg[1] = {6 * C, RB_XE, 0, 3 * p->n_pt};
    return 2;
  }
  const int64_t T = p->n_time, M = p->n_marker;
  seg[0] = {0, RB_XF, 0, 6 * C};
  seg[1] = {6 * C, RB_XE, 0, 6 * T};
  seg[2] = {6 * (C + T), RB_XF, 6 * C, 6 * M};
  return 3;
}

template <int RD, int DE, int GE, int NSLOT>
int rig_batch_run(ba_cuda_problem* p, const ba_cuda_options& opt, int32_t k, double* params, const double* observations,
                  ba_cuda_summary* summaries, ba_cuda_iteration* rows, int32_t rows_cap) {
  const double t_start = now_s();
  const Structure& S = p->S;
  const cudaStream_t st = p->st;
  const int n = (int)p->n_rcs();
  constexpr int NU = DE * (DE + 1) / 2;
  constexpr bool MB = RD == 8;
  // one region per instance; every array starts on a 32-byte boundary (J, uv and obs8 are read as double2)
  int64_t len[RB_COUNT] = {};
  len[RB_XE] = len[RB_XE_C] = len[RB_SE] = len[RB_ZB] = len[RB_YE] = S.ne * DE;
  len[RB_XF] = len[RB_XF_C] = len[RB_SF] = len[RB_VSUM] = S.nf * 6;
  len[RB_YF] = n;
  len[RB_TAB_F] = len[RB_TABC_F] = S.nf * TAB;
  len[RB_TAB_E] = len[RB_TABC_E] = MB ? S.ne * TAB : 0;
  len[RB_RES] = S.nb * RD; len[RB_JE] = S.nb * RD * DE; len[RB_JF0] = S.nb * RD * 6; len[RB_JF1] = MB ? S.nb * RD * 6 : 0;
  len[RB_ME] = S.ne * (NU + DE); len[RB_HG] = S.nf * NV_F; len[RB_WT] = MB ? S.ninc * 36 : 0; len[RB_QACC] = MB ? (int64_t)S.ndest * 36 : 0;
  len[RB_LB] = S.ne * DE * DE; len[RB_YT] = S.ninc * DE * 6; len[RB_VB] = S.ninc * 6; len[RB_PACC] = (int64_t)S.ndest * 36;
  int64_t off[RB_COUNT];
  RigBatch B;
  std::memset(&B, 0, sizeof(B));
  for (int j = 0; j < RB_COUNT; ++j) { off[j] = B.stride; B.stride += (len[j] + 3) / 4 * 4; }
  // rows one launch can record per instance: a solve records at most max_num_iterations + 1
  const int64_t R = std::max<int64_t>(1, std::min<int64_t>(RIG_ROWS_CAP, (int64_t)opt.max_num_iterations + 1));
  B.rows_stride = R;
  DVec<double> ws, obs_raw, obs;
  DVec<RigState> states;
  DVec<ba_cuda_iteration> drows;
  DVec<int32_t> perm;
  BA_TRY(ws.alloc_zero((size_t)k * B.stride, st));   // zeroed: the blocks no step touches read as they would in a fresh problem
  BA_TRY(states.alloc(k));
  BA_TRY(drows.alloc((size_t)k * R));
  const size_t D = sizeof(double);
  ParamSegment seg[3];
  const int nseg = param_segments(p, seg);
  for (int s = 0; s < nseg; ++s)
    if (seg[s].count)
      BA_CUDA_TRY(cudaMemcpy2DAsync(ws.p + off[seg[s].dst_arr] + seg[s].dst, D * B.stride, params + seg[s].src, D * p->n_params,
                                    D * seg[s].count, k, cudaMemcpyHostToDevice, st));
  if (observations) {
    const int width = MB ? 8 : 2;
    const int64_t rows_all = (int64_t)k * S.nb;
    BA_TRY(obs_raw.upload(observations, (size_t)rows_all * width, st));
    BA_TRY(perm.alloc(rows_all)); BA_TRY(obs.alloc((size_t)rows_all * width));
    BA_LAUNCH(p, KT_MISC, k_batch_perm, grid_for(rows_all, 256), 256, 0, S.perm.p, S.nb, (int64_t)k, perm.p);
    BA_LAUNCH(p, KT_MISC, k_gather_uv, grid_for(rows_all * width, 256), 256, 0, obs_raw.p, perm.p, rows_all, width, obs.p);
    BA_CUDA_TRY(cudaGetLastError());
    B.obs = obs.p; B.obs_stride = S.nb * width;
  }
  // what rig_run passes
  RigParams P;
  std::memset(&P, 0, sizeof(P));
  P.nb = S.nb; P.ne = S.ne; P.nf = S.nf; P.ninc = S.ninc; P.ndest = S.ndest; P.n = n; P.ld = n | 1;
  P.ob_e = S.ob_e.p; P.ob_f0 = S.ob_f0.p; P.ob_f1 = S.ob_f1.p; P.ob_cam = p->ob_cam.p; P.e_ptr = S.e_ptr.p;
  P.inc_e = S.inc_e; P.inc_f = S.inc_f; P.einc_ptr = S.einc_ptr; P.incobs_ptr = S.incobs_ptr.p; P.incobs = S.incobs.p;
  P.finc_ptr = S.finc_ptr.p; P.fobs_ptr = S.fobs_ptr.p; P.finc = S.finc.p; P.fobs = S.fobs.p;
  P.dest_fa = S.dest_fa.p; P.dest_fb = S.dest_fb.p; P.dpair_ptr = S.dpair_ptr.p; P.pairs = S.pairs.p;
  P.dobs_ptr = S.dobs_ptr.p; P.dobs = S.dobs.p; P.f_act_ptr = p->f_act_ptr.p;
  P.uv = p->uv.p; P.obs8 = p->obs8.p; P.intr_f = p->intr_f.p; P.half_side = p->half_side;
  // instance 0's arrays; the kernel moves them B.stride doubles further per instance
  double** const arr[RB_COUNT] = {&P.xe, &P.xf, &P.xe_c, &P.xf_c, &P.se, &P.sf, &P.tab_f, &P.tab_e, &P.tabc_f, &P.tabc_e,
                                  &P.RES, &P.JE, &P.JF0, &P.JF1, &P.ME, &P.HG, &P.Wt, &P.Qacc, &P.Lb, &P.zb, &P.Yt, &P.vb,
                                  &P.Pacc, &P.vsum, &P.yf, &P.ye};
  for (int j = 0; j < RB_COUNT; ++j) *arr[j] = ws.p + off[j];
  P.state = states.p; P.rows = drows.p;
  P.opt = opt; P.loss = LossSpec{opt.loss_function, opt.loss_scale};
  P.init.radius = opt.initial_trust_region_radius; P.init.decrease_factor = 2.0; P.init.go = 1;
  const size_t smem = rig_smem_bytes(n);
  BA_CUDA_TRY(cudaFuncSetAttribute(k_rig_lm_batch<RD, DE, GE, NSLOT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rig_smem_bytes(RIG_MAX_N)));
  std::vector<RigState> hst(k);
  std::vector<int32_t> base(k, 0);
  std::vector<double> cost0(k, 0.0);
  std::vector<ba_cuda_iteration> hrows;
  bool running = true;
  for (int64_t launch = 0; running; ++launch) {   // a solve longer than RIG_ROWS_CAP rows continues in the next launch, as in rig_run
    P.begin = launch == 0 ? 1 : 0;
    P.max_new = RIG_ROWS_CAP - P.begin;
    BA_LAUNCH(p, KT_RIG_BATCH, (k_rig_lm_batch<RD, DE, GE, NSLOT>), (unsigned)k, RIG_THREADS, smem, P, B);
    BA_CUDA_TRY(cudaGetLastError());
    BA_CUDA_TRY(cudaMemcpyAsync(hst.data(), states.p, sizeof(RigState) * k, cudaMemcpyDeviceToHost, st));
    if (launch == 0)   // row 0's cost is the summary's initial_cost
      BA_CUDA_TRY(cudaMemcpy2DAsync(cost0.data(), D, reinterpret_cast<const char*>(drows.p) + offsetof(ba_cuda_iteration, cost),
                                    sizeof(ba_cuda_iteration) * R, D, k, cudaMemcpyDeviceToHost, st));
    // the rows of this launch start at row launch * RIG_ROWS_CAP of every instance still running: fetch those the caller keeps
    const int64_t first = launch * RIG_ROWS_CAP;
    const int64_t cnt = rows ? std::min<int64_t>(R, rows_cap - first) : 0;
    if (cnt > 0) {
      hrows.resize((size_t)k * cnt);
      BA_CUDA_TRY(cudaMemcpy2DAsync(hrows.data(), sizeof(ba_cuda_iteration) * cnt, drows.p, sizeof(ba_cuda_iteration) * R,
                                    sizeof(ba_cuda_iteration) * cnt, k, cudaMemcpyDeviceToHost, st));
    }
    BA_CUDA_TRY(cudaStreamSynchronize(st));
    fam_collect(p);
    running = false;
    for (int32_t i = 0; i < k; ++i) {
      const int64_t fresh = hst[i].n_rows - base[i];
      for (int64_t r = 0; r < std::min(fresh, cnt); ++r)
        if (base[i] + r < rows_cap) rows[(int64_t)i * rows_cap + base[i] + r] = hrows[(size_t)i * cnt + r];
      base[i] = hst[i].n_rows;
      running = running || hst[i].go != 0;
    }
  }
  for (int s = 0; s < nseg; ++s)
    if (seg[s].count)
      BA_CUDA_TRY(cudaMemcpy2DAsync(params + seg[s].src, D * p->n_params, ws.p + off[seg[s].dst_arr] + seg[s].dst, D * B.stride,
                                    D * seg[s].count, k, cudaMemcpyDeviceToHost, st));
  BA_CUDA_TRY(cudaStreamSynchronize(st));
  if (summaries) {   // rig_run + lm_end + ba_cuda_solve_end, per instance
    const double total = now_s() - t_start;
    for (int32_t i = 0; i < k; ++i) {
      const RigState& s = hst[i];
      ba_cuda_summary& Z = summaries[i];
      std::memset(&Z, 0, sizeof(Z));
      Z.termination_type = s.term_type; Z.termination_reason = s.term_reason;
      Z.num_iterations = s.n_rows;
      Z.num_successful_steps = s.n_success; Z.num_unsuccessful_steps = s.n_unsuccess;
      Z.rcs_solver_used = BA_RCS_DENSE_CHOLESKY;
      Z.rcs_dim = (int32_t)(6 * p->n_active_f_global);
      Z.num_jacobian_evaluations = s.n_jac; Z.num_cost_evaluations = s.n_solves; Z.num_linear_solves = s.n_solves;
      Z.num_residuals = p->nb_global * RD;
      Z.num_free_parameters = p->n_active_e_global * DE + p->n_active_f_global * 6;
      Z.initial_cost = s.n_rows > 0 ? cost0[i] : s.x_cost;
      Z.final_cost = s.x_cost;
      Z.total_time_s = total;
      Z.path_used = BA_PATH_RIG;
    }
  }
  return BA_OK;
}

void reset_problem(ba_cuda_problem* p) {
  p->model = -1;
  p->params_set = false;
  p->rows.clear();
  p->xf_s.release(); p->xe_s.release();
  p->R.~RcsPattern();
  new (&p->R) RcsPattern();
  p->FA.~FusedA();
  new (&p->FA) FusedA();
  p->SA.~StripA();
  new (&p->SA) StripA();
  p->SX.~SparseExchange();
  new (&p->SX) SparseExchange();
  p->use_fused = false; p->use_strip = false; p->generic_ws = false;
  p->lm.began = false;
  p->S.~Structure();
  new (&p->S) Structure();
}

// ba_cuda_covariance after its checks: Model B, one rank, n <= kDenseAutoMaxN, p->loss set (ba_cov.cuh has the algebra).
int covariance_impl(ba_cuda_problem* p, const ba_cuda_options& opt, double min_pivot_ratio, double* cov_kept, double* cov_frames,
                    double* smallest_pivot_ratio) {
  const Structure& S = p->S;
  const int n = (int)p->n_rcs();
  cudaStream_t st = p->st;
  BA_TRY(prepare_solver(p, opt));   // opt.rcs_solver is BA_RCS_DENSE_CHOLESKY: Sd exists
  BA_TRY(ensure_generic_workspace(p));
  BA_TRY((eval_gradient_and_jacobian<8, 6, 32>(p, true, true)));
  BA_LAUNCH(p, KT_MISC, k_cov_unit_unused<6>, grid_for(S.ne + S.nf, 256), 256, 0, S.ne, S.e_ptr.p, p->ME.p, S.nf, p->f_act_ptr.p, p->HG.p);
  const double no_lm_diagonal_radius = INFINITY;   // D^2 = clamp(diag) / radius = 0 exactly
  BA_CUDA_TRY(cudaMemcpyAsync(p->scal.p + S_RADIUS, &no_lm_diagonal_radius, sizeof(double), cudaMemcpyHostToDevice, st));
  BA_TRY((schur_complement<8, 6>(p, opt)));
  DVec<double> diag, X, Sig, Ck, Cf;
  BA_TRY(diag.alloc(n + 1)); BA_TRY(X.alloc_zero((size_t)n * n, st)); BA_TRY(Sig.alloc((size_t)n * n)); BA_TRY(Ck.alloc((size_t)n * n));
  BA_TRY(Cf.alloc((size_t)S.ne * 36));
  BA_LAUNCH(p, KT_MISC, k_cov_save_diag, grid_for(n, 256), 256, 0, n, p->Sd.p, diag.p);
  {
    LaunchScope scope(p, KT_RCS);
    BA_TRY(launch_chol_blocked(p->cholb, n, p->Sd.p, p->rhs.p, p->yf.p, p->status.p, p->device, st));
  }
  BA_LAUNCH(p, KT_MISC, k_cov_pivot_ratio, 1, 1024, 0, n, p->Sd.p, diag.p, p->f_act_ptr.p, diag.p + n);
  BA_LAUNCH(p, KT_COV_LINV, k_cov_linv, (n + CV_NB - 1) / CV_NB, CV_THREADS, 0, n, p->Sd.p, X.p);
  const int nt = (n + CV_TB - 1) / CV_TB;
  BA_LAUNCH(p, KT_COV_INV, k_cov_inverse, nt * (nt + 1) / 2, CV_THREADS, 0, n, X.p, p->sf.p, p->f_act_ptr.p, Sig.p, Ck.p);
  fam_end(p, F_SOLVE);
  if (S.ne > 0) {
    const size_t smem = cov_frames_smem(6, S.nf);
    if (smem > 48 * 1024) BA_CUDA_TRY(cudaFuncSetAttribute(k_cov_frames<6>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    BA_LAUNCH(p, KT_COV_FRAMES, k_cov_frames<6>, (unsigned)S.ne, CV_THREADS, smem, S.ne, S.e_ptr.p, S.einc_ptr, S.inc_f, p->Yt.p, p->Lb.p,
              p->se.p, Sig.p, n, Cf.p);
  }
  BA_CUDA_TRY(cudaGetLastError());
  double ratio = 0.0;
  BA_CUDA_TRY(cudaMemcpyAsync(&ratio, diag.p + n, sizeof(double), cudaMemcpyDeviceToHost, st));
  BA_CUDA_TRY(cudaMemcpyAsync(p->h_status, p->status.p, sizeof(int), cudaMemcpyDeviceToHost, st));
  BA_CUDA_TRY(cudaStreamSynchronize(st));
  fam_collect(p);
  const int status = *p->h_status;
  if (status & 2) ratio = 0.0;   // the factorisation stopped at a pivot <= 0
  if (smallest_pivot_ratio) *smallest_pivot_ratio = ratio;
  if (status & 1) return fail(BA_ERR_RANK_DEFICIENT, "ba_cuda_covariance: E^T E of a frame pose is not positive definite");
  const double thr = min_pivot_ratio > 0.0 ? min_pivot_ratio : 1e-12;
  if (!(ratio > thr))
    return fail(BA_ERR_RANK_DEFICIENT, "ba_cuda_covariance: the reduced system is rank deficient (smallest pivot / largest diagonal entry "
                "%.3e <= %.3e)", ratio, thr);
  if (cov_kept) BA_CUDA_TRY(cudaMemcpyAsync(cov_kept, Ck.p, sizeof(double) * (size_t)n * n, cudaMemcpyDeviceToHost, st));
  if (cov_frames && S.ne > 0) BA_CUDA_TRY(cudaMemcpyAsync(cov_frames, Cf.p, sizeof(double) * (size_t)S.ne * 36, cudaMemcpyDeviceToHost, st));
  BA_CUDA_TRY(cudaStreamSynchronize(st));
  return BA_OK;
}

}  // namespace

// =======================================================================================
// C ABI
// =======================================================================================
extern "C" {

void ba_cuda_options_init(ba_cuda_options* o) {
  if (!o) return;
  std::memset(o, 0, sizeof(*o));
  o->max_num_iterations = 50; o->max_num_consecutive_invalid_steps = 5; o->jacobi_scaling = 1;
  o->rcs_solver = BA_RCS_AUTO; o->pcg_max_iterations = 500; o->pcg_min_iterations = 0;
  o->pcg_residual_reset_period = 10; o->minimizer_progress_to_stdout = 0;
  o->initial_trust_region_radius = 1e4; o->max_trust_region_radius = 1e16; o->min_trust_region_radius = 1e-32;
  o->min_relative_decrease = 1e-3; o->min_lm_diagonal = 1e-6; o->max_lm_diagonal = 1e32;
  o->function_tolerance = 1e-6; o->gradient_tolerance = 1e-10; o->parameter_tolerance = 1e-8;
  o->pcg_eta = 1e-1; o->pcg_r_tolerance = -1.0;
  o->loss_function = BA_LOSS_NONE; o->loss_scale = 1.0;
}

const char* ba_cuda_last_error(void) { return err_buf(); }

int ba_cuda_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

int ba_cuda_create(ba_cuda_problem** out, int device_id) {
  if (!out) return fail(BA_ERR_INVALID_ARGUMENT, "out is NULL");
  *out = nullptr;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
    cudaGetLastError();
    return fail(BA_ERR_NO_DEVICE, "no CUDA device: this library has no CPU fallback");
  }
  if (device_id < 0 || device_id >= n) return fail(BA_ERR_INVALID_ARGUMENT, "device %d out of range [0,%d)", device_id, n);
  BA_CUDA_TRY(cudaSetDevice(device_id));
  ba_cuda_problem* p = new ba_cuda_problem();
  p->device = device_id;
  ++g_live_problems;   // ba_cuda_destroy counts it down again
  const int rc = [&]() -> int {
    BA_CUDA_TRY(cudaStreamCreateWithFlags(&p->own_st, cudaStreamNonBlocking));
    p->st = p->own_st;
    for (int f = 0; f < F_COUNT; ++f) { BA_CUDA_TRY(cudaEventCreate(&p->ev[f][0])); BA_CUDA_TRY(cudaEventCreate(&p->ev[f][1])); }
    BA_CUDA_TRY(cudaEventCreate(&p->k0)); BA_CUDA_TRY(cudaEventCreate(&p->k1));
    BA_CUDA_TRY(cudaStreamCreateWithFlags(&p->copy_st, cudaStreamNonBlocking));
    BA_CUDA_TRY(cudaEventCreateWithFlags(&p->copy_go, cudaEventDisableTiming));
    BA_CUDA_TRY(cudaEventCreateWithFlags(&p->copy_done, cudaEventDisableTiming));
    BA_CUDA_TRY(cudaMallocHost((void**)&p->h_scal, sizeof(double) * S_COUNT));
    BA_CUDA_TRY(cudaMallocHost((void**)&p->h_status, sizeof(int)));
    return BA_OK;
  }();
  if (rc != BA_OK) { ba_cuda_destroy(p); return rc; }   // destroy copes with whatever was created so far
  *out = p;
  return BA_OK;
}

void ba_cuda_release_cached_memory(void) { DevCache::get().trim(); }

void ba_cuda_destroy(ba_cuda_problem* p) {
  if (!p) return;
  cudaSetDevice(p->device);
  if (p->st) cudaStreamSynchronize(p->st);
  if (p->comm && nccl().ok()) nccl().CommDestroy(p->comm);
  for (int f = 0; f < F_COUNT; ++f) { if (p->ev[f][0]) cudaEventDestroy(p->ev[f][0]); if (p->ev[f][1]) cudaEventDestroy(p->ev[f][1]); }
  if (p->k0) cudaEventDestroy(p->k0);
  if (p->k1) cudaEventDestroy(p->k1);
  if (p->copy_st) { cudaStreamSynchronize(p->copy_st); cudaStreamDestroy(p->copy_st); }
  if (p->copy_go) cudaEventDestroy(p->copy_go);
  if (p->copy_done) cudaEventDestroy(p->copy_done);
  if (p->h_scal) cudaFreeHost(p->h_scal);
  if (p->h_status) cudaFreeHost(p->h_status);
  if (p->h_rig) cudaFreeHost(p->h_rig);
  for (cudaEvent_t e : p->ev_pool) cudaEventDestroy(e);
  cudaStream_t st = p->own_st, used = p->st;
  DevCache::current_stream() = used;
  delete p;
  DevCache::get().mark_clean(used);  // synchronised above
  if (st) cudaStreamDestroy(st);
  if (--g_live_problems == 0) DevCache::get().trim();  // the cache only lives as long as some problem does
}

int ba_cuda_comm_unique_id(uint8_t id[BA_CUDA_UNIQUE_ID_BYTES]) {
  if (!nccl().ok()) return fail(BA_ERR_NCCL, "libnccl.so.2 could not be loaded");
  NcclUniqueId u;
  const int rc = nccl().GetUniqueId(&u);
  if (rc != 0) return fail(BA_ERR_NCCL, "ncclGetUniqueId failed (%d)", rc);
  std::memcpy(id, u.internal, BA_CUDA_UNIQUE_ID_BYTES);
  return BA_OK;
}

int ba_cuda_comm_init(ba_cuda_problem* p, int rank, int world_size, const uint8_t id[BA_CUDA_UNIQUE_ID_BYTES]) {
  if (!p || world_size < 1 || rank < 0 || rank >= world_size) return fail(BA_ERR_INVALID_ARGUMENT, "bad rank/world");
  if (world_size > kMaxWorld) return fail(BA_ERR_UNSUPPORTED, "at most %d ranks", kMaxWorld);
  BA_TRY(use_device(p));
  p->rank = rank; p->world = world_size;
  if (world_size == 1) return BA_OK;
  if (!nccl().ok()) return fail(BA_ERR_NCCL, "libnccl.so.2 could not be loaded");
  NcclUniqueId u;
  std::memcpy(u.internal, id, BA_CUDA_UNIQUE_ID_BYTES);
  const int rc = nccl().CommInitRank(&p->comm, world_size, u, rank);
  if (rc != 0) return fail(BA_ERR_NCCL, "ncclCommInitRank failed: %s", nccl().GetErrorString ? nccl().GetErrorString(rc) : "?");
  return BA_OK;
}

int ba_cuda_shard_blocks(int64_t n_blocks, const int64_t* weight, int world_size, int64_t* range_begin) {
  if (n_blocks < 0 || world_size < 1 || !range_begin) return fail(BA_ERR_INVALID_ARGUMENT, "bad shard arguments");
  long double total = 0;
  for (int64_t i = 0; i < n_blocks; ++i) total += weight ? (long double)weight[i] : 1.0L;
  range_begin[0] = 0;
  int64_t i = 0;
  long double acc = 0;
  for (int r = 1; r < world_size; ++r) {
    const long double target = total * r / world_size;
    while (i < n_blocks && acc + (weight ? weight[i] : 1) * 0.5L <= target) { acc += weight ? weight[i] : 1; ++i; }
    range_begin[r] = i;
  }
  range_begin[world_size] = n_blocks;
  return BA_OK;
}

static int set_model_a_impl(ba_cuda_problem* p, int32_t n_cam, int64_t n_pt, int64_t n_obs, const int32_t* cam_idx,
                            const int32_t* pt_idx, const double* obs_xy, const double* intr, int32_t intr_stride) {
  if (!p || n_cam < 1 || n_pt < 0 || n_obs < 0 || (n_obs > 0 && (!cam_idx || !pt_idx || !obs_xy)) || !intr ||
      (intr_stride != 0 && intr_stride != 4))
    return fail(BA_ERR_INVALID_ARGUMENT, "ba_cuda_set_model_a: bad arguments");
  if (n_pt >= (int64_t)INT32_MAX) return fail(BA_ERR_UNSUPPORTED, "too many points for one GPU shard");
  PhaseTimer T;
  BA_TRY(use_device(p));
  reset_problem(p);
  p->building = true;
  T.lap("reset");
  p->n_cam = n_cam; p->n_pt = n_pt; p->n_time = 0; p->n_marker = 0;
  p->n_params = 6 * (int64_t)n_cam + 3 * n_pt;
  // Rig sizes (Test1 / Test2 of the reference: 16..200 observations, one or two cameras): the solve will run in the one-CTA
  // kernel (ba_rig.cuh) or, if the caller asks otherwise, in the generic pipeline; neither needs the tile / strip structures
  // of the fused passes.  The lists are made on the host and uploaded in one copy (ba_structure.cuh, build_structure_host).
  const int64_t host_build_max = env_int("BA_HOST_BUILD_MAX", 0, 1 << 20, 4096);
  if (n_obs > 0 && n_obs <= host_build_max && 2 * n_obs <= RIG_MAX_ROWS && 6 * (int64_t)n_cam <= RIG_MAX_N && p->world == 1 &&
      env_int("BA_RIG", 0, 1, 1) != 0) {
    for (int64_t i = 0; i < n_obs; ++i)
      if (cam_idx[i] < 0 || cam_idx[i] >= n_cam || pt_idx[i] < 0 || pt_idx[i] >= n_pt)
        return fail(BA_ERR_INVALID_ARGUMENT, "observation %lld references camera %d / point %d out of range", (long long)i, cam_idx[i], pt_idx[i]);
    BA_TRY(build_structure_host(p->S, n_obs, n_pt, n_cam, pt_idx, cam_idx, nullptr, p->st));
    T.lap("host build_structure");
    p->model = 0;
    {
      DVec<double> tmp;
      BA_TRY(tmp.upload(obs_xy, 2 * (size_t)n_obs, p->st));
      BA_TRY(p->uv.alloc(n_obs));
      k_gather_uv<<<grid_for(2 * n_obs, 256), 256, 0, p->st>>>(tmp.p, p->S.perm.p, n_obs, 2, reinterpret_cast<double*>(p->uv.p));
      std::vector<double> K(4 * (size_t)n_cam);
      for (int32_t c = 0; c < n_cam; ++c)
        for (int q = 0; q < 4; ++q) K[4 * c + q] = intr[(size_t)intr_stride * c + q];
      BA_TRY(p->intr_f.upload(K.data(), K.size(), p->st));
      BA_CUDA_TRY(cudaStreamSynchronize(p->st));
    }
    p->h_perm.clear();
    BA_TRY(alloc_workspace(p, 2, 3));
    p->use_fused = false; p->use_strip = false;
    BA_TRY(ensure_generic_workspace(p));
    T.lap("uploads + workspace");
    return build_activity(p);
  }
  // The image points (16 B per observation, two thirds of the upload) travel on a second stream while the index
  // structure is built from the indices: the copy is queued behind the index uploads (so those reach the device
  // first) and joined again just before the gather into sorted order.
  DVec<double> obs_tmp;
  BA_TRY(obs_tmp.alloc(2 * (size_t)n_obs));
  {
    const int rc = build_structure(p->S, n_obs, n_pt, n_cam, pt_idx, cam_idx, nullptr, p->st, [&](const int32_t* d_pt, const int32_t* d_cam) {
      BA_CUDA_TRY(cudaEventRecord(p->copy_go, p->st));
      BA_CUDA_TRY(cudaStreamWaitEvent(p->copy_st, p->copy_go, 0));
      if (n_obs > 0) BA_CUDA_TRY(cudaMemcpyAsync(obs_tmp.p, obs_xy, sizeof(double) * 2 * n_obs, cudaMemcpyHostToDevice, p->copy_st));
      BA_CUDA_TRY(cudaEventRecord(p->copy_done, p->copy_st));
      // the uploaded index arrays are checked on the device before anything is built from them
      DVec<unsigned long long> bad;
      BA_TRY(bad.alloc(1));
      BA_CUDA_TRY(cudaMemsetAsync(bad.p, 0xff, sizeof(unsigned long long), p->st));
      k_validate_a<<<grid_for(n_obs, 256), 256, 0, p->st>>>(n_obs, d_cam, d_pt, n_cam, n_pt, bad.p);
      unsigned long long h = 0;
      BA_CUDA_TRY(cudaMemcpyAsync(&h, bad.p, sizeof(h), cudaMemcpyDeviceToHost, p->st));
      BA_CUDA_TRY(cudaStreamSynchronize(p->st));
      if (h != ~0ull)
        return fail(BA_ERR_INVALID_ARGUMENT, "observation %lld references camera %d / point %d out of range", (long long)h, cam_idx[h], pt_idx[h]);
      return (int)BA_OK;
    });
    if (rc != BA_OK) { cudaStreamSynchronize(p->copy_st); reset_problem(p); return rc; }
  }
  T.lap("upload + validate + build_structure");
  p->model = 0;
  // observations in sorted order, intrinsics per f-block
  {
    BA_CUDA_TRY(cudaStreamWaitEvent(p->st, p->copy_done, 0));
    BA_TRY(p->uv.alloc(n_obs));
    k_gather_uv<<<grid_for(2 * n_obs, 256), 256, 0, p->st>>>(obs_tmp.p, p->S.perm.p, n_obs, 2, reinterpret_cast<double*>(p->uv.p));
    std::vector<double> K(4 * (size_t)n_cam);
    for (int32_t c = 0; c < n_cam; ++c)
      for (int q = 0; q < 4; ++q) K[4 * c + q] = intr[(size_t)intr_stride * c + q];
    BA_TRY(p->intr_f.upload(K.data(), K.size(), p->st));
    BA_CUDA_TRY(cudaStreamSynchronize(p->st));
  }
  T.lap("observations upload");
  p->h_perm.clear();  // fetched on demand by ba_cuda_eval
  BA_TRY(alloc_workspace(p, 2, 3));
  T.lap("alloc_workspace");
  {  // fused two-pass pipeline when every point has <= FA_KMAX observations, else the generic one; pass 1 on strips of
     // tiles when the cameras of a strip fit (ba_strip_a.cuh), else on single tiles (ba_fused_a.cuh)
    // Multi-GPU: every rank must run the same pipeline (the collectives carry its buffers: a shard on strips and a shard
    // on tiles would disagree on their layout), so the choice is the minimum over the ranks of what each shard fits.
    int rc = build_strip_a(p->SA, p->FA, p->S, p->uv.p, p->st);
    if (rc != BA_OK && rc != BA_ERR_UNSUPPORTED) return rc;
    int ok = rc == BA_OK ? 1 : 0;
    BA_TRY(agree_min(p, &ok));
    p->use_strip = ok != 0;
    if (!p->use_strip) {
      p->SA.~StripA();
      new (&p->SA) StripA();
      rc = build_fused_a(p->FA, p->S, p->st);
      if (rc != BA_OK && rc != BA_ERR_UNSUPPORTED) return rc;
      ok = rc == BA_OK ? 1 : 0;
      BA_TRY(agree_min(p, &ok));
      if (!ok) { p->FA.~FusedA(); new (&p->FA) FusedA(); }
    }
    p->use_fused = ok != 0;
    if (p->use_fused) {
      BA_TRY(p->fa_part.alloc((size_t)7 * p->FA.n_tiles));
    } else {
      static std::atomic<bool> warned{false};
      if (n_obs > 0 && !warned.exchange(true))
        std::fprintf(stderr, "[ba_cuda] Model A problem does not fit the fused pipeline (a point with more than %d observations); "
                             "using the generic materialised-Jacobian pipeline (ba_cuda_summary.path_used = BA_PATH_GENERIC)\n", FA_KMAX);
      BA_TRY(ensure_generic_workspace(p));
    }
  }
  T.lap("build_fused_a");
  const int rc = build_activity(p);
  T.lap("build_activity");
  return rc;
}

static int set_model_b_impl(ba_cuda_problem* p, int32_t n_cam, int32_t n_time, int32_t n_marker, int64_t n_mobs,
                            const int32_t* time_idx, const int32_t* cam_idx, const int32_t* marker_idx, const double* obs8,
                            const double* intr4_per_cam, double marker_side, int32_t fix_cam0, int32_t fix_marker0) {
  if (!p || n_cam < 1 || n_time < 0 || n_marker < 1 || n_mobs < 0 || (n_mobs > 0 && (!time_idx || !cam_idx || !marker_idx || !obs8)) ||
      !intr4_per_cam)
    return fail(BA_ERR_INVALID_ARGUMENT, "ba_cuda_set_model_b: bad arguments");
  if (!fix_cam0) return fail(BA_ERR_UNSUPPORTED, "camera 0 is never a parameter block in the reference (fix_cam0 must be 1)");
  std::vector<int32_t> f0(n_mobs), f1(n_mobs);
  for (int64_t i = 0; i < n_mobs; ++i) {
    if (time_idx[i] < 0 || time_idx[i] >= n_time || cam_idx[i] < 0 || cam_idx[i] >= n_cam || marker_idx[i] < 0 || marker_idx[i] >= n_marker)
      return fail(BA_ERR_INVALID_ARGUMENT, "marker observation %lld has an index out of range", (long long)i);
    f0[i] = cam_idx[i] == 0 ? -1 : cam_idx[i];                                    // bundle_adjustment_manager.cpp:26
    f1[i] = (fix_marker0 && marker_idx[i] == 0) ? -1 : n_cam + marker_idx[i];     // bundle_adjustment_manager.cpp:28,58
  }
  BA_TRY(use_device(p));
  reset_problem(p);
  p->building = true;
  p->n_cam = n_cam; p->n_time = n_time; p->n_marker = n_marker; p->n_pt = 0;
  p->n_params = 6 * ((int64_t)n_cam + n_time + n_marker);
  p->half_side = marker_side / 2;
  const int64_t nf = (int64_t)n_cam + n_marker;
  PhaseTimer T;
  // rig sizes: the lists are made on the host and uploaded in one copy (ba_structure.cuh, build_structure_host)
  const int64_t host_build_max = env_int("BA_HOST_BUILD_MAX", 0, 1 << 20, 4096);
  if (n_mobs > 0 && n_mobs <= host_build_max && p->world == 1)
    BA_TRY(build_structure_host(p->S, n_mobs, n_time, nf, time_idx, f0.data(), f1.data(), p->st));
  else
    BA_TRY(build_structure(p->S, n_mobs, n_time, nf, time_idx, f0.data(), f1.data(), p->st,
                           [](const int32_t*, const int32_t*) { return (int)BA_OK; }));  // validated above, on the host
  T.lap("build_structure");
  p->model = 1;
  {
    DVec<double> tmp;
    DVec<int32_t> cam_in, mk_in;
    BA_TRY(tmp.upload(obs8, 8 * n_mobs, p->st));
    BA_TRY(cam_in.upload(cam_idx, n_mobs, p->st));
    BA_TRY(mk_in.upload(marker_idx, n_mobs, p->st));
    BA_TRY(p->obs8.alloc(8 * n_mobs)); BA_TRY(p->ob_cam.alloc(n_mobs)); BA_TRY(p->ob_marker.alloc(n_mobs));
    k_gather_uv<<<grid_for(8 * n_mobs, 256), 256, 0, p->st>>>(tmp.p, p->S.perm.p, n_mobs, 8, p->obs8.p);
    k_gather_i32<<<grid_for(n_mobs, 256), 256, 0, p->st>>>(p->ob_cam.p, cam_in.p, p->S.perm.p, n_mobs);
    k_gather_i32<<<grid_for(n_mobs, 256), 256, 0, p->st>>>(p->ob_marker.p, mk_in.p, p->S.perm.p, n_mobs);
    std::vector<double> K(4 * (size_t)nf, 0.0);
    std::memcpy(K.data(), intr4_per_cam, sizeof(double) * 4 * n_cam);
    BA_TRY(p->intr_f.upload(K.data(), K.size(), p->st));
    BA_CUDA_TRY(cudaStreamSynchronize(p->st));
  }
  T.lap("observations upload");
  p->h_perm.clear();
  BA_TRY(alloc_workspace(p, 8, 6));
  T.lap("alloc_workspace");
  p->use_fused = false;
  BA_TRY(ensure_generic_workspace(p));
  T.lap("generic workspace");
  const int rc_act = build_activity(p);
  T.lap("build_activity");
  return rc_act;
}

// A failure after the old model was dropped (allocation, NCCL, an index out of range found on the device) must not leave
// p->model set over unallocated buffers: the problem goes back to "no model".
static int finish_set_model(ba_cuda_problem* p, int rc) {
  if (!p) return rc;
  if (rc != BA_OK && p->building) {
    if (p->st) cudaStreamSynchronize(p->st);
    if (p->copy_st) cudaStreamSynchronize(p->copy_st);
    cudaGetLastError();
    reset_problem(p);
  }
  p->building = false;
  return rc;
}
int ba_cuda_set_model_a(ba_cuda_problem* p, int32_t n_cam, int64_t n_pt, int64_t n_obs, const int32_t* cam_idx,
                        const int32_t* pt_idx, const double* obs_xy, const double* intr, int32_t intr_stride) {
  return finish_set_model(p, set_model_a_impl(p, n_cam, n_pt, n_obs, cam_idx, pt_idx, obs_xy, intr, intr_stride));
}
int ba_cuda_set_model_b(ba_cuda_problem* p, int32_t n_cam, int32_t n_time, int32_t n_marker, int64_t n_mobs,
                        const int32_t* time_idx, const int32_t* cam_idx, const int32_t* marker_idx, const double* obs8,
                        const double* intr4_per_cam, double marker_side, int32_t fix_cam0, int32_t fix_marker0) {
  return finish_set_model(p, set_model_b_impl(p, n_cam, n_time, n_marker, n_mobs, time_idx, cam_idx, marker_idx, obs8, intr4_per_cam,
                                              marker_side, fix_cam0, fix_marker0));
}

int64_t ba_cuda_num_parameters(const ba_cuda_problem* p) { return p ? p->n_params : 0; }

int ba_cuda_set_parameters(ba_cuda_problem* p, const double* params, int64_t n) {
  if (!p || !params) return fail(BA_ERR_INVALID_ARGUMENT, "NULL argument");
  if (p->model < 0) return fail(BA_ERR_STATE, "set_model_* must be called first");
  if (n != p->n_params) return fail(BA_ERR_INVALID_ARGUMENT, "expected %lld parameters, got %lld", (long long)p->n_params, (long long)n);
  BA_TRY(use_device(p));
  const size_t D = sizeof(double);
  if (p->model == 0) {
    BA_CUDA_TRY(cudaMemcpyAsync(p->xf.p, params, D * 6 * p->n_cam, cudaMemcpyHostToDevice, p->st));
    if (p->n_pt) BA_CUDA_TRY(cudaMemcpyAsync(p->xe.p, params + 6 * (int64_t)p->n_cam, D * 3 * p->n_pt, cudaMemcpyHostToDevice, p->st));
  } else {
    const int64_t C = p->n_cam, T = p->n_time, M = p->n_marker;
    BA_CUDA_TRY(cudaMemcpyAsync(p->xf.p, params, D * 6 * C, cudaMemcpyHostToDevice, p->st));
    if (T) BA_CUDA_TRY(cudaMemcpyAsync(p->xe.p, params + 6 * C, D * 6 * T, cudaMemcpyHostToDevice, p->st));
    BA_CUDA_TRY(cudaMemcpyAsync(p->xf.p + 6 * C, params + 6 * (C + T), D * 6 * M, cudaMemcpyHostToDevice, p->st));
  }
  BA_CUDA_TRY(cudaStreamSynchronize(p->st));
  p->params_set = true;
  return BA_OK;
}

int ba_cuda_get_parameters(ba_cuda_problem* p, double* params, int64_t n) {
  if (!p || !params) return fail(BA_ERR_INVALID_ARGUMENT, "NULL argument");
  if (p->model < 0 || !p->params_set) return fail(BA_ERR_STATE, "no parameters have been set");
  if (n != p->n_params) return fail(BA_ERR_INVALID_ARGUMENT, "expected %lld parameters, got %lld", (long long)p->n_params, (long long)n);
  BA_TRY(use_device(p));
  const size_t D = sizeof(double);
  if (p->model == 0) {
    BA_CUDA_TRY(cudaMemcpyAsync(params, p->xf.p, D * 6 * p->n_cam, cudaMemcpyDeviceToHost, p->st));
    if (p->n_pt) BA_CUDA_TRY(cudaMemcpyAsync(params + 6 * (int64_t)p->n_cam, p->xe.p, D * 3 * p->n_pt, cudaMemcpyDeviceToHost, p->st));
  } else {
    const int64_t C = p->n_cam, T = p->n_time, M = p->n_marker;
    BA_CUDA_TRY(cudaMemcpyAsync(params, p->xf.p, D * 6 * C, cudaMemcpyDeviceToHost, p->st));
    if (T) BA_CUDA_TRY(cudaMemcpyAsync(params + 6 * C, p->xe.p, D * 6 * T, cudaMemcpyDeviceToHost, p->st));
    BA_CUDA_TRY(cudaMemcpyAsync(params + 6 * (C + T), p->xf.p + 6 * C, D * 6 * M, cudaMemcpyDeviceToHost, p->st));
  }
  BA_CUDA_TRY(cudaStreamSynchronize(p->st));
  return BA_OK;
}

int ba_cuda_save_parameters(ba_cuda_problem* p) {
  if (!p) return fail(BA_ERR_INVALID_ARGUMENT, "NULL problem");
  if (p->model < 0 || !p->params_set) return fail(BA_ERR_STATE, "no parameters have been set");
  BA_TRY(use_device(p));
  if (p->xf_s.n != p->xf.n) BA_TRY(p->xf_s.alloc(p->xf.n));
  if (p->xe_s.n != p->xe.n) BA_TRY(p->xe_s.alloc(p->xe.n));
  BA_CUDA_TRY(cudaMemcpyAsync(p->xf_s.p, p->xf.p, p->xf.bytes(), cudaMemcpyDeviceToDevice, p->st));
  BA_CUDA_TRY(cudaMemcpyAsync(p->xe_s.p, p->xe.p, p->xe.bytes(), cudaMemcpyDeviceToDevice, p->st));
  return BA_OK;
}

int ba_cuda_restore_parameters(ba_cuda_problem* p) {
  if (!p) return fail(BA_ERR_INVALID_ARGUMENT, "NULL problem");
  if (p->model < 0 || p->xf_s.n != p->xf.n || p->xe_s.n != p->xe.n || p->xf_s.p == nullptr)
    return fail(BA_ERR_STATE, "ba_cuda_save_parameters has not been called for this problem");
  BA_TRY(use_device(p));
  BA_CUDA_TRY(cudaMemcpyAsync(p->xf.p, p->xf_s.p, p->xf.bytes(), cudaMemcpyDeviceToDevice, p->st));
  BA_CUDA_TRY(cudaMemcpyAsync(p->xe.p, p->xe_s.p, p->xe.bytes(), cudaMemcpyDeviceToDevice, p->st));
  return BA_OK;
}

int ba_cuda_solve_begin(ba_cuda_problem* p, const ba_cuda_options* options) {
  if (!p) return fail(BA_ERR_INVALID_ARGUMENT, "NULL problem");
  if (p->model < 0 || !p->params_set) return fail(BA_ERR_STATE, "set_model_* and set_parameters must be called before solve");
  BA_TRY(use_device(p));
  ba_cuda_options opt;
  if (options) opt = *options; else ba_cuda_options_init(&opt);
  if (opt.loss_function < BA_LOSS_NONE || opt.loss_function > BA_LOSS_CAUCHY || (opt.loss_function != BA_LOSS_NONE && !(opt.loss_scale > 0.0)))
    return fail(BA_ERR_INVALID_ARGUMENT, "loss_function %d with scale %g", opt.loss_function, opt.loss_scale);
  p->loss = LossSpec{opt.loss_function, opt.loss_scale};
  BA_TRY(prepare_solver(p, opt));
  if (p->model == 0 && (opt.force_generic_path || !p->use_fused)) BA_TRY(ensure_generic_workspace(p));
  return p->model == 0 ? lm_begin<2, 3, 1, 1>(p, opt) : lm_begin<8, 6, 32, 2>(p, opt);
}

int ba_cuda_solve_iterate(ba_cuda_problem* p, int32_t max_new_iterations, int32_t* finished) {
  if (!p) return fail(BA_ERR_INVALID_ARGUMENT, "NULL problem");
  if (!p->lm.began) return fail(BA_ERR_STATE, "ba_cuda_solve_begin must be called first");
  BA_TRY(use_device(p));
  const int rc = p->model == 0 ? lm_iterate<2, 3, 1, 1>(p, max_new_iterations) : lm_iterate<8, 6, 32, 2>(p, max_new_iterations);
  if (finished) *finished = p->lm.go ? 0 : 1;
  return rc;
}

int ba_cuda_solve_end(ba_cuda_problem* p, ba_cuda_summary* summary) {
  if (!p) return fail(BA_ERR_INVALID_ARGUMENT, "NULL problem");
  if (!p->lm.began) return fail(BA_ERR_STATE, "ba_cuda_solve_begin must be called first");
  BA_TRY(use_device(p));
  lm_end(p, summary);
  p->loss = LossSpec{0, 1.0};   // ba_cuda_eval / ba_cuda_reprojection_error report plain residuals
  if (summary) {
    const int64_t ae = p->n_active_e_global, af = p->n_active_f_global;
    summary->num_free_parameters = ae * (p->model == 0 ? 3 : 6) + af * 6;
    summary->rcs_dim = (int32_t)(6 * af);
  }
  return BA_OK;
}

int ba_cuda_solve(ba_cuda_problem* p, const ba_cuda_options* options, ba_cuda_summary* summary) {
  if (p) p->one_shot = true;
  const int rc_begin = ba_cuda_solve_begin(p, options);
  if (p) p->one_shot = false;
  BA_TRY(rc_begin);
  int32_t finished = 0;
  BA_TRY(ba_cuda_solve_iterate(p, INT32_MAX, &finished));
  return ba_cuda_solve_end(p, summary);
}

int ba_cuda_solve_batch(ba_cuda_problem* p, const ba_cuda_options* options, int32_t k, double* params, const double* observations,
                        ba_cuda_summary* summaries, ba_cuda_iteration* rows, int32_t rows_cap) {
  if (!p) return fail(BA_ERR_INVALID_ARGUMENT, "NULL problem");
  if (p->model < 0) return fail(BA_ERR_STATE, "set_model_* must be called before ba_cuda_solve_batch");
  if (p->lm.began && p->lm.go) return fail(BA_ERR_STATE, "ba_cuda_solve_batch between ba_cuda_solve_begin and the end of the solve");
  if (k < 1 || !params || (rows && rows_cap < 1))
    return fail(BA_ERR_INVALID_ARGUMENT, "ba_cuda_solve_batch: k = %d, params %s, rows_cap = %d", k, params ? "set" : "NULL", rows_cap);
  ba_cuda_options opt;
  if (options) opt = *options; else ba_cuda_options_init(&opt);
  if (opt.loss_function < BA_LOSS_NONE || opt.loss_function > BA_LOSS_CAUCHY || (opt.loss_function != BA_LOSS_NONE && !(opt.loss_scale > 0.0)))
    return fail(BA_ERR_INVALID_ARGUMENT, "loss_function %d with scale %g", opt.loss_function, opt.loss_scale);
  int solver = opt.rcs_solver;   // as prepare_solver resolves it
  if (solver == BA_RCS_AUTO) solver = p->n_rcs() <= kDenseAutoMaxN ? BA_RCS_DENSE_CHOLESKY : BA_RCS_PCG;
  if (solver != BA_RCS_DENSE_CHOLESKY && solver != BA_RCS_PCG) return fail(BA_ERR_INVALID_ARGUMENT, "unknown rcs_solver %d", opt.rcs_solver);
  if (!rig_fits(p, solver, opt.force_generic_path != 0, RIG_MAX_ROWS))
    return fail(BA_ERR_UNSUPPORTED, "ba_cuda_solve_batch takes rig-size problems only (reduced system %lld <= %d, residual rows %lld <= %lld, "
                "dense rcs_solver, force_generic_path = 0, one GPU): got %lld, %lld, rcs_solver %d, force_generic_path %d, world size %d",
                (long long)p->n_rcs(), RIG_MAX_N, (long long)(p->S.nb * (p->model == 0 ? 2 : 8)), (long long)RIG_MAX_ROWS,
                (long long)p->n_rcs(), (long long)(p->S.nb * (p->model == 0 ? 2 : 8)), solver, opt.force_generic_path, p->world);
  if (observations && (int64_t)k * p->S.nb > (int64_t)INT32_MAX)
    return fail(BA_ERR_UNSUPPORTED, "ba_cuda_solve_batch: %d instances of %lld observations are too many for one call", k, (long long)p->S.nb);
  BA_TRY(use_device(p));
  BA_TRY(ensure_generic_workspace(p));   // the pair lists of the structure
  const bool profile = p->profile;
  p->profile = opt.profile_kernels != 0;
  const int rc = p->model == 0 ? rig_batch_run<2, 3, 1, 1>(p, opt, k, params, observations, summaries, rows, rows_cap)
                               : rig_batch_run<8, 6, 32, 2>(p, opt, k, params, observations, summaries, rows, rows_cap);
  p->profile = profile;
  if (rc != BA_OK) {   // the per-instance buffers are gone; the problem's own were never touched
    cudaStreamSynchronize(p->st);
    p->pending.clear();
    p->ev_next = 0;
  }
  return rc;
}

int ba_cuda_set_stream(ba_cuda_problem* p, void* cuda_stream) {
  if (!p) return fail(BA_ERR_INVALID_ARGUMENT, "NULL problem");
  BA_TRY(use_device(p));
  BA_CUDA_TRY(cudaStreamSynchronize(p->st));
  DevCache::get().mark_clean(p->st);
  p->st = cuda_stream ? (cudaStream_t)cuda_stream : p->own_st;
  DevCache::current_stream() = p->st;
  return BA_OK;
}

// compulsory HBM traffic of one launch of each kernel on the current problem (DESIGN.md, "kernels and rooflines")
static double algorithmic_bytes(const ba_cuda_problem* p, int kt) {
  const Structure& S = p->S;
  const double nb = (double)S.nb, ne = (double)S.ne, nf = (double)S.nf, ninc = (double)S.ninc;
  const bool A = p->model == 0;
  switch (kt) {
    case KT_JAC:  // idx + obs in, r + J out, parameter blocks once
      return A ? nb * 184.0 + nf * 80.0 + ne * 24.0 : nb * 1292.0 + (nf + ne) * 48.0;
    case KT_COST: return A ? nb * 24.0 + nf * 80.0 + ne * 24.0 : nb * 76.0 + (nf + ne) * 48.0;
    case KT_FOBS: return A ? nb * (96.0 + 16.0 + 4.0) + nf * 216.0 : nb * 2.0 * (384.0 + 64.0 + 4.0) + nf * 216.0;
    case KT_EM: return A ? nb * 64.0 + ne * 72.0 : nb * 448.0 + ne * 216.0;
    case KT_ECHOL: return A ? ne * (72.0 + 72.0 + 24.0) : ne * (216.0 + 288.0 + 48.0);
    case KT_INCY: return A ? nb * (144.0 + 144.0 + 48.0) + ne * 96.0 : ninc * (288.0 + 288.0 + 48.0) + ne * 336.0;
    case KT_FINC: return ninc * 52.0 + nf * 48.0;
    case KT_PAIRS: return (double)S.npairs * (8.0 + (A ? 288.0 : 576.0)) + (double)S.ndest * 288.0;
    case KT_BACKSUB: return A ? ninc * (144.0 + 4.0) + ne * 120.0 : ninc * (288.0 + 4.0) + ne * 384.0;
    case KT_MODELCOST: return A ? nb * (160.0 + 8.0) + ne * 24.0 : nb * (1216.0 + 12.0) + ne * 48.0;
    // fused Model A passes, accounted with the bytes of the materialised layout they replace (SURVEY.md 8d):
    // pass 1 = K1 (184 B/obs) + K2 (168 B/obs read, 72 B/point, 336 B/camera, 288 B/stored block written)
    case KT_FA_P1: return nb * (184.0 + 168.0) + ne * (24.0 + 72.0) + nf * (80.0 + 336.0) + (double)S.ndest * 288.0;
    // the light variants of pass 1 (Jacobi scaling at iteration 0; cost + gradient after the last step): K1 + the F^T F / F^T r
    // and E^T E / E^T r accumulations, nothing eliminated
    case KT_FA_P1L: return nb * (184.0 + 116.0 + 64.0) + ne * (24.0 + 72.0) + nf * (80.0 + 216.0);
    // pass 2 = K4 (152 B/obs + 72 B/point read, 24 B/point + 48 B/camera written) + cost-only evaluation (24 B/obs)
    case KT_FA_P2: return nb * (152.0 + 24.0) + ne * (72.0 + 24.0 + 24.0) + nf * (48.0 + 80.0);
    // covariance (ba_cov.cuh), n = 6 nf: L^-1 reads L and writes X (lower triangles); X^T X reads X and writes two full n x n
    // matrices; the frame blocks read Yt, Lb, se and S^-1 once (every later read of S^-1 is an L2 hit) and write 36 per frame
    case KT_COV_LINV: return 8.0 * (36.0 * nf * nf);
    case KT_COV_INV: return 20.0 * (36.0 * nf * nf);
    case KT_COV_FRAMES: return ninc * 288.0 + ne * (288.0 + 48.0 + 288.0) + 8.0 * (36.0 * nf * nf);
    default: return 0.0;
  }
}

int ba_cuda_get_kernel_stats(ba_cuda_problem* p, ba_cuda_kernel_stat* stats, int cap) {
  if (!p) return fail(BA_ERR_INVALID_ARGUMENT, "NULL problem");
  int n = 0;
  for (int k = 0; k < KT_COUNT; ++k) {
    if (p->kt_launches[k] == 0) continue;
    if (stats && n < cap) {
      std::memset(&stats[n], 0, sizeof(stats[n]));
      std::snprintf(stats[n].name, sizeof(stats[n].name), "%s", kKtName[k]);
      stats[n].launches = p->kt_launches[k];
      stats[n].total_ms = p->kt_ms[k];
      stats[n].algorithmic_bytes_per_launch = p->model >= 0 ? algorithmic_bytes(p, k) : 0.0;
    }
    ++n;
  }
  return n;
}

int64_t ba_cuda_num_launches(const ba_cuda_problem* p) {
  int64_t n = 0;
  if (p) for (int k = 0; k < KT_COUNT; ++k) n += p->kt_launches[k];
  return n;
}

void ba_cuda_reset_stats(ba_cuda_problem* p) {
  if (!p) return;
  for (int k = 0; k < KT_COUNT; ++k) { p->kt_launches[k] = 0; p->kt_ms[k] = 0.0; }
}

int ba_cuda_get_iterations(ba_cuda_problem* p, ba_cuda_iteration* rows, int cap) {
  if (!p) return fail(BA_ERR_INVALID_ARGUMENT, "NULL problem");
  const int n = (int)p->rows.size();
  if (rows) for (int i = 0; i < std::min(n, cap); ++i) rows[i] = p->rows[i];
  return n;
}

int ba_cuda_eval(ba_cuda_problem* p, double* cost, double* residuals, double* jac) {
  if (!p) return fail(BA_ERR_INVALID_ARGUMENT, "NULL problem");
  if (p->model < 0 || !p->params_set) return fail(BA_ERR_STATE, "set_model_* and set_parameters must be called before eval");
  // eval resets the Jacobi scaling and overwrites the residual / Jacobian buffers the open solve works on
  if (p->lm.began && p->lm.go) return fail(BA_ERR_STATE, "ba_cuda_eval between ba_cuda_solve_begin and the end of the solve");
  BA_TRY(use_device(p));
  const Structure& S = p->S;
  const int RD = p->model == 0 ? 2 : 8, DE = p->model == 0 ? 3 : 6;
  BA_TRY(ensure_jacobian_buffers(p));
  BA_LAUNCH(p, KT_MISC, k_fill, grid_for(S.ne * DE, 256), 256, 0, p->se.p, S.ne * DE, 1.0);
  BA_LAUNCH(p, KT_MISC, k_fill, grid_for(S.nf * 6, 256), 256, 0, p->sf.p, S.nf * 6, 1.0);
  BA_TRY(build_tables(p, false));  // warm the tables outside the timed kernel
  BA_CUDA_TRY(cudaEventRecord(p->k0, p->st));
  BA_TRY(run_jacobian(p));
  BA_CUDA_TRY(cudaEventRecord(p->k1, p->st));
  BA_TRY(allreduce(p, p->scal.p + S_COST, 1, kNcclSum));
  BA_TRY(fetch_scalars(p));
  BA_CUDA_TRY(cudaEventElapsedTime(&p->last_kernel_ms, p->k0, p->k1));
  if (cost) *cost = 0.5 * p->h_scal[S_COST];
  if ((residuals || jac) && (int64_t)p->h_perm.size() != S.nb) {
    p->h_perm.resize(S.nb);
    BA_CUDA_TRY(cudaMemcpy(p->h_perm.data(), S.perm.p, sizeof(int32_t) * S.nb, cudaMemcpyDeviceToHost));
  }
  if (residuals) {
    std::vector<double> h(S.nb * RD);
    BA_CUDA_TRY(cudaMemcpy(h.data(), p->RES.p, sizeof(double) * h.size(), cudaMemcpyDeviceToHost));
    for (int64_t b = 0; b < S.nb; ++b) std::memcpy(residuals + (int64_t)p->h_perm[b] * RD, &h[b * RD], sizeof(double) * RD);
  }
  if (jac) {
    std::vector<double> he(S.nb * RD * DE), h0(S.nb * RD * 6), h1;
    BA_CUDA_TRY(cudaMemcpy(he.data(), p->JE.p, sizeof(double) * he.size(), cudaMemcpyDeviceToHost));
    BA_CUDA_TRY(cudaMemcpy(h0.data(), p->JF0.p, sizeof(double) * h0.size(), cudaMemcpyDeviceToHost));
    if (p->model == 1) { h1.resize(S.nb * RD * 6); BA_CUDA_TRY(cudaMemcpy(h1.data(), p->JF1.p, sizeof(double) * h1.size(), cudaMemcpyDeviceToHost)); }
    for (int64_t b = 0; b < S.nb; ++b) {
      const int64_t o = p->h_perm[b];
      if (p->model == 0) {
        std::memcpy(jac + o * 18, &h0[b * 12], sizeof(double) * 12);
        std::memcpy(jac + o * 18 + 12, &he[b * 6], sizeof(double) * 6);
      } else {
        std::memcpy(jac + o * 144, &h0[b * 48], sizeof(double) * 48);
        std::memcpy(jac + o * 144 + 48, &he[b * 48], sizeof(double) * 48);
        std::memcpy(jac + o * 144 + 96, &h1[b * 48], sizeof(double) * 48);
      }
    }
  }
  return BA_OK;
}

int ba_cuda_covariance(ba_cuda_problem* p, const ba_cuda_options* options, double min_pivot_ratio, double* cov_kept,
                       double* cov_frames, double* smallest_pivot_ratio) {
  if (!p) return fail(BA_ERR_INVALID_ARGUMENT, "NULL problem");
  if (p->model < 0 || !p->params_set) return fail(BA_ERR_STATE, "set_model_b and set_parameters must be called before ba_cuda_covariance");
  // the covariance overwrites the Jacobian, the scaling and the Schur workspace the open solve works on
  if (p->lm.began && p->lm.go) return fail(BA_ERR_STATE, "ba_cuda_covariance between ba_cuda_solve_begin and the end of the solve");
  if (p->model != 1)
    return fail(BA_ERR_UNSUPPORTED, "ba_cuda_covariance: Model A is not supported (every camera is free, so J^T J has the 7-dimensional "
                "gauge null space of a similarity transform, and there are no constant blocks to remove it)");
  if (p->world > 1) return fail(BA_ERR_UNSUPPORTED, "ba_cuda_covariance runs on one GPU (world size %d)", p->world);
  if (p->n_rcs() > kDenseAutoMaxN)
    return fail(BA_ERR_UNSUPPORTED, "ba_cuda_covariance: reduced system of dimension %lld is above %lld", (long long)p->n_rcs(),
                (long long)kDenseAutoMaxN);
  ba_cuda_options opt;
  ba_cuda_options_init(&opt);
  if (options) {
    opt.loss_function = options->loss_function; opt.loss_scale = options->loss_scale;
    opt.profile_kernels = options->profile_kernels;
  }
  if (opt.loss_function < BA_LOSS_NONE || opt.loss_function > BA_LOSS_CAUCHY || (opt.loss_function != BA_LOSS_NONE && !(opt.loss_scale > 0.0)))
    return fail(BA_ERR_INVALID_ARGUMENT, "loss_function %d with scale %g", opt.loss_function, opt.loss_scale);
  opt.rcs_solver = BA_RCS_DENSE_CHOLESKY;
  BA_TRY(use_device(p));
  const bool profile = p->profile;
  p->loss = LossSpec{opt.loss_function, opt.loss_scale};
  p->profile = opt.profile_kernels != 0;
  const int rc = covariance_impl(p, opt, min_pivot_ratio, cov_kept, cov_frames, smallest_pivot_ratio);
  p->loss = LossSpec{0, 1.0};
  p->profile = profile;
  return rc;
}

int ba_cuda_reprojection_error(ba_cuda_problem* p, double* sum_half_sq, double* rms_per_coord) {
  if (!p) return fail(BA_ERR_INVALID_ARGUMENT, "NULL problem");
  if (p->model < 0 || !p->params_set) return fail(BA_ERR_STATE, "set_model_* and set_parameters must be called first");
  BA_TRY(use_device(p));
  // evaluate at x through the candidate buffers (same kernel as the LM cost evaluation)
  BA_CUDA_TRY(cudaMemcpyAsync(p->xf_c.p, p->xf.p, p->xf.bytes(), cudaMemcpyDeviceToDevice, p->st));
  BA_CUDA_TRY(cudaMemcpyAsync(p->xe_c.p, p->xe.p, p->xe.bytes(), cudaMemcpyDeviceToDevice, p->st));
  BA_TRY(build_tables(p, true));
  BA_CUDA_TRY(cudaEventRecord(p->k0, p->st));
  BA_TRY(run_cost_candidate(p));
  BA_CUDA_TRY(cudaEventRecord(p->k1, p->st));
  BA_TRY(allreduce(p, p->scal.p + S_CAND, 1, kNcclSum));
  BA_TRY(fetch_scalars(p));
  BA_CUDA_TRY(cudaEventElapsedTime(&p->last_kernel_ms, p->k0, p->k1));
  const double err = 0.5 * p->h_scal[S_CAND];
  const double n_points = (double)(p->model == 0 ? p->nb_global : 4 * p->nb_global);
  if (sum_half_sq) *sum_half_sq = err;
  if (rms_per_coord) *rms_per_coord = n_points > 0 ? std::pow((err * 2.0) / (n_points * 2.0), 0.5) : 0.0;   // no point: no error, not NaN
  return BA_OK;
}

// shared body: rotations either from rvecs (Rodrigues on the device) or given as matrices
static int project_points_impl(ba_cuda_problem* p, int64_t n_points, const double* xyz, const int32_t* cam_of_point, int32_t n_cam,
                               const double* rvec3 /* n_cam x 3 or NULL */, const double* rot9 /* n_cam x 9 or NULL */,
                               const double* tvec3 /* n_cam x 3 */, const double* intr4, const float* image_xy, double* sum_half_sq,
                               double* rms_per_coord, double* reprojected_xy) {
  for (int64_t i = 0; i < n_points; ++i)
    if (cam_of_point[i] < 0 || cam_of_point[i] >= n_cam) return fail(BA_ERR_INVALID_ARGUMENT, "point %lld: camera out of range", (long long)i);
  BA_TRY(use_device(p));
  cudaStream_t st = p->st;
  DVec<double> d_xyz, d_rt, d_t, d_K, d_R, d_rep, d_part, d_out;
  DVec<int32_t> d_cam;
  DVec<float> d_img;
  BA_TRY(d_xyz.upload(xyz, 3 * n_points, st)); BA_TRY(d_cam.upload(cam_of_point, n_points, st));
  BA_TRY(d_img.upload(image_xy, 2 * n_points, st)); BA_TRY(d_t.upload(tvec3, 3 * (size_t)n_cam, st));
  BA_TRY(d_K.upload(intr4, 4 * (size_t)n_cam, st));
  if (rot9) {
    BA_TRY(d_R.upload(rot9, 9 * (size_t)n_cam, st));
  } else {
    std::vector<double> rt(6 * (size_t)n_cam, 0.0);
    for (int32_t c = 0; c < n_cam; ++c) std::memcpy(&rt[6 * (size_t)c], rvec3 + 3 * (size_t)c, sizeof(double) * 3);
    BA_TRY(d_rt.upload(rt.data(), rt.size(), st));
    BA_TRY(d_R.alloc(9 * (size_t)n_cam));
    BA_LAUNCH(p, KT_MISC, k_rodrigues_cv, grid_for(n_cam, 64), 64, 0, d_rt.p, n_cam, d_R.p, nullptr);
    BA_CUDA_TRY(cudaStreamSynchronize(st));  // rt (host staging) must outlive the copy
  }
  const int grid = (int)grid_for(n_points, 256);
  BA_TRY(d_rep.alloc(reprojected_xy ? 2 * n_points : 0)); BA_TRY(d_part.alloc(grid)); BA_TRY(d_out.alloc(1));
  BA_CUDA_TRY(cudaEventRecord(p->k0, st));
  BA_LAUNCH(p, KT_COST, k_project_error, grid, 256, 0, n_points, d_xyz.p, d_cam.p, d_R.p, d_t.p, d_K.p, d_img.p,
            reprojected_xy ? d_rep.p : nullptr, d_part.p);
  BA_LAUNCH(p, KT_FOLD, k_fold_partials, 1, 1024, 0, d_part.p, grid, d_out.p, 0, 0);
  BA_CUDA_TRY(cudaEventRecord(p->k1, st));
  BA_CUDA_TRY(cudaGetLastError());
  double err = 0.0;
  BA_CUDA_TRY(cudaMemcpyAsync(&err, d_out.p, sizeof(double), cudaMemcpyDeviceToHost, st));
  if (reprojected_xy) BA_CUDA_TRY(cudaMemcpyAsync(reprojected_xy, d_rep.p, sizeof(double) * 2 * n_points, cudaMemcpyDeviceToHost, st));
  BA_CUDA_TRY(cudaStreamSynchronize(st));
  BA_CUDA_TRY(cudaEventElapsedTime(&p->last_kernel_ms, p->k0, p->k1));
  if (n_points == 0) err = 0.0;
  if (sum_half_sq) *sum_half_sq = err;
  if (rms_per_coord) *rms_per_coord = n_points > 0 ? std::pow((err * 2.0) / (n_points * 2.0), 0.5) : 0.0;   // no point: no error, not NaN
  return BA_OK;
}

int ba_cuda_project_points_error(ba_cuda_problem* p, int64_t n_points, const double* xyz, const int32_t* cam_of_point,
                                 int32_t n_cam, const double* rvec_tvec6, const double* intr4, const float* image_xy,
                                 double* sum_half_sq, double* rms_per_coord, double* reprojected_xy) {
  if (!p || n_points < 0 || n_cam < 1 || !rvec_tvec6 || !intr4 || (n_points > 0 && (!xyz || !cam_of_point || !image_xy)))
    return fail(BA_ERR_INVALID_ARGUMENT, "ba_cuda_project_points_error: bad arguments");
  std::vector<double> r(3 * (size_t)n_cam), t(3 * (size_t)n_cam);
  for (int32_t c = 0; c < n_cam; ++c)
    for (int k = 0; k < 3; ++k) { r[3 * (size_t)c + k] = rvec_tvec6[6 * (size_t)c + k]; t[3 * (size_t)c + k] = rvec_tvec6[6 * (size_t)c + 3 + k]; }
  return project_points_impl(p, n_points, xyz, cam_of_point, n_cam, r.data(), nullptr, t.data(), intr4, image_xy, sum_half_sq,
                             rms_per_coord, reprojected_xy);
}

int ba_cuda_project_points_error_rt(ba_cuda_problem* p, int64_t n_points, const double* xyz, const int32_t* cam_of_point,
                                    int32_t n_cam, const double* rot9, const double* tvec3, const double* intr4,
                                    const float* image_xy, double* sum_half_sq, double* rms_per_coord, double* reprojected_xy) {
  if (!p || n_points < 0 || n_cam < 1 || !rot9 || !tvec3 || !intr4 || (n_points > 0 && (!xyz || !cam_of_point || !image_xy)))
    return fail(BA_ERR_INVALID_ARGUMENT, "ba_cuda_project_points_error_rt: bad arguments");
  return project_points_impl(p, n_points, xyz, cam_of_point, n_cam, nullptr, rot9, tvec3, intr4, image_xy, sum_half_sq, rms_per_coord,
                             reprojected_xy);
}

int ba_cuda_model_b_outputs(ba_cuda_problem* p, double* rot9, double* inv12, double* corners) {
  if (!p) return fail(BA_ERR_INVALID_ARGUMENT, "NULL problem");
  if (p->model != 1 || !p->params_set) return fail(BA_ERR_STATE, "a Model B problem with parameters is required");
  BA_TRY(use_device(p));
  cudaStream_t st = p->st;
  const int C = p->n_cam;
  const Structure& S = p->S;
  DVec<double> d_R, d_inv, d_c;
  BA_TRY(d_R.alloc(9 * (size_t)C)); BA_TRY(d_inv.alloc(12 * (size_t)C)); BA_TRY(d_c.alloc(12 * S.nb));
  k_rodrigues_cv<<<grid_for(C, 64), 64, 0, st>>>(p->xf.p, C, d_R.p, d_inv.p);  // the first C f-blocks are the cameras
  BA_TRY(build_tables(p, false));
  k_corners_b<<<grid_for(S.nb * 4, 256), 256, 0, st>>>(S.nb, S.perm.p, S.ob_e.p, p->ob_marker.p, C, p->tab_f.p, p->tab_e.p, p->half_side, d_c.p);
  BA_CUDA_TRY(cudaGetLastError());
  if (rot9) BA_CUDA_TRY(cudaMemcpyAsync(rot9, d_R.p, d_R.bytes(), cudaMemcpyDeviceToHost, st));
  if (inv12) BA_CUDA_TRY(cudaMemcpyAsync(inv12, d_inv.p, d_inv.bytes(), cudaMemcpyDeviceToHost, st));
  if (corners && S.nb) BA_CUDA_TRY(cudaMemcpyAsync(corners, d_c.p, d_c.bytes(), cudaMemcpyDeviceToHost, st));
  BA_CUDA_TRY(cudaStreamSynchronize(st));
  return BA_OK;
}

int ba_cuda_marker_corners(ba_cuda_problem* p, int64_t n, const double* rvec_tvec6, double marker_side, double* corners) {
  if (!p || n < 0 || (n > 0 && (!rvec_tvec6 || !corners))) return fail(BA_ERR_INVALID_ARGUMENT, "ba_cuda_marker_corners: bad arguments");
  BA_TRY(use_device(p));
  DVec<double> d_in, d_out;
  BA_TRY(d_in.upload(rvec_tvec6, 6 * (size_t)n, p->st)); BA_TRY(d_out.alloc(12 * (size_t)n));
  if (n > 0) BA_LAUNCH(p, KT_MISC, k_marker_corners, grid_for(n, 128), 128, 0, n, d_in.p, marker_side / 2, d_out.p);
  BA_CUDA_TRY(cudaGetLastError());
  if (n > 0) BA_CUDA_TRY(cudaMemcpyAsync(corners, d_out.p, sizeof(double) * 12 * n, cudaMemcpyDeviceToHost, p->st));
  BA_CUDA_TRY(cudaStreamSynchronize(p->st));
  return BA_OK;
}

int ba_cuda_compose_poses(ba_cuda_problem* p, int64_t n, const double* a6, const double* b6, int32_t invert_b, double* out6) {
  if (!p || n < 0 || (n > 0 && (!a6 || !b6 || !out6))) return fail(BA_ERR_INVALID_ARGUMENT, "ba_cuda_compose_poses: bad arguments");
  BA_TRY(use_device(p));
  DVec<double> d_a, d_b, d_out;
  BA_TRY(d_a.upload(a6, 6 * (size_t)n, p->st)); BA_TRY(d_b.upload(b6, 6 * (size_t)n, p->st)); BA_TRY(d_out.alloc(6 * (size_t)n));
  if (n > 0) BA_LAUNCH(p, KT_MISC, k_compose_poses, grid_for(n, 128), 128, 0, n, d_a.p, d_b.p, invert_b ? 1 : 0, d_out.p);
  BA_CUDA_TRY(cudaGetLastError());
  if (n > 0) BA_CUDA_TRY(cudaMemcpyAsync(out6, d_out.p, sizeof(double) * 6 * n, cudaMemcpyDeviceToHost, p->st));
  BA_CUDA_TRY(cudaStreamSynchronize(p->st));
  return BA_OK;
}

double ba_cuda_last_kernel_ms(const ba_cuda_problem* p) { return p ? (double)p->last_kernel_ms : 0.0; }

}  // extern "C"
