// clc_api.cu -- host side of libclc_b200.so: the C ABI declared in include/clc_b200.h.
//
// No CPU fallback lives here: every entry point drives the sm_100a kernels of clc_kernels.cuh and fails loudly
// (status code + clc_last_error()) when CUDA is unusable.  The only host arithmetic is O(1) dense work on the
// reduced 6x6 / 9x9 systems for the two diagnostic outputs the reference prints (singular values, closed form).
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>  // types only; the library is dlopen()ed so that single-GPU use has no NCCL dependency

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include <cub/device/device_scan.cuh>

#include "../../include/clc_b200.h"
#include "clc_kernels.cuh"
#include "clc_linefit.cuh"
#include "clc_scans.cuh"
#include "clc_small.cuh"

namespace {

thread_local std::string g_last_error;
std::atomic<int64_t> g_launches{0};

int fail(int code, const std::string& msg) {
  g_last_error = msg;
  return code;
}

#define CLC_CUDA(expr)                                                                                   \
  do {                                                                                                   \
    cudaError_t _e = (expr);                                                                             \
    if (_e != cudaSuccess)                                                                               \
      return fail(CLC_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e) + " (" __FILE__ ":" + \
                                    std::to_string(__LINE__) + ")");                                     \
  } while (0)

#define CLC_LAUNCH_CHECK()                  \
  do {                                      \
    g_launches.fetch_add(1);                \
    CLC_CUDA(cudaGetLastError());           \
  } while (0)

// ---- NCCL through dlopen -------------------------------------------------------------------------------------
struct NcclApi {
  void* handle = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  std::string error;
};

NcclApi* nccl_api() {
  static NcclApi api;
  static bool tried = false;
  if (tried) return &api;
  tried = true;
  const char* names[] = {"libnccl.so.2", "libnccl.so"};
  for (const char* n : names) {
    api.handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    if (api.handle) break;
  }
  if (!api.handle) {
    api.error = std::string("dlopen(libnccl.so.2) failed: ") + dlerror();
    return &api;
  }
  api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(dlsym(api.handle, "ncclGetUniqueId"));
  api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(dlsym(api.handle, "ncclCommInitRank"));
  api.AllReduce = reinterpret_cast<decltype(api.AllReduce)>(dlsym(api.handle, "ncclAllReduce"));
  api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(dlsym(api.handle, "ncclCommDestroy"));
  api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(dlsym(api.handle, "ncclGetErrorString"));
  if (!api.GetUniqueId || !api.CommInitRank || !api.AllReduce || !api.CommDestroy || !api.GetErrorString) {
    api.error = "libnccl.so.2 lacks a required symbol";
    api.handle = nullptr;
  }
  return &api;
}

#define CLC_NCCL(expr)                                                                                   \
  do {                                                                                                   \
    ncclResult_t _r = (expr);                                                                            \
    if (_r != ncclSuccess)                                                                               \
      return fail(CLC_ERR_NCCL, std::string(#expr) + ": " + nccl_api()->GetErrorString(_r));            \
  } while (0)

// ---- O(1) dense helpers on the reduced systems ------------------------------------------------------------------

// cyclic Jacobi: symmetric A (n x n, row-major, n <= 9) = V diag(w) V^T
template <int N>
void sym_eig(const double* Ain, double* w, double* V) {
  double A[N * N];
  std::memcpy(A, Ain, sizeof(A));
  for (int i = 0; i < N; ++i)
    for (int j = 0; j < N; ++j) V[i * N + j] = (i == j) ? 1.0 : 0.0;
  for (int sweep = 0; sweep < 64; ++sweep) {
    double off = 0.0, dg = 0.0;
    for (int i = 0; i < N; ++i) {
      dg += A[i * N + i] * A[i * N + i];
      for (int j = i + 1; j < N; ++j) off += A[i * N + j] * A[i * N + j];
    }
    if (off <= 1e-60 || off <= 1e-34 * dg) break;
    for (int p = 0; p < N - 1; ++p)
      for (int q = p + 1; q < N; ++q) {
        const double apq = A[p * N + q];
        if (apq == 0.0) continue;
        const double theta = (A[q * N + q] - A[p * N + p]) / (2.0 * apq);
        const double t = (theta >= 0.0 ? 1.0 : -1.0) / (std::fabs(theta) + std::sqrt(theta * theta + 1.0));
        const double c = 1.0 / std::sqrt(t * t + 1.0), s = t * c;
        for (int k = 0; k < N; ++k) {
          const double a = A[k * N + p], b = A[k * N + q];
          A[k * N + p] = c * a - s * b;
          A[k * N + q] = s * a + c * b;
        }
        for (int k = 0; k < N; ++k) {
          const double a = A[p * N + k], b = A[q * N + k];
          A[p * N + k] = c * a - s * b;
          A[q * N + k] = s * a + c * b;
        }
        for (int k = 0; k < N; ++k) {
          const double a = V[k * N + p], b = V[k * N + q];
          V[k * N + p] = c * a - s * b;
          V[k * N + q] = s * a + c * b;
        }
      }
  }
  for (int i = 0; i < N; ++i) w[i] = A[i * N + i];
}

template <int N>
void sym_singular_values(const double* A, double* sv) {
  double w[N], V[N * N];
  sym_eig<N>(A, w, V);
  for (int i = 0; i < N; ++i) sv[i] = std::fabs(w[i]);
  std::sort(sv, sv + N, [](double a, double b) { return a > b; });
}

// LDL^T with diagonal pivoting for the positive semi-definite 9x9 of the closed form
void ldlt9_solve(const double* Ain, const double* bin, double* x) {
  constexpr int n = 9;
  double A[81], b[9];
  int perm[9];
  std::memcpy(A, Ain, sizeof(A));
  std::memcpy(b, bin, sizeof(b));
  for (int i = 0; i < n; ++i) perm[i] = i;
  for (int k = 0; k < n; ++k) {
    int piv = k;
    for (int i = k + 1; i < n; ++i)
      if (std::fabs(A[i * n + i]) > std::fabs(A[piv * n + piv])) piv = i;
    if (piv != k) {
      for (int j = 0; j < n; ++j) std::swap(A[k * n + j], A[piv * n + j]);
      for (int j = 0; j < n; ++j) std::swap(A[j * n + k], A[j * n + piv]);
      std::swap(b[k], b[piv]);
      std::swap(perm[k], perm[piv]);
    }
    const double d = A[k * n + k];
    if (d == 0.0) continue;
    for (int i = k + 1; i < n; ++i) {
      const double l = A[i * n + k] / d;
      for (int j = k + 1; j < n; ++j) A[i * n + j] -= l * A[k * n + j];
      A[i * n + k] = l;
    }
  }
  double z[9], y[9];
  for (int i = 0; i < n; ++i) {
    double s = b[i];
    for (int k = 0; k < i; ++k) s -= A[i * n + k] * z[k];
    z[i] = s;
  }
  for (int i = 0; i < n; ++i) z[i] = (A[i * n + i] != 0.0) ? z[i] / A[i * n + i] : 0.0;
  for (int i = n - 1; i >= 0; --i) {
    double s = z[i];
    for (int k = i + 1; k < n; ++k) s -= A[k * n + i] * y[k];
    y[i] = s;
  }
  for (int i = 0; i < n; ++i) x[perm[i]] = y[i];
}

int64_t round_up(int64_t v, int64_t m) { return (v + m - 1) / m * m; }

}  // namespace

// ---- pinned host mirrors: pooled process-wide (cudaMallocHost costs milliseconds) ---------------------------------
struct PinnedBlock {
  clc::LmState lm;
  double sums[clc::kMaxOut];
  double pose[8];
  int done;
  int nonplanar;
};
namespace {
std::mutex g_pinned_mutex;
std::vector<PinnedBlock*> g_pinned_free;
PinnedBlock* pinned_acquire() {
  {
    std::lock_guard<std::mutex> lock(g_pinned_mutex);
    if (!g_pinned_free.empty()) {
      PinnedBlock* b = g_pinned_free.back();
      g_pinned_free.pop_back();
      return b;
    }
  }
  PinnedBlock* b = nullptr;
  if (cudaMallocHost(&b, sizeof(PinnedBlock)) != cudaSuccess) return nullptr;
  return b;
}
void pinned_release(PinnedBlock* b) {
  if (!b) return;
  std::lock_guard<std::mutex> lock(g_pinned_mutex);
  g_pinned_free.push_back(b);
}
}  // namespace

// ---- the communicator and problem objects ------------------------------------------------------------------------
struct clc_comm {
  ncclComm_t comm = nullptr;
  int nranks = 1, rank = 0, device = 0;
  // fused peer exchange: one cudaMalloc block per rank = mailbox [2][nranks][kMailboxSlot][2] words, then the counter
  void* p2p_block = nullptr;
  void* peer_block[clc::kMaxRanks] = {};
  bool p2p_ready = false;
  bool local = false;  // in-process group: peer_block[] are plain peer-access pointers (no IPC handles, no NCCL communicator)
  size_t mailbox_bytes() const { return sizeof(unsigned long long) * 2 * 2 * (size_t)nranks * clc::kMailboxSlot; }
  size_t block_bytes() const { return mailbox_bytes() + sizeof(unsigned long long); }  // + exchange counter
};

struct clc_problem {
  int device = 0;
  cudaStream_t stream = nullptr;
  int num_sms = 0;
  int grid = 0;
  int64_t n_frames = 0, n_points = 0, n_points_padded = 0, n_edges = 0;
  int use_loss = 1;
  double cauchy_a = 0.05;
  // device buffers
  double *x = nullptr, *y = nullptr, *z = nullptr;  // views into xy_block / z_block
  void *xy_block = nullptr, *z_block = nullptr;     // the allocations (x and y share one; z is created only when needed)
  double* frame_pose = nullptr;
  double* frame_pose_true = nullptr;  // synthetic problems with a camera model: the poses the points were generated from
  double* plane = nullptr;
  int64_t* offsets = nullptr;
  int* warp_first_frame = nullptr;
  double* edge_plane = nullptr;
  double* edge_pt = nullptr;
  unsigned long long* partials_ll = nullptr;  // tagged block partials (clc_kernels.cuh)
  unsigned int* launch_seq = nullptr;
  unsigned long long* pose_ll = nullptr;      // looping grids: next pose + done flag as tagged words
  double* sums = nullptr;
  double* pose = nullptr;
  clc::LmState* lm = nullptr;
  double* flush_buf = nullptr;
  int64_t flush_n = 0;
  unsigned long long* timing = nullptr;  // profiling hook (clc_debug_sweep_timing)
  bool use_pdl = true;                   // CLC_PDL=0 disables programmatic dependent launch in the LM loop
  int64_t l2_persist_bytes = 0;          // persisting-L2 window over the coordinate arrays during LM solves (0 = off)
  bool l2_window_set = false;
  bool small_kernel = true;              // CLC_SMALL_KERNEL=0: never use the one-cluster kernel of clc_small.cuh
  int loop_in_kernel = 1;                // CLC_LOOP_IN_KERNEL: 0 one launch per LM iteration; 1 single-block problems run the whole
                                         // LM loop in one launch; 2 every problem does (persistent grid, block 0 hands out the poses)
  // pinned host mirrors (views into one pooled block)
  PinnedBlock* pinned = nullptr;
  double* h_sums = nullptr;
  int* h_done = nullptr;
  clc::LmState* h_lm = nullptr;
  // communicator (borrowed)
  clc_comm* comm_obj = nullptr;
  ncclComm_t comm = nullptr;
  int nranks = 1, rank = 0;
  int* p2p_error = nullptr;
  int allreduce_mode = 0;
  int64_t per_warp = 0;
  int grid_full = 0;  // SM count x resident blocks
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;  // device time of clc_solve_lm
  // planar data (every z exactly 0: a 2-D laser): the z stream is dropped and the two-stream kernels run
  int* d_nonplanar = nullptr;  // raised by the upload kernel when a z != 0 was seen
  bool z_all_zero = false;     // property of the data
  bool host_planarity_known = false;  // the host packers checked every z (clc_upload.inl): no device-side verdict to fetch
  bool planar = false;         // the two-stream kernels are in use (z_all_zero && planar_mode != 0 && large enough)
  int planar_mode = 1;         // 1 = automatic (default), 0 = always the general three-stream kernels
  int64_t planar_min_points = 0;
};

namespace {

clc::ProblemView make_view(const clc_problem* p) {
  clc::ProblemView v;
  v.x = p->x; v.y = p->y; v.z = p->z;
  v.plane = p->plane;
  v.offsets = p->offsets;
  v.warp_first_frame = p->warp_first_frame;
  v.edge_plane = p->edge_plane;
  v.edge_pt = p->edge_pt;
  v.n_frames = p->n_frames;
  v.n_points = p->n_points;
  v.n_edges = p->n_edges;
  v.per_warp = p->per_warp;
  v.a2 = p->cauchy_a * p->cauchy_a;
  v.inv_a2 = 1.0 / v.a2;
  return v;
}

int set_device(const clc_problem* p) {
  CLC_CUDA(cudaSetDevice(p->device));
  return CLC_OK;
}

// one K1 launch on the problem's stream
// collective: the sums of this launch are to be all-reduced (in-kernel when the peer path is active)
int launch_sweep(clc_problem* p, int mode, bool loss, bool edges, const double* d_pose, const int* d_done,
                 clc::LmState* d_lm, bool collective = true, bool pdl = false, int loop_sweeps = 1) {
  clc::SweepArgs a;
  a.pose7 = d_pose;
  a.done = d_done;
  a.partials_ll = p->partials_ll;
  a.sums = p->sums;
  a.launch_seq = p->launch_seq;
  a.pose_ll = p->pose_ll;
  a.lm = d_lm;
  a.use_loss = loss ? 1 : 0;
  a.use_edges = edges ? 1 : 0;
  a.loop_sweeps = loop_sweeps;
  a.timing = p->timing;
  a.nranks = 1;
  a.rank = 0;
  a.seq_counter = nullptr;
  a.error = p->p2p_error;
  if (p->nranks > 1 && p->allreduce_mode == 1 && collective) {
    clc_comm* c = p->comm_obj;
    a.nranks = c->nranks;
    a.rank = c->rank;
    a.seq_counter = reinterpret_cast<unsigned long long*>(static_cast<char*>(c->p2p_block) + c->mailbox_bytes());
    for (int r = 0; r < c->nranks; ++r) a.peer_mailbox[r] = static_cast<unsigned long long*>(c->peer_block[r]);
  }
  const clc::ProblemView v = make_view(p);
  // cudaLaunchKernelEx so that back-to-back sweeps of the LM loop can use programmatic dependent launch
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)p->grid);
  cfg.blockDim = dim3(clc::kThreads);
  cfg.dynamicSmemBytes = clc::dyn_smem_bytes(p->planar);
  cfg.stream = p->stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = pdl ? 1 : 0;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t le;
  if (!p->planar && p->z == nullptr) return fail(CLC_ERR_INVALID, "internal: general sweep without a z stream");
  if (mode == clc::kModeClosedForm) {
    le = p->planar ? cudaLaunchKernelEx(&cfg, clc::clc_sweep_kernel<false, clc::kModeClosedForm, true>, v, a)
                   : cudaLaunchKernelEx(&cfg, clc::clc_sweep_kernel<false, clc::kModeClosedForm, false>, v, a);
  } else if (loop_sweeps > 1) {
    // the instantiations that loop the LM inside the kernel (one launch per solve)
    if (d_lm == nullptr) return fail(CLC_ERR_INVALID, "internal: looping sweep without an LM state");
    if (loss)
      le = p->planar ? cudaLaunchKernelEx(&cfg, clc::clc_sweep_kernel<true, clc::kModeLM, true, true>, v, a)
                     : cudaLaunchKernelEx(&cfg, clc::clc_sweep_kernel<true, clc::kModeLM, false, true>, v, a);
    else
      le = p->planar ? cudaLaunchKernelEx(&cfg, clc::clc_sweep_kernel<false, clc::kModeLM, true, true>, v, a)
                     : cudaLaunchKernelEx(&cfg, clc::clc_sweep_kernel<false, clc::kModeLM, false, true>, v, a);
  } else if (loss) {
    le = p->planar ? cudaLaunchKernelEx(&cfg, clc::clc_sweep_kernel<true, clc::kModeLM, true>, v, a)
                   : cudaLaunchKernelEx(&cfg, clc::clc_sweep_kernel<true, clc::kModeLM, false>, v, a);
  } else {
    le = p->planar ? cudaLaunchKernelEx(&cfg, clc::clc_sweep_kernel<false, clc::kModeLM, true>, v, a)
                   : cudaLaunchKernelEx(&cfg, clc::clc_sweep_kernel<false, clc::kModeLM, false>, v, a);
  }
  if (le != cudaSuccess) return fail(CLC_ERR_CUDA, std::string("sweep launch: ") + cudaGetErrorString(le));
  CLC_LAUNCH_CHECK();
  return CLC_OK;
}

int allreduce_sums(clc_problem* p, int count) {
  if (p->nranks <= 1 || p->allreduce_mode == 1) return CLC_OK;  // single rank, or already reduced inside the kernel
  CLC_NCCL(nccl_api()->AllReduce(p->sums, p->sums, (size_t)count, ncclDouble, ncclSum, p->comm, p->stream));
  return CLC_OK;
}

// Waits for a stream with a short spin before blocking: a blocking cudaStreamSynchronize puts the thread to sleep and the wake-up
// costs tens of microseconds (measured: 40-90 us per mid-solve poll inside a CPU-quota'd container, profiles/r2_loop_modes2.txt),
// which is as long as a whole sweep at BASELINE configs[1].  Work that takes longer than the spin budget falls back to blocking.
cudaError_t sync_stream_low_latency(cudaStream_t st) {
  const auto t0 = std::chrono::steady_clock::now();
  for (;;) {
    const cudaError_t e = cudaStreamQuery(st);
    if (e != cudaErrorNotReady) return e;
    if (std::chrono::steady_clock::now() - t0 > std::chrono::microseconds(400)) return cudaStreamSynchronize(st);
#if defined(__x86_64__) || defined(__i386__)
    __builtin_ia32_pause();
#endif
  }
}

// a peer that never answered the in-kernel exchange (5 s time-out) is an error, not a hang
int check_p2p_error(clc_problem* p) {
  // only a multi-block gather or a peer exchange can raise the flag: single-block / one-cluster problems skip the round trip
  if (p->grid <= 1 && p->nranks <= 1) return CLC_OK;
  int err = 0;
  CLC_CUDA(cudaMemcpyAsync(&err, p->p2p_error, sizeof(int), cudaMemcpyDeviceToHost, p->stream));
  CLC_CUDA(sync_stream_low_latency(p->stream));
  if (err == 2) return fail(CLC_ERR_CUDA, "sweep kernel: the persistent grid was not co-resident (ticket wait timed out)");
  if (err) return fail(CLC_ERR_NCCL, "peer exchange timed out: a rank did not reach the collective");
  return CLC_OK;
}

// common tail of the two create paths: planes, warp table, work buffers
int materialise_z(clc_problem* p);

// Static work partition of the sweep kernels: launch grid, points per warp, first frame of every warp.  Depends on the
// kernel family (the planar kernels use longer stages), so it is redone when the planar mode changes.
int partition(clc_problem* p) {
  const int chunk = p->planar ? clc::kPlanarChunk : clc::kChunk;
  p->grid = p->grid_full;
  {
    // small problems (the reference's own sizes: a few thousand points) do not need the whole machine: a warp takes at
    // least one stage, so launch only as many blocks as there are stages to hand out -- fewer tickets and
    // partial sums on the serial tail of every LM iteration
    const int64_t stages = (p->n_points + chunk - 1) / chunk;
    const int64_t blocks_needed = std::max<int64_t>(1, (stages + clc::kWarps - 1) / clc::kWarps);
    if (blocks_needed < p->grid) p->grid = (int)blocks_needed;
    // the reference's own sizes (50 boards x 180 beams, reference main/calibr_simulation.cpp:34,79) fit ONE block: a
    // single-block grid lets the kernel run the whole LM loop by itself (no launch, no inter-block exchange per iteration)
    int64_t single_block_max = (int64_t)clc::kWarps * 8 * clc::kChunk;  // up to 8 stages per warp and sweep (16384 points)
    if (const char* env = std::getenv("CLC_SINGLE_BLOCK_MAX_POINTS")) single_block_max = std::atoll(env);
    if (p->n_points <= single_block_max) p->grid = 1;
  }
  const int64_t n_warps = (int64_t)p->grid * clc::kWarps;
  p->per_warp = std::max<int64_t>(chunk, round_up((p->n_points + n_warps - 1) / n_warps, chunk));  // whole stages
  if (p->warp_first_frame) CLC_CUDA(cudaFreeAsync(p->warp_first_frame, p->stream));
  if (p->partials_ll) CLC_CUDA(cudaFreeAsync(p->partials_ll, p->stream));
  p->warp_first_frame = nullptr;
  p->partials_ll = nullptr;
  CLC_CUDA(cudaMallocAsync(&p->warp_first_frame, sizeof(int) * n_warps, p->stream));
  const size_t ll_bytes = sizeof(unsigned long long) * 2 * (size_t)p->grid * clc::kMaxOut;
  CLC_CUDA(cudaMallocAsync(&p->partials_ll, ll_bytes, p->stream));
  CLC_CUDA(cudaMemsetAsync(p->partials_ll, 0, ll_bytes, p->stream));  // tag 0 never matches a launch (sequence numbers start at 1)
  const int threads = 256;
  const int blocks = (int)((n_warps + threads - 1) / threads);
  clc::clc_warp_table_kernel<<<blocks, threads, 0, p->stream>>>(p->offsets, p->n_frames, p->n_points, p->per_warp, n_warps,
                                                                p->warp_first_frame);
  CLC_LAUNCH_CHECK();
  return CLC_OK;
}

int finish_create(clc_problem* p) {
  const int threads = 256;
  if (p->n_frames > 0) {
    const int blocks = (int)((p->n_frames + threads - 1) / threads);
    clc::clc_planes_kernel<<<blocks, threads, 0, p->stream>>>(p->frame_pose, p->n_frames, p->plane, p->edge_plane);
    CLC_LAUNCH_CHECK();
  }
  // persistent grid: SM count x resident blocks per SM (the smallest occupancy of the instantiations used); queried once
  // per device and cached -- problem creation is on the latency path of the reference-facing calls
  static std::mutex cfg_mutex;
  static int cached_blocks_per_sm[64] = {};
  int blocks_per_sm = 0;
  {
    std::lock_guard<std::mutex> lock(cfg_mutex);
    if (p->device < 64) blocks_per_sm = cached_blocks_per_sm[p->device];
  }
  if (blocks_per_sm == 0) {
    int occ = 0, occ_min = 1 << 30;
    const void* variants[] = {
        (const void*)clc::clc_sweep_kernel<true, clc::kModeLM, false>,         (const void*)clc::clc_sweep_kernel<true, clc::kModeLM, true>,
        (const void*)clc::clc_sweep_kernel<false, clc::kModeLM, false>,        (const void*)clc::clc_sweep_kernel<false, clc::kModeLM, true>,
        (const void*)clc::clc_sweep_kernel<false, clc::kModeClosedForm, false>, (const void*)clc::clc_sweep_kernel<false, clc::kModeClosedForm, true>,
        (const void*)clc::clc_sweep_kernel<true, clc::kModeLM, false, true>,   (const void*)clc::clc_sweep_kernel<true, clc::kModeLM, true, true>,
        (const void*)clc::clc_sweep_kernel<false, clc::kModeLM, false, true>,  (const void*)clc::clc_sweep_kernel<false, clc::kModeLM, true, true>};
    for (int v = 0; v < 10; ++v) {
      const void* fn = variants[v];
      const int smem = clc::dyn_smem_bytes((v & 1) != 0);  // odd entries are the planar instantiations
      CLC_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
      CLC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fn, clc::kThreads, smem));
      occ_min = std::min(occ_min, occ);
    }
    if (occ_min < 1) return fail(CLC_ERR_CUDA, "the sweep kernel does not fit on this device");
    blocks_per_sm = std::max(1, std::min(occ_min, clc::kBlocksPerSM));
    if (const char* env = std::getenv("CLC_BLOCKS_PER_SM")) {
      const int v = std::atoi(env);
      if (v >= 1) blocks_per_sm = std::min(v, std::max(1, occ_min));
    }
    std::lock_guard<std::mutex> lock(cfg_mutex);
    if (p->device < 64) cached_blocks_per_sm[p->device] = blocks_per_sm;
  }
  p->grid_full = p->num_sms * blocks_per_sm;
  if (const char* env = std::getenv("CLC_PDL")) p->use_pdl = std::atoi(env) != 0;
  if (const char* env = std::getenv("CLC_LOOP_IN_KERNEL")) p->loop_in_kernel = std::atoi(env);
  if (const char* env = std::getenv("CLC_SMALL_KERNEL")) p->small_kernel = std::atoi(env) != 0;
  if (const char* env = std::getenv("CLC_L2_PERSIST_MB")) p->l2_persist_bytes = (int64_t)std::atoll(env) << 20;
  CLC_CUDA(cudaMallocAsync(&p->sums, sizeof(double) * clc::kMaxOut, p->stream));
  CLC_CUDA(cudaMallocAsync(&p->pose, sizeof(double) * 8, p->stream));
  CLC_CUDA(cudaMallocAsync(&p->launch_seq, sizeof(unsigned int), p->stream));
  CLC_CUDA(cudaMallocAsync(&p->pose_ll, sizeof(unsigned long long) * 16, p->stream));
  CLC_CUDA(cudaMemsetAsync(p->pose_ll, 0, sizeof(unsigned long long) * 16, p->stream));
  CLC_CUDA(cudaMallocAsync(&p->lm, sizeof(clc::LmState), p->stream));
  CLC_CUDA(cudaMallocAsync(&p->p2p_error, sizeof(int), p->stream));
  CLC_CUDA(cudaMemsetAsync(p->p2p_error, 0, sizeof(int), p->stream));
  CLC_CUDA(cudaMemsetAsync(p->launch_seq, 0, sizeof(unsigned int), p->stream));
  CLC_CUDA(cudaMemsetAsync(p->sums, 0, sizeof(double) * clc::kMaxOut, p->stream));
  p->pinned = pinned_acquire();
  if (!p->pinned) return fail(CLC_ERR_CUDA, "cudaMallocHost failed");
  p->h_sums = p->pinned->sums;
  p->h_done = &p->pinned->done;
  p->h_lm = &p->pinned->lm;
  if (p->host_planarity_known) {
    CLC_CUDA(cudaStreamSynchronize(p->stream));
  } else {
    p->pinned->nonplanar = 1;
    CLC_CUDA(cudaMemcpyAsync(&p->pinned->nonplanar, p->d_nonplanar, sizeof(int), cudaMemcpyDeviceToHost, p->stream));
    CLC_CUDA(cudaStreamSynchronize(p->stream));
    p->z_all_zero = p->pinned->nonplanar == 0;
  }
  if (const char* env = std::getenv("CLC_PLANAR")) p->planar_mode = std::atoi(env) != 0 ? 1 : 0;
  // The planar kernels stream 256-point stages; they pay off once every warp of the full grid has at least one such stage.
  // Smaller problems (the reference's own 50 x 180) are latency-bound and keep the 128-point stages of the general kernels.
  p->planar_min_points = (int64_t)p->grid_full * clc::kWarps * clc::kPlanarChunk;
  if (const char* env = std::getenv("CLC_PLANAR_MIN_POINTS")) p->planar_min_points = std::atoll(env);
  p->planar = p->z_all_zero && p->planar_mode != 0 && p->n_points >= p->planar_min_points;
  if (p->planar && p->z != nullptr) {
    // a third of the point storage goes back to the pool
    CLC_CUDA(cudaFreeAsync(p->z_block, p->stream));
    p->z = nullptr;
    p->z_block = nullptr;
  } else if (!p->planar) {
    int rc = materialise_z(p);
    if (rc != CLC_OK) return rc;
  }
  return partition(p);
}

int init_device(clc_problem* p, int device) {
  int count = 0;
  CLC_CUDA(cudaGetDeviceCount(&count));
  if (count <= 0) return fail(CLC_ERR_CUDA, "no CUDA device");
  if (device < 0) CLC_CUDA(cudaGetDevice(&device));
  if (device >= count) return fail(CLC_ERR_INVALID, "device ordinal out of range");
  p->device = device;
  CLC_CUDA(cudaSetDevice(device));
  // per-device facts are queried once (cudaGetDeviceProperties alone costs about a millisecond, which would dominate
  // the reference-sized calls: 50 frames x 180 points solve in 0.25 ms)
  struct DeviceInfo { bool valid = false; int major = 0, minor = 0, sms = 0; };
  static std::mutex info_mutex;
  static DeviceInfo info[64];
  DeviceInfo di;
  {
    std::lock_guard<std::mutex> lock(info_mutex);
    if (device < 64) di = info[device];
  }
  if (!di.valid) {
    CLC_CUDA(cudaDeviceGetAttribute(&di.major, cudaDevAttrComputeCapabilityMajor, device));
    CLC_CUDA(cudaDeviceGetAttribute(&di.minor, cudaDevAttrComputeCapabilityMinor, device));
    CLC_CUDA(cudaDeviceGetAttribute(&di.sms, cudaDevAttrMultiProcessorCount, device));
    // keep freed device memory in the pool instead of returning it to the driver at every synchronisation
    cudaMemPool_t pool;
    CLC_CUDA(cudaDeviceGetDefaultMemPool(&pool, device));
    uint64_t threshold = UINT64_MAX;
    CLC_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &threshold));
    di.valid = true;
    std::lock_guard<std::mutex> lock(info_mutex);
    if (device < 64) info[device] = di;
  }
  if (di.major < 10)
    return fail(CLC_ERR_CUDA, std::string("libclc_b200 is built for sm_100a only; device is sm_") + std::to_string(di.major) +
                                  std::to_string(di.minor));
  p->num_sms = di.sms;
  CLC_CUDA(cudaStreamCreateWithFlags(&p->stream, cudaStreamNonBlocking));
  return CLC_OK;
}

// Placement of the coordinate arrays relative to each other.  Measured at BASELINE configs[2] (profiles/r2_layout_ab.txt):
// the sweep kernel streams fastest when x, y and z start at the same offset within a 2 MiB page, so that a warp's three
// bulk copies of one stage cross page boundaries together; any other relative shift that was tried costs 3-8 %.  x and y
// live in one allocation, y starting skew_y bytes after the end of x (default: up to the next address congruent to x mod
// 2 MiB; small problems are packed); z is its own allocation (it exists only for non-planar data) whose start is shifted so
// that (z - x) mod 2 MiB == skew_z (default 0).  CLC_SKEW_Y / CLC_SKEW_Z (bytes) override both: the experiment knobs.
int64_t env_skew(const char* name, int64_t dflt) {
  const char* env = std::getenv(name);
  if (!env) return dflt;
  const int64_t v = std::atoll(env);
  return v < 0 ? 0 : (v / 512) * 512;  // bulk copies want 16-byte alignment; keep whole 512-byte units
}
constexpr int64_t kSkewPeriod = (int64_t)2 << 20;

int alloc_z(clc_problem* p) {
  const size_t bytes = sizeof(double) * (size_t)p->n_points_padded;
  CLC_CUDA(cudaMallocAsync(&p->z_block, bytes + (size_t)kSkewPeriod, p->stream));
  const int64_t want = env_skew("CLC_SKEW_Z", 0) % kSkewPeriod;
  const int64_t have = (int64_t)((reinterpret_cast<uintptr_t>(p->z_block) - reinterpret_cast<uintptr_t>(p->x)) % (uintptr_t)kSkewPeriod);
  const int64_t shift = ((want - have) % kSkewPeriod + kSkewPeriod) % kSkewPeriod;
  p->z = reinterpret_cast<double*>(static_cast<char*>(p->z_block) + shift);
  if (std::getenv("CLC_DEBUG_LAYOUT")) std::fprintf(stderr, "CLC_DEBUG_LAYOUT x=%p y=%p z=%p (z block %p)\n", (void*)p->x, (void*)p->y, (void*)p->z, p->z_block);
  return CLC_OK;
}

int alloc_points(clc_problem* p, bool with_z) {
  p->n_points_padded = round_up(p->n_points, clc::kMaxChunk) + clc::kMaxChunk;
  const size_t bytes = sizeof(double) * (size_t)p->n_points_padded;
  const int64_t congruent = (kSkewPeriod - (int64_t)(bytes % (size_t)kSkewPeriod)) % kSkewPeriod;
  const int64_t skew_y = env_skew("CLC_SKEW_Y", bytes >= (size_t)(4 * kSkewPeriod) ? congruent : 0);
  CLC_CUDA(cudaMallocAsync(&p->xy_block, 2 * bytes + (size_t)skew_y, p->stream));
  p->x = static_cast<double*>(p->xy_block);
  p->y = reinterpret_cast<double*>(static_cast<char*>(p->xy_block) + bytes + skew_y);
  if (with_z) {
    int rc = alloc_z(p);
    if (rc != CLC_OK) return rc;
  }
  CLC_CUDA(cudaMallocAsync(&p->d_nonplanar, sizeof(int), p->stream));
  CLC_CUDA(cudaMemsetAsync(p->d_nonplanar, 0, sizeof(int), p->stream));
  // zero the padding (finite values are required beyond the last point)
  const int64_t tail = p->n_points_padded - p->n_points;
  CLC_CUDA(cudaMemsetAsync(p->x + p->n_points, 0, sizeof(double) * tail, p->stream));
  CLC_CUDA(cudaMemsetAsync(p->y + p->n_points, 0, sizeof(double) * tail, p->stream));
  if (with_z) CLC_CUDA(cudaMemsetAsync(p->z + p->n_points, 0, sizeof(double) * tail, p->stream));
  return CLC_OK;
}

// all-zero z stream for the general kernels on planar data (clc_problem_set_planar_mode(p, 0))
int materialise_z(clc_problem* p) {
  if (p->z != nullptr) return CLC_OK;
  int rc = alloc_z(p);
  if (rc != CLC_OK) return rc;
  CLC_CUDA(cudaMemsetAsync(p->z, 0, sizeof(double) * (size_t)p->n_points_padded, p->stream));
  return CLC_OK;
}

}  // namespace

struct clc_group;
extern "C" int clc_problem_destroy(clc_problem* p);
extern "C" int clc_group_create_gather(clc_group** out, const clc_gather_desc* desc, const int* devices, int n_devices);
static clc_problem* group_release_single(clc_group* g);

#include "clc_upload.inl"

extern "C" {

const char* clc_last_error(void) { return g_last_error.c_str(); }

int clc_device_count(int* count) {
  if (!count) return fail(CLC_ERR_INVALID, "count is NULL");
  CLC_CUDA(cudaGetDeviceCount(count));
  return CLC_OK;
}

int64_t clc_launch_count(void) { return g_launches.load(); }

void clc_lm_default_options(clc_lm_options* o) {
  o->max_num_iterations = 100;  // reference src/LaseCamCalCeres.cpp:304
  o->initial_trust_region_radius = 1e4;
  o->max_trust_region_radius = 1e16;
  o->min_trust_region_radius = 1e-32;
  o->min_relative_decrease = 1e-3;
  o->min_lm_diagonal = 1e-6;
  o->max_lm_diagonal = 1e32;
  o->function_tolerance = 1e-6;
  o->gradient_tolerance = 1e-10;
  o->parameter_tolerance = 1e-8;
  o->max_num_consecutive_invalid_steps = 5;
  o->jacobi_scaling = 1;
  o->iterations_per_sync = 8;
  o->reserved = 0;
}

void clc_T_to_pose7(const double T[16], double pose7[7]) {
  const double R[9] = {T[0], T[1], T[2], T[4], T[5], T[6], T[8], T[9], T[10]};
  clc::rot_to_quat(R, pose7 + 3);
  pose7[0] = T[3]; pose7[1] = T[7]; pose7[2] = T[11];
}

void clc_pose7_to_T(const double pose7[7], double T[16]) {
  double R[9];
  clc::quat_to_rot(pose7 + 3, R);
  for (int r = 0; r < 3; ++r) {
    for (int c = 0; c < 3; ++c) T[r * 4 + c] = R[r * 3 + c];
    T[r * 4 + 3] = pose7[r];
  }
  T[12] = T[13] = T[14] = 0.0;
  T[15] = 1.0;
}

int clc_problem_destroy(clc_problem* p) {
  if (!p) return CLC_OK;
  cudaSetDevice(p->device);
  if (p->stream) cudaStreamSynchronize(p->stream);
  if (p->stream) {
    void* bufs[] = {p->xy_block, p->z_block, p->d_nonplanar, p->frame_pose, p->frame_pose_true, p->plane, p->offsets, p->warp_first_frame, p->edge_plane, p->edge_pt,
                    p->partials_ll, p->sums, p->pose, p->launch_seq, p->pose_ll, p->lm, p->flush_buf, p->p2p_error};
    for (void* b : bufs)
      if (b) cudaFreeAsync(b, p->stream);  // back to the device's memory pool: re-creating a problem is cheap
    cudaStreamSynchronize(p->stream);
    cudaStreamDestroy(p->stream);
  }
  if (p->l2_persist_bytes > 0) cudaCtxResetPersistingL2Cache();  // hand the set-aside lines back
  if (p->ev0) cudaEventDestroy(p->ev0);
  if (p->ev1) cudaEventDestroy(p->ev1);
  pinned_release(p->pinned);
  delete p;
  return CLC_OK;
}

// ---- creation from host data: shell (allocations + the small arrays) -> pipelined point upload -> finish ----------------

namespace {

// one shard's worth of the caller's data (all host pointers)
struct HostSource {
  int64_t n_frames = 0;
  const double* frame_pose = nullptr;          // [n_frames*7]
  const int64_t* offsets = nullptr;            // [n_frames+1] prefix local to the shard (offsets[0] == 0)
  const double* const* frame_points = nullptr; // gather: [n_frames] arrays of AoS xyz ...
  const double* flat = nullptr;                // ... or one flat AoS xyz array
  const double* edge_points = nullptr;         // [n_frames*6] or NULL
};

int create_shell(clc_problem** out, const HostSource& src, int use_loss, double cauchy_a, int device, UploadShard* us) {
  *out = nullptr;
  const int64_t N = src.n_frames;
  const int64_t P = N > 0 ? src.offsets[N] : 0;
  clc_problem* p = new clc_problem();
  int rc = init_device(p, device);
  if (rc != CLC_OK) { clc_problem_destroy(p); return rc; }
  p->n_frames = N;
  p->n_points = P;
  p->n_edges = src.edge_points ? 2 * N : 0;
  p->use_loss = use_loss;
  p->cauchy_a = cauchy_a;
  auto body = [&]() -> int {
    // the z stream is created only if a z != 0 turns up (pack path) -- a pinned flat source is laid out by the device
    // kernel that also checks planarity, which needs it from the start
    int rc2 = alloc_points(p, /*with_z=*/false);
    if (rc2 != CLC_OK) return rc2;
    CLC_CUDA(cudaMallocAsync(&p->frame_pose, sizeof(double) * 7 * std::max<int64_t>(N, 1), p->stream));
    CLC_CUDA(cudaMallocAsync(&p->plane, sizeof(double) * 4 * std::max<int64_t>(N, 1), p->stream));
    CLC_CUDA(cudaMallocAsync(&p->offsets, sizeof(int64_t) * (N + 1), p->stream));
    if (N > 0) {
      CLC_CUDA(cudaMemcpyAsync(p->frame_pose, src.frame_pose, sizeof(double) * 7 * N, cudaMemcpyHostToDevice, p->stream));
      CLC_CUDA(cudaMemcpyAsync(p->offsets, src.offsets, sizeof(int64_t) * (N + 1), cudaMemcpyHostToDevice, p->stream));
    } else {
      CLC_CUDA(cudaMemsetAsync(p->offsets, 0, sizeof(int64_t), p->stream));
    }
    if (p->n_edges > 0) {
      CLC_CUDA(cudaMallocAsync(&p->edge_plane, sizeof(double) * 4 * p->n_edges, p->stream));
      CLC_CUDA(cudaMallocAsync(&p->edge_pt, sizeof(double) * 3 * p->n_edges, p->stream));
      // [n_frames*6] front,back == [n_edges*3]
      CLC_CUDA(cudaMemcpyAsync(p->edge_pt, src.edge_points, sizeof(double) * 3 * p->n_edges, cudaMemcpyHostToDevice, p->stream));
    }
    return CLC_OK;
  };
  rc = body();
  if (rc != CLC_OK) { clc_problem_destroy(p); return rc; }
  us->p = p;
  us->frame_points = src.frame_points;
  us->flat = src.flat;
  us->offsets = src.offsets;
  us->n_frames = N;
  *out = p;
  return CLC_OK;
}

int validate_offsets(int64_t N, const int64_t* offsets) {
  if (N > 0 && offsets[0] != 0) return fail(CLC_ERR_INVALID, "offsets[0] must be 0");
  for (int64_t f = 0; f < N; ++f)
    if (offsets[f + 1] < offsets[f]) return fail(CLC_ERR_INVALID, "offsets must be non-decreasing");
  if (N >= ((int64_t)1 << 31)) return fail(CLC_ERR_INVALID, "too many frames");
  return CLC_OK;
}

// uploads and finishes a set of freshly created shells; destroys all of them on failure
int upload_and_finish(std::vector<clc_problem*>& problems, std::vector<UploadShard>& shards) {
  const auto t0 = std::chrono::steady_clock::now();
  int rc = upload_points(shards);
  const auto t1 = std::chrono::steady_clock::now();
  for (size_t g = 0; g < problems.size() && rc == CLC_OK; ++g) {
    cudaSetDevice(problems[g]->device);
    rc = finish_create(problems[g]);
  }
  if (std::getenv("CLC_UPLOAD_TIMING"))
    std::fprintf(stderr, "CLC_UPLOAD_TIMING upload_points_ms=%.3f finish_create_ms=%.3f\n",
                 std::chrono::duration<double, std::milli>(t1 - t0).count(),
                 std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t1).count());
  if (rc != CLC_OK) {
    const std::string msg = g_last_error;
    for (clc_problem* p : problems) clc_problem_destroy(p);
    problems.clear();
    g_last_error = msg;
  }
  return rc;
}

}  // namespace

int clc_problem_create(clc_problem** out, const clc_problem_desc* d) {
  if (!out || !d) return fail(CLC_ERR_INVALID, "NULL argument");
  *out = nullptr;
  if (d->n_frames < 0 || (d->n_frames > 0 && (!d->frame_pose || !d->offsets)))
    return fail(CLC_ERR_INVALID, "frame_pose/offsets missing");
  if (!(d->cauchy_a > 0.0)) return fail(CLC_ERR_INVALID, "cauchy_a must be positive");
  const int64_t N = d->n_frames;
  int rc = validate_offsets(N, d->offsets);
  if (rc != CLC_OK) return rc;
  if (N > 0 && d->offsets[N] > 0 && !d->points) return fail(CLC_ERR_INVALID, "points missing");
  const int64_t zero = 0;
  HostSource src;
  src.n_frames = N;
  src.frame_pose = d->frame_pose;
  src.offsets = N > 0 ? d->offsets : &zero;
  src.flat = d->points;
  src.edge_points = d->edge_points;
  std::vector<clc_problem*> ps(1, nullptr);
  std::vector<UploadShard> us(1);
  rc = create_shell(&ps[0], src, d->use_loss, d->cauchy_a, d->device, &us[0]);
  if (rc != CLC_OK) return rc;
  rc = upload_and_finish(ps, us);
  if (rc != CLC_OK) return rc;
  *out = ps[0];
  return CLC_OK;
}

int clc_problem_create_gather(clc_problem** out, const clc_gather_desc* d) {
  if (!out || !d) return fail(CLC_ERR_INVALID, "NULL argument");
  *out = nullptr;
  clc_group* g = nullptr;
  const int device = d->device;
  int rc = clc_group_create_gather(&g, d, &device, 1);
  if (rc != CLC_OK) return rc;
  *out = group_release_single(g);
  return CLC_OK;
}

int clc_problem_create_synthetic(clc_problem** out, const clc_synthetic_desc* d) {
  if (!out || !d) return fail(CLC_ERR_INVALID, "NULL argument");
  *out = nullptr;
  if (d->frame_begin < 0 || d->frame_end < d->frame_begin || d->frame_end > d->n_frames_total || d->beams <= 0)
    return fail(CLC_ERR_INVALID, "bad frame range / beams");
  if (!(d->cauchy_a > 0.0)) return fail(CLC_ERR_INVALID, "cauchy_a must be positive");
  const int64_t N = d->frame_end - d->frame_begin;
  if (N >= ((int64_t)1 << 31)) return fail(CLC_ERR_INVALID, "too many frames");
  clc_problem* p = new clc_problem();
  int rc = init_device(p, d->device);
  if (rc != CLC_OK) { clc_problem_destroy(p); return rc; }
  p->n_frames = N;
  p->n_points = N * d->beams;
  p->n_edges = d->with_edges ? 2 * N : 0;
  p->use_loss = d->use_loss;
  p->cauchy_a = d->cauchy_a;
  auto body = [&]() -> int {
    // the simulated laser is two-dimensional (calibr_simulation.cpp:82,88): planar by construction, no z stream
    int rc2 = alloc_points(p, /*with_z=*/false);
    if (rc2 != CLC_OK) return rc2;
    CLC_CUDA(cudaMallocAsync(&p->frame_pose, sizeof(double) * 7 * std::max<int64_t>(N, 1), p->stream));
    CLC_CUDA(cudaMallocAsync(&p->plane, sizeof(double) * 4 * std::max<int64_t>(N, 1), p->stream));
    CLC_CUDA(cudaMallocAsync(&p->offsets, sizeof(int64_t) * (N + 1), p->stream));
    if (p->n_edges > 0) {
      CLC_CUDA(cudaMallocAsync(&p->edge_plane, sizeof(double) * 4 * p->n_edges, p->stream));
      CLC_CUDA(cudaMallocAsync(&p->edge_pt, sizeof(double) * 3 * p->n_edges, p->stream));
    }
    clc::CameraDesc cam;
    cam.model = d->camera_model;
    for (int k = 0; k < 8; ++k) cam.intr[k] = d->camera_intrinsics[k];
    cam.pixel_sigma = d->pixel_sigma;
    cam.grid_rows = d->grid_rows;
    cam.grid_cols = d->grid_cols;
    cam.tag_size = d->tag_size;
    cam.tag_spacing = d->tag_spacing;
    if (cam.model != clc::kCameraNone) {
      if (cam.model != clc::kCameraPinholeRadtan && cam.model != clc::kCameraEquidistant)
        return fail(CLC_ERR_INVALID, "unknown camera_model");
      if (cam.grid_rows < 1 || cam.grid_cols < 1 || 4 * cam.grid_rows * cam.grid_cols > 256 || !(cam.tag_size > 0.0) ||
          d->image_width < 1 || d->image_height < 1 || !(cam.intr[0] > 0.0) || !(cam.intr[1] > 0.0))
        return fail(CLC_ERR_INVALID, "bad camera / grid description");
      CLC_CUDA(cudaMallocAsync(&p->frame_pose_true, sizeof(double) * 7 * std::max<int64_t>(N, 1), p->stream));
    }
    if (N > 0) {
      clc::clc_gen_frames_kernel<<<(unsigned)((N + 63) / 64), 64, 0, p->stream>>>(
          d->seed, d->frame_begin, N, d->beams, d->with_edges, cam, d->image_width, d->image_height, p->frame_pose,
          p->frame_pose_true, p->offsets, p->edge_pt);
      CLC_LAUNCH_CHECK();
      clc::clc_gen_points_kernel<<<(unsigned)N, 256, 0, p->stream>>>(d->seed, d->sigma, d->frame_begin, d->beams,
                                                                    p->frame_pose_true ? p->frame_pose_true : p->frame_pose,
                                                                    p->x, p->y, p->z);
      CLC_LAUNCH_CHECK();
    } else {
      CLC_CUDA(cudaMemsetAsync(p->offsets, 0, sizeof(int64_t), p->stream));
    }
    return finish_create(p);
  };
  rc = body();
  if (rc != CLC_OK) { clc_problem_destroy(p); return rc; }
  *out = p;
  return CLC_OK;
}

int clc_problem_sizes(const clc_problem* p, int64_t* n_frames, int64_t* n_points, int* has_edges) {
  if (!p) return fail(CLC_ERR_INVALID, "NULL problem");
  if (n_frames) *n_frames = p->n_frames;
  if (n_points) *n_points = p->n_points;
  if (has_edges) *has_edges = p->n_edges > 0;
  return CLC_OK;
}

int clc_problem_download_true_poses(const clc_problem* p, double* frame_pose_true) {
  if (!p || !frame_pose_true) return fail(CLC_ERR_INVALID, "NULL argument");
  int rc = set_device(p);
  if (rc != CLC_OK) return rc;
  CLC_CUDA(cudaStreamSynchronize(p->stream));
  if (p->n_frames > 0)
    CLC_CUDA(cudaMemcpy(frame_pose_true, p->frame_pose_true ? p->frame_pose_true : p->frame_pose,
                        sizeof(double) * 7 * p->n_frames, cudaMemcpyDeviceToHost));
  return CLC_OK;
}

int clc_problem_algorithmic_bytes(const clc_problem* p, int64_t* bytes) {
  if (!p || !bytes) return fail(CLC_ERR_INVALID, "NULL argument");
  *bytes = 24 * p->n_points + 40 * p->n_frames + 56 * p->n_edges + 224;
  return CLC_OK;
}

int clc_problem_streamed_bytes(const clc_problem* p, int64_t* bytes) {
  if (!p || !bytes) return fail(CLC_ERR_INVALID, "NULL argument");
  *bytes = (p->planar ? 16 : 24) * p->n_points + 40 * p->n_frames + 56 * p->n_edges + 224;
  return CLC_OK;
}

int clc_problem_set_planar_mode(clc_problem* p, int mode) {
  if (!p) return fail(CLC_ERR_INVALID, "NULL problem");
  if (mode != 0 && mode != 1) return fail(CLC_ERR_INVALID, "planar mode must be 0 or 1");
  int rc = set_device(p);
  if (rc != CLC_OK) return rc;
  p->planar_mode = mode;
  const bool planar = p->z_all_zero && mode != 0 && p->n_points >= p->planar_min_points;
  if (planar == p->planar) return CLC_OK;
  CLC_CUDA(cudaStreamSynchronize(p->stream));
  p->planar = planar;
  if (!p->planar) {
    rc = materialise_z(p);
    if (rc != CLC_OK) return rc;
  }
  return partition(p);
}

int clc_problem_download(const clc_problem* p, double* frame_pose, int64_t* offsets, double* points,
                         double* edge_points, double* planes) {
  if (!p) return fail(CLC_ERR_INVALID, "NULL problem");
  int rc = set_device(p);
  if (rc != CLC_OK) return rc;
  CLC_CUDA(cudaStreamSynchronize(p->stream));
  if (frame_pose && p->n_frames > 0)
    CLC_CUDA(cudaMemcpy(frame_pose, p->frame_pose, sizeof(double) * 7 * p->n_frames, cudaMemcpyDeviceToHost));
  if (offsets) CLC_CUDA(cudaMemcpy(offsets, p->offsets, sizeof(int64_t) * (p->n_frames + 1), cudaMemcpyDeviceToHost));
  if (planes && p->n_frames > 0)
    CLC_CUDA(cudaMemcpy(planes, p->plane, sizeof(double) * 4 * p->n_frames, cudaMemcpyDeviceToHost));
  if (edge_points && p->n_edges > 0)
    CLC_CUDA(cudaMemcpy(edge_points, p->edge_pt, sizeof(double) * 3 * p->n_edges, cudaMemcpyDeviceToHost));
  if (points && p->n_points > 0) {
    double* aos = nullptr;
    CLC_CUDA(cudaMallocAsync(&aos, sizeof(double) * 3 * p->n_points, p->stream));
    clc::clc_soa_to_aos_kernel<<<(unsigned)((p->n_points + 255) / 256), 256, 0, p->stream>>>(p->x, p->y, p->z, 0,
                                                                                          p->n_points, aos);
    g_launches.fetch_add(1);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(points, aos, sizeof(double) * 3 * p->n_points, cudaMemcpyDeviceToHost, p->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(p->stream);
    cudaFreeAsync(aos, p->stream);
    if (e != cudaSuccess) return fail(CLC_ERR_CUDA, cudaGetErrorString(e));
  }
  return CLC_OK;
}

// ---- evaluation -------------------------------------------------------------------------------------------------
// Every collective operation is split into an enqueue phase and a wait phase, so that ONE host thread can drive the
// shards of an in-process multi-GPU group: enqueue on every device first (the fused exchange makes block 0 of every
// device's kernel wait for its peers' kernels), then wait for all of them.

static int eval_enqueue(clc_problem* p, const double pose7[7], bool loss, bool edges, int mode, int count) {
  int rc = set_device(p);
  if (rc != CLC_OK) return rc;
  double* h_pose = p->pinned->pose;  // pinned: the copy below is truly asynchronous
  if (mode == clc::kModeLM) {
    if (!pose7) return fail(CLC_ERR_INVALID, "pose7 is NULL");
    for (int i = 0; i < 7; ++i) h_pose[i] = pose7[i];
  } else {
    const double ident[7] = {0, 0, 0, 0, 0, 0, 1};
    for (int i = 0; i < 7; ++i) h_pose[i] = ident[i];
  }
  CLC_CUDA(cudaMemcpyAsync(p->pose, h_pose, sizeof(double) * 7, cudaMemcpyHostToDevice, p->stream));
  const bool with_edges = edges && p->n_edges > 0;
  if (mode == clc::kModeLM && p->small_kernel && p->nranks <= 1 &&
      p->n_points + (with_edges ? p->n_edges : 0) <= clc::kSmallMaxResiduals) {
    // a small problem: one evaluation by the one-cluster kernel (clc_small.cuh)
    const clc::ProblemView v = make_view(p);
    if (loss)
      clc::clc_small_lm_kernel<true, true><<<clc::kSmallCluster, clc::kSmallThreads, 0, p->stream>>>(v, nullptr, 1, with_edges ? 1 : 0, p->pose, p->sums);
    else
      clc::clc_small_lm_kernel<false, true><<<clc::kSmallCluster, clc::kSmallThreads, 0, p->stream>>>(v, nullptr, 1, with_edges ? 1 : 0, p->pose, p->sums);
    CLC_LAUNCH_CHECK();
  } else {
    rc = launch_sweep(p, mode, loss, edges, p->pose, nullptr, nullptr);
    if (rc != CLC_OK) return rc;
  }
  rc = allreduce_sums(p, count);
  if (rc != CLC_OK) return rc;
  CLC_CUDA(cudaMemcpyAsync(p->h_sums, p->sums, sizeof(double) * count, cudaMemcpyDeviceToHost, p->stream));
  return CLC_OK;
}

static int eval_wait(clc_problem* p) {
  int rc = set_device(p);
  if (rc != CLC_OK) return rc;
  CLC_CUDA(sync_stream_low_latency(p->stream));
  return check_p2p_error(p);
}

// runs one sweep on every shard of `ps` (a single problem, or the shards of a group); afterwards ps[0]->h_sums holds the
// (all-reduced) sums
static int eval_all(clc_problem* const* ps, int n, const double pose7[7], int which /*0 eval, 1 information, 2 closed form*/) {
  int first_rc = CLC_OK;
  for (int g = 0; g < n; ++g) {
    clc_problem* p = ps[g];
    int rc;
    if (which == 0) rc = eval_enqueue(p, pose7, p->use_loss != 0, p->n_edges > 0, clc::kModeLM, clc::kNumSums);
    else if (which == 1) rc = eval_enqueue(p, pose7, false, false, clc::kModeLM, clc::kNumSums);  // reference :318-381: no loss, no edges
    else rc = eval_enqueue(p, nullptr, false, false, clc::kModeClosedForm, clc::kMaxOut);
    if (rc != CLC_OK && first_rc == CLC_OK) first_rc = rc;
  }
  for (int g = 0; g < n; ++g) {
    const int rc = eval_wait(ps[g]);
    if (rc != CLC_OK && first_rc == CLC_OK) first_rc = rc;
  }
  return first_rc;
}

static void unpack_H(const double* sums, double* H36) {
  int k = 0;
  for (int i = 0; i < 6; ++i)
    for (int j = i; j < 6; ++j) {
      H36[i * 6 + j] = sums[k];
      H36[j * 6 + i] = sums[k];
      ++k;
    }
}

static void eval_post(const double* sums, double H36[36], double g6[6], double* cost) {
  if (H36) unpack_H(sums, H36);
  if (g6) for (int i = 0; i < 6; ++i) g6[i] = sums[21 + i];
  if (cost) *cost = sums[27];
}

static void information_post(const double* sums, double H36[36], double b6[6], double* chi, double sv6[6], double V36[36]) {
  double H[36];
  unpack_H(sums, H);
  if (H36) std::memcpy(H36, H, sizeof(H));
  if (b6) for (int i = 0; i < 6; ++i) b6[i] = -sums[21 + i];
  if (chi) *chi = 2.0 * sums[27];
  if (sv6 || V36) {
    // H is symmetric: singular values = |eigenvalues|, right singular vectors = eigenvectors (Eigen::JacobiSVD, :366)
    double w[6], V[36];
    sym_eig<6>(H, w, V);
    int order[6] = {0, 1, 2, 3, 4, 5};
    std::sort(order, order + 6, [&](int a, int b) { return std::fabs(w[a]) > std::fabs(w[b]); });
    for (int c = 0; c < 6; ++c) {
      if (sv6) sv6[c] = std::fabs(w[order[c]]);
      if (V36)
        for (int r = 0; r < 6; ++r) V36[r * 6 + c] = V[r * 6 + order[c]];
    }
  }
}

static void closed_form_post(const double* sums, double Tlc[16], int* unobservable, double AtA81[81], double Atb9[9]) {
  double AtA[81], Atb[9];
  int k = 0;
  for (int i = 0; i < 9; ++i)
    for (int j = i; j < 9; ++j) {
      AtA[i * 9 + j] = sums[k];
      AtA[j * 9 + i] = sums[k];
      ++k;
    }
  for (int i = 0; i < 9; ++i) Atb[i] = sums[45 + i];
  if (AtA81) std::memcpy(AtA81, AtA, sizeof(AtA));
  if (Atb9) std::memcpy(Atb9, Atb, sizeof(Atb));
  double sv[9];
  sym_singular_values<9>(AtA, sv);
  int unobs = 0;
  for (int i = 0; i < 9; ++i)
    if (sv[i] < 1e-10) unobs = 1;  // reference :165-171
  if (unobservable) *unobservable = unobs;
  double h[9];
  ldlt9_solve(AtA, Atb, h);  // reference :181
  const double* h1 = h;
  const double* h2 = h + 3;
  const double* h3 = h + 6;
  double h12[3];
  clc::cross3(h1, h2, h12);
  // Rlc = [h1 h2 h1xh2]^T (rows), tlc = -Rlc h3 before orthogonalisation (reference :187-192)
  const double Rlc[9] = {h1[0], h1[1], h1[2], h2[0], h2[1], h2[2], h12[0], h12[1], h12[2]};
  double tlc[3];
  for (int r = 0; r < 3; ++r) tlc[r] = -(Rlc[r * 3] * h3[0] + Rlc[r * 3 + 1] * h3[1] + Rlc[r * 3 + 2] * h3[2]);
  // U V^T of Rlc (reference :195-196) = Rlc (Rlc^T Rlc)^(-1/2); no determinant check, as in the reference
  double G[9], w[3], V[9], S[9], Ro[9];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) G[i * 3 + j] = Rlc[i] * Rlc[j] + Rlc[3 + i] * Rlc[3 + j] + Rlc[6 + i] * Rlc[6 + j];
  sym_eig<3>(G, w, V);
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) {
      double s = 0.0;
      for (int q = 0; q < 3; ++q) s += V[i * 3 + q] * (1.0 / std::sqrt(w[q])) * V[j * 3 + q];
      S[i * 3 + j] = s;
    }
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) Ro[i * 3 + j] = Rlc[i * 3] * S[j] + Rlc[i * 3 + 1] * S[3 + j] + Rlc[i * 3 + 2] * S[6 + j];
  for (int i = 0; i < 16; ++i) Tlc[i] = 0.0;
  for (int r = 0; r < 3; ++r) {
    for (int c = 0; c < 3; ++c) Tlc[r * 4 + c] = Ro[r * 3 + c];
    Tlc[r * 4 + 3] = tlc[r];
  }
  Tlc[15] = 1.0;
}

int clc_eval(clc_problem* p, const double pose7[7], double H36[36], double g6[6], double* cost) {
  if (!p) return fail(CLC_ERR_INVALID, "NULL problem");
  int rc = eval_all(&p, 1, pose7, 0);
  if (rc != CLC_OK) return rc;
  eval_post(p->h_sums, H36, g6, cost);
  return CLC_OK;
}

int clc_information(clc_problem* p, const double pose7[7], double H36[36], double b6[6], double* chi, double sv6[6],
                    double V36[36]) {
  if (!p) return fail(CLC_ERR_INVALID, "NULL problem");
  int rc = eval_all(&p, 1, pose7, 1);
  if (rc != CLC_OK) return rc;
  information_post(p->h_sums, H36, b6, chi, sv6, V36);
  return CLC_OK;
}

int clc_closed_form(clc_problem* p, double Tlc[16], int* unobservable, double AtA81[81], double Atb9[9]) {
  if (!p || !Tlc) return fail(CLC_ERR_INVALID, "NULL argument");
  int rc = eval_all(&p, 1, nullptr, 2);
  if (rc != CLC_OK) return rc;
  closed_form_post(p->h_sums, Tlc, unobservable, AtA81, Atb9);
  return CLC_OK;
}

// ---- the on-device LM solve ------------------------------------------------------------------------------------

namespace {

struct SolveCtx {
  clc_lm_options opt;
  int max_sweeps = 0;
  int launched = 0;
  bool fused_update = true, loss = true, edges = false;
};

// L2 residency across LM iterations: every iteration re-reads the same coordinate arrays.  When they are not much larger than
// the 126 MB L2, a persisting access-policy window over the x,y block keeps a hash-selected share of their lines (hitRatio =
// set-aside / window) resident from one sweep to the next, so that share is not fetched from HBM again.  The set-aside is a
// device-wide limit: it is raised on first use and left in place.  Only the solve loop runs under the window; the measurement
// hook clc_bench_eval (L2 flushed between launches: the 24 B / 16 B roofline rows) does not.
int l2_window(clc_problem* p, bool on) {
  if (p->l2_persist_bytes <= 0 || !p->xy_block) return CLC_OK;
  if (on == p->l2_window_set) return CLC_OK;
  cudaStreamAttrValue attr;
  std::memset(&attr, 0, sizeof(attr));
  if (on) {
    int max_persist = 0, max_window = 0;
    CLC_CUDA(cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, p->device));
    CLC_CUDA(cudaDeviceGetAttribute(&max_window, cudaDevAttrMaxAccessPolicyWindowSize, p->device));
    const size_t set_aside = (size_t)std::min<int64_t>(p->l2_persist_bytes, max_persist);
    if (set_aside == 0 || max_window <= 0) return CLC_OK;
    size_t cur = 0;
    CLC_CUDA(cudaDeviceGetLimit(&cur, cudaLimitPersistingL2CacheSize));
    if (cur < set_aside) CLC_CUDA(cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, set_aside));
    const size_t span = sizeof(double) * (size_t)(p->y - p->x) + sizeof(double) * (size_t)p->n_points;  // x .. end of y
    const size_t window = std::min(span, (size_t)max_window);
    attr.accessPolicyWindow.base_ptr = p->xy_block;
    attr.accessPolicyWindow.num_bytes = window;
    attr.accessPolicyWindow.hitRatio = (float)std::min(1.0, (double)set_aside / (double)window);
    attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
    attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
  } else {
    attr.accessPolicyWindow.num_bytes = 0;  // disables the window for later launches on the stream
  }
  CLC_CUDA(cudaStreamSetAttribute(p->stream, cudaStreamAttributeAccessPolicyWindow, &attr));
  p->l2_window_set = on;
  return CLC_OK;
}

int solve_begin(clc_problem* p, const double pose7[7], const clc_lm_options& opt, SolveCtx* ctx) {
  int rc = set_device(p);
  if (rc != CLC_OK) return rc;
  rc = l2_window(p, true);
  if (rc != CLC_OK) return rc;
  ctx->opt = opt;
  clc::lm_init(&p->h_lm->core, pose7, opt);
  if (!p->ev0) CLC_CUDA(cudaEventCreate(&p->ev0));  // kept for the life of the problem (destroyed with it)
  if (!p->ev1) CLC_CUDA(cudaEventCreate(&p->ev1));
  if (p->p2p_error) CLC_CUDA(cudaMemsetAsync(p->p2p_error, 0, sizeof(int), p->stream));  // a fresh solve starts clean
  CLC_CUDA(cudaMemcpyAsync(&p->lm->core, &p->h_lm->core, sizeof(clc::LmCore), cudaMemcpyHostToDevice, p->stream));
  CLC_CUDA(cudaEventRecord(p->ev0, p->stream));
  ctx->fused_update = (p->nranks <= 1) || p->allreduce_mode == 1;
  ctx->loss = p->use_loss != 0;
  ctx->edges = p->n_edges > 0;
  // every LM iteration needs exactly one sweep; invalid steps need none -> at most max_iterations + 1 sweeps
  ctx->max_sweeps = opt.max_num_iterations + 2;
  ctx->launched = 0;
  *p->h_done = 0;
  return CLC_OK;
}

// one LM iteration: the fused sweep (+ NCCL all-reduce and the LM kernel when the exchange is not fused)
int solve_launch_one(clc_problem* p, SolveCtx* ctx, int loop_sweeps = 1) {
  int rc = set_device(p);
  if (rc != CLC_OK) return rc;
  // fused mode: one kernel per LM iteration, chained with programmatic dependent launch (the next sweep prefetches
  // its first stages while this one's block 0 reduces and updates)
  rc = launch_sweep(p, clc::kModeLM, ctx->loss, ctx->edges, p->lm->core.cand, &p->lm->core.done,
                    ctx->fused_update ? p->lm : nullptr, /*collective=*/true, /*pdl=*/ctx->fused_update && p->use_pdl, loop_sweeps);
  if (rc != CLC_OK) return rc;
  if (!ctx->fused_update) {
    rc = allreduce_sums(p, clc::kNumSums);
    if (rc != CLC_OK) return rc;
    clc::clc_lm_kernel<<<1, 32, 0, p->stream>>>(p->lm, p->sums);
    CLC_LAUNCH_CHECK();
  }
  ctx->launched++;
  return CLC_OK;
}

int solve_poll_enqueue(clc_problem* p) {
  int rc = set_device(p);
  if (rc != CLC_OK) return rc;
  CLC_CUDA(cudaMemcpyAsync(p->h_done, &p->lm->core.done, sizeof(int), cudaMemcpyDeviceToHost, p->stream));
  return CLC_OK;
}

int solve_finish(clc_problem* p, double pose7[7], clc_lm_summary* summary, clc_lm_iteration* trace, int trace_cap) {
  int rc = set_device(p);
  if (rc != CLC_OK) return rc;
  CLC_CUDA(cudaEventRecord(p->ev1, p->stream));
  rc = l2_window(p, false);
  if (rc != CLC_OK) return rc;
  CLC_CUDA(cudaMemcpyAsync(p->h_lm, p->lm, sizeof(clc::LmState), cudaMemcpyDeviceToHost, p->stream));
  CLC_CUDA(sync_stream_low_latency(p->stream));
  float ms = 0.f;
  CLC_CUDA(cudaEventElapsedTime(&ms, p->ev0, p->ev1));
  rc = check_p2p_error(p);
  if (rc != CLC_OK) return rc;
  const clc::LmCore& s = p->h_lm->core;
  const clc_lm_iteration* dev_trace = p->h_lm->trace;
  if (pose7)
    for (int i = 0; i < 7; ++i) pose7[i] = s.x[i];  // the last accepted point (a terminating candidate is not applied)
  if (summary) {
    summary->termination = s.done ? s.done : CLC_TERM_NO_CONVERGENCE;
    summary->num_iterations = s.n_trace;
    summary->num_successful_steps = s.num_successful;
    summary->num_unsuccessful_steps = s.num_unsuccessful;
    summary->num_sweeps = s.sweeps;
    summary->reserved = 0;
    summary->initial_cost = s.initial_cost;
    summary->final_cost = s.x_cost;
    summary->device_ms = ms;
  }
  if (trace) {
    const int n = std::min(std::min(s.n_trace, clc::kTraceMax), trace_cap);
    for (int i = 0; i < n; ++i) trace[i] = dev_trace[i];
  }
  return CLC_OK;
}

// the whole solve over the shards `ps` (n == 1: a plain problem, possibly one rank of a multi-process job)
int solve_all(clc_problem* const* ps, int n, double pose7[7], const clc_lm_options* opt_in, clc_lm_summary* summary,
              clc_lm_iteration* trace, int trace_cap) {
  clc_lm_options opt;
  if (opt_in) opt = *opt_in; else clc_lm_default_options(&opt);
  if (opt.max_num_iterations < 0) return fail(CLC_ERR_INVALID, "max_num_iterations < 0");
  if (opt.iterations_per_sync < 1) opt.iterations_per_sync = 1;
  std::vector<SolveCtx> ctx((size_t)n);
  int rc = CLC_OK;
  for (int g = 0; g < n && rc == CLC_OK; ++g) rc = solve_begin(ps[g], pose7, opt, &ctx[g]);
  if (rc != CLC_OK) return rc;
  const int max_sweeps = ctx[0].max_sweeps;
  int launched = 0;
  // Small problems (the reference's own sizes): the whole solve in one launch of one thread-block cluster that keeps every
  // residual in registers (clc_small.cuh) -- no TMA rings, no gather, no global round trip between two LM iterations.
  if (n == 1 && ps[0]->small_kernel && ps[0]->loop_in_kernel >= 1 && ps[0]->nranks <= 1 && ctx[0].fused_update &&
      ps[0]->n_points + (ctx[0].edges ? ps[0]->n_edges : 0) <= clc::kSmallMaxResiduals) {
    clc_problem* p = ps[0];
    rc = set_device(p);
    if (rc != CLC_OK) return rc;
    const clc::ProblemView v = make_view(p);
    if (ctx[0].loss)
      clc::clc_small_lm_kernel<true><<<clc::kSmallCluster, clc::kSmallThreads, 0, p->stream>>>(v, p->lm, max_sweeps, ctx[0].edges ? 1 : 0, nullptr, nullptr);
    else
      clc::clc_small_lm_kernel<false><<<clc::kSmallCluster, clc::kSmallThreads, 0, p->stream>>>(v, p->lm, max_sweeps, ctx[0].edges ? 1 : 0, nullptr, nullptr);
    CLC_LAUNCH_CHECK();
    launched = max_sweeps;
  }
  bool loop_launch = launched == 0;
  for (int g = 0; g < n; ++g)
    loop_launch = loop_launch && ctx[g].fused_update &&
                  (ps[g]->loop_in_kernel >= 2 || (ps[g]->loop_in_kernel == 1 && ps[g]->grid == 1 && ps[g]->nranks <= 1));
  if (loop_launch) {
    // ONE launch per device runs the whole LM loop (sweep, reduce, [peer exchange,] lm_update, next sweep)
    for (int g = 0; g < n; ++g) {
      rc = solve_launch_one(ps[g], &ctx[g], max_sweeps);
      if (rc != CLC_OK) return rc;
    }
    launched = max_sweeps;
  }
  while (launched < max_sweeps) {
    // the first batch is twice as long: a solve from the identity or from the closed form takes 6-16 sweeps (reference sizes and
    // BASELINE configs alike), and every host poll in the middle of a solve stalls the device for longer than the two or three
    // no-op sweeps a too-long batch costs (3 us each; profiles/r2_loop_modes2.txt)
    const int batch = std::min(launched == 0 ? 2 * opt.iterations_per_sync : opt.iterations_per_sync, max_sweeps - launched);
    // iteration-major order: sweep i of every shard is queued before sweep i+1 of any, so no device's queue can fill up
    // with kernels that wait for a peer whose launches have not been issued yet
    for (int i = 0; i < batch; ++i)
      for (int g = 0; g < n; ++g) {
        rc = solve_launch_one(ps[g], &ctx[g]);
        if (rc != CLC_OK) return rc;
      }
    launched += batch;
    for (int g = 0; g < n; ++g) {
      rc = solve_poll_enqueue(ps[g]);
      if (rc != CLC_OK) return rc;
    }
    bool all_done = true;
    for (int g = 0; g < n; ++g) {
      rc = set_device(ps[g]);
      if (rc != CLC_OK) return rc;
      CLC_CUDA(sync_stream_low_latency(ps[g]->stream));
      all_done = all_done && (*ps[g]->h_done != 0);
    }
    if (all_done) break;
  }
  double ms_max = 0.0;
  int first_rc = CLC_OK;
  for (int g = n - 1; g >= 0; --g) {  // shard 0 last: its pose / summary / trace are the ones returned (all shards agree)
    clc_lm_summary sg;
    rc = solve_finish(ps[g], g == 0 ? pose7 : nullptr, &sg, g == 0 ? trace : nullptr, trace_cap);
    if (rc != CLC_OK && first_rc == CLC_OK) first_rc = rc;
    if (rc == CLC_OK) {
      ms_max = std::max(ms_max, sg.device_ms);
      if (g == 0 && summary) *summary = sg;
    }
  }
  if (first_rc != CLC_OK) return first_rc;
  if (summary) summary->device_ms = ms_max;
  return CLC_OK;
}

}  // namespace

int clc_solve_lm(clc_problem* p, double pose7[7], const clc_lm_options* opt_in, clc_lm_summary* summary,
                 clc_lm_iteration* trace, int trace_cap) {
  if (!p || !pose7) return fail(CLC_ERR_INVALID, "NULL argument");
  return solve_all(&p, 1, pose7, opt_in, summary, trace, trace_cap);
}

// ---- LineFittingCeres, batched ------------------------------------------------------------------------------------

int clc_problem_line_fit(clc_problem* p, double* lines, int max_num_iterations, double* info) {
  if (!p || !lines || max_num_iterations < 0) return fail(CLC_ERR_INVALID, "bad line-fit arguments");
  int rc = set_device(p);
  if (rc != CLC_OK) return rc;
  const int64_t N = p->n_frames;
  if (N == 0) return CLC_OK;
  double *d_lines = nullptr, *d_info = nullptr;
  cudaError_t e = cudaMallocAsync(&d_lines, sizeof(double) * 2 * N, p->stream);
  if (e == cudaSuccess && info) e = cudaMallocAsync(&d_info, sizeof(double) * 4 * N, p->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_lines, lines, sizeof(double) * 2 * N, cudaMemcpyHostToDevice, p->stream);
  if (e == cudaSuccess) {
    const int warps = 8;
    clc::clc_line_fit_kernel<<<(unsigned)((N + warps - 1) / warps), warps * 32, 0, p->stream>>>(
        p->x, p->y, p->offsets, N, max_num_iterations, p->cauchy_a, d_lines, d_info);
    g_launches.fetch_add(1);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaMemcpyAsync(lines, d_lines, sizeof(double) * 2 * N, cudaMemcpyDeviceToHost, p->stream);
  if (e == cudaSuccess && info) e = cudaMemcpyAsync(info, d_info, sizeof(double) * 4 * N, cudaMemcpyDeviceToHost, p->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(p->stream);
  if (d_lines) cudaFreeAsync(d_lines, p->stream);
  if (d_info) cudaFreeAsync(d_info, p->stream);
  if (e != cudaSuccess) return fail(CLC_ERR_CUDA, cudaGetErrorString(e));
  return CLC_OK;
}

// One scan per call, as the reference calls it (main/calibr_offline.cpp:124, a few hundred points): no problem object, no
// layout kernels -- a per-thread cache of one stream, one device buffer and one pinned scratch, three driver calls and a
// one-warp kernel on the scan's own AoS array.
namespace {
struct LineFitCache {
  int device = -1;
  cudaStream_t stream = nullptr;
  double* d_pts = nullptr;   // [capacity * 3] + 2 (the line)
  int64_t capacity = 0;
  double* h_line = nullptr;  // pinned, 2 doubles
  ~LineFitCache() {
    if (device < 0) return;
    // no CUDA calls at thread exit: the context may already be gone; the few KB are reclaimed with the process
  }
};
thread_local LineFitCache g_line_cache;
}  // namespace

int clc_line_fit_points(const double* points_xyz, int64_t n, double line[2], int max_num_iterations) {
  if (!points_xyz || n < 0 || !line || max_num_iterations < 0) return fail(CLC_ERR_INVALID, "bad line-fit arguments");
  LineFitCache& c = g_line_cache;
  int device = 0;
  CLC_CUDA(cudaGetDevice(&device));
  if (c.device != device) {
    int major = 0;
    CLC_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
    if (major < 10) return fail(CLC_ERR_CUDA, "libclc_b200 is built for sm_100a only");
    if (c.stream) { cudaStreamDestroy(c.stream); c.stream = nullptr; }
    if (c.d_pts) { cudaFree(c.d_pts); c.d_pts = nullptr; c.capacity = 0; }
    CLC_CUDA(cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking));
    if (!c.h_line) CLC_CUDA(cudaMallocHost(&c.h_line, 2 * sizeof(double)));
    c.device = device;
  }
  if (n > c.capacity) {
    if (c.d_pts) CLC_CUDA(cudaFree(c.d_pts));
    c.d_pts = nullptr;
    c.capacity = std::max<int64_t>(2 * n, 4096);
    CLC_CUDA(cudaMalloc(&c.d_pts, sizeof(double) * (3 * (size_t)c.capacity + 2)));
  }
  double* d_line = c.d_pts + 3 * c.capacity;
  c.h_line[0] = line[0];
  c.h_line[1] = line[1];
  if (n > 0) CLC_CUDA(cudaMemcpyAsync(c.d_pts, points_xyz, sizeof(double) * 3 * (size_t)n, cudaMemcpyHostToDevice, c.stream));
  CLC_CUDA(cudaMemcpyAsync(d_line, c.h_line, 2 * sizeof(double), cudaMemcpyHostToDevice, c.stream));
  clc::clc_line_fit_single_kernel<<<1, 32, 0, c.stream>>>(c.d_pts, n, max_num_iterations, 0.05, d_line);  // CauchyLoss(0.05), reference :416
  CLC_LAUNCH_CHECK();
  CLC_CUDA(cudaMemcpyAsync(c.h_line, d_line, 2 * sizeof(double), cudaMemcpyDeviceToHost, c.stream));
  CLC_CUDA(cudaStreamSynchronize(c.stream));
  line[0] = c.h_line[0];
  line[1] = c.h_line[1];
  return CLC_OK;
}

int clc_scan_segments(const float* ranges, int64_t n_scans, int64_t n_beams, double angle_min, double angle_increment,
                      double range_min, int32_t* seg_start, int32_t* seg_end, int device) {
  if (!ranges || n_scans < 0 || n_beams < 0 || !seg_start || !seg_end) return fail(CLC_ERR_INVALID, "bad scan arguments");
  if (n_scans == 0) return CLC_OK;
  int count = 0;
  CLC_CUDA(cudaGetDeviceCount(&count));
  if (device < 0) CLC_CUDA(cudaGetDevice(&device));
  if (device >= count) return fail(CLC_ERR_INVALID, "device ordinal out of range");
  CLC_CUDA(cudaSetDevice(device));
  float* d_r = nullptr;
  int *d_s = nullptr, *d_e = nullptr;
  cudaStream_t st;
  CLC_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
  cudaError_t e = cudaMallocAsync(&d_r, sizeof(float) * (size_t)n_scans * (size_t)std::max<int64_t>(n_beams, 1), st);
  if (e == cudaSuccess) e = cudaMallocAsync(&d_s, sizeof(int) * n_scans, st);
  if (e == cudaSuccess) e = cudaMallocAsync(&d_e, sizeof(int) * n_scans, st);
  if (e == cudaSuccess && n_beams > 0)
    e = cudaMemcpyAsync(d_r, ranges, sizeof(float) * (size_t)n_scans * (size_t)n_beams, cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) {
    clc::clc_scan_segments_kernel<<<(unsigned)((n_scans + 127) / 128), 128, 0, st>>>(d_r, n_scans, n_beams, angle_min,
                                                                                   angle_increment, range_min, d_s, d_e);
    g_launches.fetch_add(1);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaMemcpyAsync(seg_start, d_s, sizeof(int) * n_scans, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaMemcpyAsync(seg_end, d_e, sizeof(int) * n_scans, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (d_r) cudaFreeAsync(d_r, st);
  if (d_s) cudaFreeAsync(d_s, st);
  if (d_e) cudaFreeAsync(d_e, st);
  cudaStreamSynchronize(st);
  cudaStreamDestroy(st);
  if (e != cudaSuccess) return fail(CLC_ERR_CUDA, cudaGetErrorString(e));
  return CLC_OK;
}

// ---- the offline driver's scan loop on the device (clc_scans.cuh) --------------------------------------------------

namespace {
struct ScanStats {
  float ms[6] = {};
  int64_t bytes_h2d = 0, bytes_d2h = 0;
};
thread_local ScanStats g_scan_stats;

// an empty problem on `device` with its stream: the caller fills the sizes and allocates
int scan_problem_shell(clc_problem** out, const clc_scan_desc* d) {
  clc_problem* p = new clc_problem();
  *out = p;
  int rc = init_device(p, d->device);
  if (rc != CLC_OK) return rc;
  p->use_loss = d->use_loss;
  p->cauchy_a = d->cauchy_a;
  // a 2-D laser: every z is 0 by construction, no z stream to scan (finish_create materialises an all-zero one only
  // for the general kernels, below the planar size rule)
  p->z_all_zero = true;
  p->host_planarity_known = true;
  return CLC_OK;
}

// the arrays of a problem of N frames and P points (as create_shell allocates them)
int scan_problem_alloc(clc_problem* p, int64_t N, int64_t P, bool with_edges) {
  p->n_frames = N;
  p->n_points = P;
  p->n_edges = with_edges ? 2 * N : 0;
  int rc = alloc_points(p, /*with_z=*/false);
  if (rc != CLC_OK) return rc;
  CLC_CUDA(cudaMallocAsync(&p->frame_pose, sizeof(double) * 7 * std::max<int64_t>(N, 1), p->stream));
  CLC_CUDA(cudaMallocAsync(&p->plane, sizeof(double) * 4 * std::max<int64_t>(N, 1), p->stream));
  CLC_CUDA(cudaMallocAsync(&p->offsets, sizeof(int64_t) * (N + 1), p->stream));
  CLC_CUDA(cudaMemsetAsync(p->offsets, 0, sizeof(int64_t), p->stream));
  if (p->n_edges > 0) {
    CLC_CUDA(cudaMallocAsync(&p->edge_plane, sizeof(double) * 4 * p->n_edges, p->stream));
    CLC_CUDA(cudaMallocAsync(&p->edge_pt, sizeof(double) * 3 * p->n_edges, p->stream));
  }
  return CLC_OK;
}
}  // namespace

int clc_problems_create_from_scans(const clc_scan_desc* d, clc_problem** points_out, clc_problem** on_line_out,
                                   int32_t* scan_info, double* scan_line) {
  if (points_out) *points_out = nullptr;
  if (on_line_out) *on_line_out = nullptr;
  if (!d) return fail(CLC_ERR_INVALID, "NULL scan description");
  const int64_t S = d->n_scans, B = d->n_beams, K = d->n_poses;
  if (S < 0 || B < 0 || K < 0) return fail(CLC_ERR_INVALID, "negative scan / beam / pose count");
  if (B > INT32_MAX) return fail(CLC_ERR_INVALID, "n_beams exceeds INT32_MAX (beam indices are int32)");
  if (S >= ((int64_t)1 << 31)) return fail(CLC_ERR_INVALID, "too many scans (frame indices are int32)");
  if (S > 0 && B > 0 && !d->ranges) return fail(CLC_ERR_INVALID, "ranges is NULL");
  if (S > 0 && !d->scan_stamp) return fail(CLC_ERR_INVALID, "scan_stamp is NULL");
  if (K > 0 && (!d->pose_stamp || !d->pose_wc)) return fail(CLC_ERR_INVALID, "pose_stamp / pose_wc is NULL");
  if (!clc::is_finite(d->angle_increment)) return fail(CLC_ERR_INVALID, "angle_increment must be finite");
  if (!(d->max_dt > 0.0)) return fail(CLC_ERR_INVALID, "max_dt must be positive");
  if (!(d->cauchy_a > 0.0)) return fail(CLC_ERR_INVALID, "cauchy_a must be positive");
  if (d->line_fit_max_iterations < 0) return fail(CLC_ERR_INVALID, "line_fit_max_iterations < 0");

  ScanStats st;
  clc_problem *pa = nullptr, *pb = nullptr;
  float* d_ranges = nullptr;
  double *d_stamp = nullptr, *d_pose_stamp = nullptr, *d_pose_wc = nullptr, *d_lines = nullptr, *d_scan_line = nullptr;
  int* d_info = nullptr;
  int64_t *d_cnt = nullptr, *d_excl = nullptr;
  void* d_tmp = nullptr;
  cudaEvent_t ev[7] = {};
  auto body = [&]() -> int {
    int rc = scan_problem_shell(&pa, d);
    if (rc != CLC_OK) return rc;
    rc = scan_problem_shell(&pb, d);
    if (rc != CLC_OK) return rc;
    cudaStream_t sa = pa->stream;
    for (cudaEvent_t& e : ev) CLC_CUDA(cudaEventCreate(&e));
    // -- H2D: the ranges (4 B per beam), the stamps and the poses; nothing else crosses PCIe towards the device
    CLC_CUDA(cudaEventRecord(ev[0], sa));
    const size_t range_bytes = sizeof(float) * (size_t)S * (size_t)B;
    CLC_CUDA(cudaMallocAsync(&d_ranges, std::max<size_t>(range_bytes, 4), sa));
    CLC_CUDA(cudaMallocAsync(&d_stamp, sizeof(double) * std::max<int64_t>(S, 1), sa));
    CLC_CUDA(cudaMallocAsync(&d_pose_stamp, sizeof(double) * std::max<int64_t>(K, 1), sa));
    CLC_CUDA(cudaMallocAsync(&d_pose_wc, sizeof(double) * 7 * std::max<int64_t>(K, 1), sa));
    CLC_CUDA(cudaMallocAsync(&d_info, sizeof(int) * 4 * std::max<int64_t>(S, 1), sa));
    CLC_CUDA(cudaMallocAsync(&d_cnt, sizeof(int64_t) * 2 * (S + 1), sa));
    CLC_CUDA(cudaMallocAsync(&d_excl, sizeof(int64_t) * 2 * (S + 1), sa));
    if (range_bytes > 0) CLC_CUDA(cudaMemcpyAsync(d_ranges, d->ranges, range_bytes, cudaMemcpyHostToDevice, sa));
    if (S > 0) CLC_CUDA(cudaMemcpyAsync(d_stamp, d->scan_stamp, sizeof(double) * S, cudaMemcpyHostToDevice, sa));
    if (K > 0) {
      CLC_CUDA(cudaMemcpyAsync(d_pose_stamp, d->pose_stamp, sizeof(double) * K, cudaMemcpyHostToDevice, sa));
      CLC_CUDA(cudaMemcpyAsync(d_pose_wc, d->pose_wc, sizeof(double) * 7 * K, cudaMemcpyHostToDevice, sa));
    }
    st.bytes_h2d = (int64_t)range_bytes + 8 * S + 8 * K + 56 * K;
    CLC_CUDA(cudaEventRecord(ev[1], sa));
    // -- classify: segment + nearest pose per scan
    CLC_CUDA(cudaMemsetAsync(d_excl, 0, sizeof(int64_t) * 2 * (S + 1), sa));
    if (S > 0) {
      clc::clc_scan_classify_kernel<<<(unsigned)((S + clc::kClassifyThreads) / clc::kClassifyThreads), clc::kClassifyThreads, 0, sa>>>(
          d_ranges, S, B, d->angle_min, d->angle_increment, d->range_min, d_stamp, d_pose_stamp, K, d->max_dt, d_info, d_cnt);
      CLC_LAUNCH_CHECK();
    }
    CLC_CUDA(cudaEventRecord(ev[2], sa));
    // -- exclusive scans (integer: deterministic) -> frame index per scan, point offset per scan; the totals at [S]
    int64_t totals[2] = {0, 0};
    if (S > 0) {
      size_t tmp_bytes = 0;
      CLC_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, d_cnt, d_excl, S + 1, sa));
      CLC_CUDA(cudaMallocAsync(&d_tmp, tmp_bytes, sa));
      CLC_CUDA(cub::DeviceScan::ExclusiveSum(d_tmp, tmp_bytes, d_cnt, d_excl, S + 1, sa));
      CLC_CUDA(cub::DeviceScan::ExclusiveSum(d_tmp, tmp_bytes, d_cnt + S + 1, d_excl + S + 1, S + 1, sa));
      g_launches.fetch_add(2);
      CLC_CUDA(cudaMemcpyAsync(&totals[0], d_excl + S, sizeof(int64_t), cudaMemcpyDeviceToHost, sa));
      CLC_CUDA(cudaMemcpyAsync(&totals[1], d_excl + 2 * S + 1, sizeof(int64_t), cudaMemcpyDeviceToHost, sa));
    }
    CLC_CUDA(cudaEventRecord(ev[3], sa));
    CLC_CUDA(cudaStreamSynchronize(sa));  // the only host sync before the allocations
    st.bytes_d2h = S > 0 ? 16 : 0;
    const int64_t F = totals[0], P = totals[1];
    // -- allocate both problems, gather the points problem
    rc = scan_problem_alloc(pa, F, P, false);
    if (rc != CLC_OK) return rc;
    rc = scan_problem_alloc(pb, F, 2 * F, d->with_edges != 0);
    if (rc != CLC_OK) return rc;
    CLC_CUDA(cudaStreamSynchronize(pb->stream));  // pb's arrays are written on sa below
    if (S > 0) {
      const int warps = 8;
      clc::clc_scan_gather_kernel<<<(unsigned)((S + warps - 1) / warps), warps * 32, 0, sa>>>(
          d_ranges, S, B, d->angle_min, d->angle_increment, d->range_min, d_pose_wc, d_cnt, d_excl, d_info, pa->x, pa->y,
          pa->frame_pose, pa->offsets);
      CLC_LAUNCH_CHECK();
    }
    CLC_CUDA(cudaFreeAsync(d_ranges, sa));  // the largest buffer goes back to the pool before the line fit
    d_ranges = nullptr;
    CLC_CUDA(cudaEventRecord(ev[4], sa));
    // -- batched LineFittingCeres from a zero start (calibr_offline.cpp:123-124; CauchyLoss(0.05), LaseCamCalCeres.cpp:416),
    //    then the on-line problem device to device
    CLC_CUDA(cudaMallocAsync(&d_lines, sizeof(double) * 2 * std::max<int64_t>(F, 1), sa));
    if (F > 0) {
      CLC_CUDA(cudaMemsetAsync(d_lines, 0, sizeof(double) * 2 * F, sa));
      const int warps = 8;
      clc::clc_line_fit_kernel<<<(unsigned)((F + warps - 1) / warps), warps * 32, 0, sa>>>(
          pa->x, pa->y, pa->offsets, F, d->line_fit_max_iterations, 0.05, d_lines, nullptr);
      CLC_LAUNCH_CHECK();
      clc::clc_scan_on_line_kernel<<<(unsigned)((F + 255) / 256), 256, 0, sa>>>(pa->x, pa->y, pa->offsets, pa->frame_pose, d_lines, F,
                                                                               pb->x, pb->y, pb->frame_pose, pb->offsets, pb->edge_pt);
      CLC_LAUNCH_CHECK();
    }
    if (scan_line && S > 0) {
      CLC_CUDA(cudaMallocAsync(&d_scan_line, sizeof(double) * 2 * S, sa));
      clc::clc_scan_lines_kernel<<<(unsigned)((S + 255) / 256), 256, 0, sa>>>(d_info, S, d_lines, d_scan_line);
      CLC_LAUNCH_CHECK();
      CLC_CUDA(cudaMemcpyAsync(scan_line, d_scan_line, sizeof(double) * 2 * S, cudaMemcpyDeviceToHost, sa));
      st.bytes_d2h += 16 * S;
    }
    if (scan_info && S > 0) {
      CLC_CUDA(cudaMemcpyAsync(scan_info, d_info, sizeof(int) * 4 * S, cudaMemcpyDeviceToHost, sa));
      st.bytes_d2h += 16 * S;
    }
    CLC_CUDA(cudaEventRecord(ev[5], sa));
    // -- planes, partition (finish_create synchronises each problem's stream: pb's inputs were written on sa, which is
    //    complete once finish_create(pa) returns)
    rc = finish_create(pa);
    if (rc != CLC_OK) return rc;
    rc = finish_create(pb);
    if (rc != CLC_OK) return rc;
    CLC_CUDA(cudaEventRecord(ev[6], pb->stream));
    CLC_CUDA(cudaEventSynchronize(ev[6]));
    for (int i = 0; i < 6; ++i) CLC_CUDA(cudaEventElapsedTime(&st.ms[i], ev[i], ev[i + 1]));
    return CLC_OK;
  };
  int rc = body();
  if (pa && pa->stream) {
    void* bufs[] = {d_ranges, d_stamp, d_pose_stamp, d_pose_wc, d_lines, d_scan_line, d_info, d_cnt, d_excl, d_tmp};
    for (void* b : bufs)
      if (b) cudaFreeAsync(b, pa->stream);
  }
  for (cudaEvent_t e : ev)
    if (e) cudaEventDestroy(e);
  if (rc == CLC_OK && pa && pa->stream) {
    cudaError_t e = cudaStreamSynchronize(pa->stream);
    if (e != cudaSuccess) rc = fail(CLC_ERR_CUDA, cudaGetErrorString(e));
  }
  if (rc != CLC_OK) {
    const std::string msg = g_last_error;
    clc_problem_destroy(pa);
    clc_problem_destroy(pb);
    g_last_error = msg;
    return rc;
  }
  g_scan_stats = st;
  if (points_out) *points_out = pa; else clc_problem_destroy(pa);
  if (on_line_out) *on_line_out = pb; else clc_problem_destroy(pb);
  return CLC_OK;
}

int clc_scan_last_stats(float phase_ms6[6], int64_t* bytes_h2d, int64_t* bytes_d2h) {
  if (phase_ms6)
    for (int i = 0; i < 6; ++i) phase_ms6[i] = g_scan_stats.ms[i];
  if (bytes_h2d) *bytes_h2d = g_scan_stats.bytes_h2d;
  if (bytes_d2h) *bytes_d2h = g_scan_stats.bytes_d2h;
  return CLC_OK;
}

int clc_estimate_board_poses(const clc_camera_desc* cam, int64_t n_frames, const int64_t* det_offsets, const int32_t* tag_ids,
                             const float* corners_uv, double* pose_wc, int32_t* ok, int device) {
  if (!cam || n_frames < 0 || !det_offsets || !pose_wc || !ok) return fail(CLC_ERR_INVALID, "bad pose-estimation arguments");
  if (cam->camera_model != clc::kCameraPinholeRadtan && cam->camera_model != clc::kCameraEquidistant)
    return fail(CLC_ERR_INVALID, "unknown camera_model");
  if (cam->grid_rows < 1 || cam->grid_cols < 1 || !(cam->tag_size > 0.0) || !(cam->intrinsics[0] > 0.0) ||
      !(cam->intrinsics[1] > 0.0))
    return fail(CLC_ERR_INVALID, "bad camera / grid description");
  if (n_frames == 0) return CLC_OK;
  if (det_offsets[0] != 0) return fail(CLC_ERR_INVALID, "det_offsets[0] must be 0");
  for (int64_t f = 0; f < n_frames; ++f)
    if (det_offsets[f + 1] < det_offsets[f]) return fail(CLC_ERR_INVALID, "det_offsets must be non-decreasing");
  const int64_t D = det_offsets[n_frames];
  if (D > 0 && (!tag_ids || !corners_uv)) return fail(CLC_ERR_INVALID, "detections missing");
  int count = 0;
  CLC_CUDA(cudaGetDeviceCount(&count));
  if (device < 0) CLC_CUDA(cudaGetDevice(&device));
  if (device >= count) return fail(CLC_ERR_INVALID, "device ordinal out of range");
  CLC_CUDA(cudaSetDevice(device));
  clc::CameraDesc c;
  c.model = cam->camera_model;
  for (int k = 0; k < 8; ++k) c.intr[k] = cam->intrinsics[k];
  c.pixel_sigma = 0.0;
  c.grid_rows = cam->grid_rows;
  c.grid_cols = cam->grid_cols;
  c.tag_size = cam->tag_size;
  c.tag_spacing = cam->tag_spacing;
  int64_t* d_off = nullptr;
  int *d_ids = nullptr, *d_ok = nullptr;
  float *d_uv = nullptr, *d_lift = nullptr;
  double* d_pose = nullptr;
  cudaStream_t st;
  CLC_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
  const size_t Dm = (size_t)std::max<int64_t>(D, 1);
  cudaError_t e = cudaMallocAsync(&d_off, sizeof(int64_t) * (n_frames + 1), st);
  if (e == cudaSuccess) e = cudaMallocAsync(&d_ids, sizeof(int) * Dm, st);
  if (e == cudaSuccess) e = cudaMallocAsync(&d_uv, sizeof(float) * 8 * Dm, st);
  if (e == cudaSuccess) e = cudaMallocAsync(&d_lift, sizeof(float) * 8 * Dm, st);
  if (e == cudaSuccess) e = cudaMallocAsync(&d_pose, sizeof(double) * 7 * n_frames, st);
  if (e == cudaSuccess) e = cudaMallocAsync(&d_ok, sizeof(int) * n_frames, st);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_off, det_offsets, sizeof(int64_t) * (n_frames + 1), cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess && D > 0) e = cudaMemcpyAsync(d_ids, tag_ids, sizeof(int) * D, cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess && D > 0) e = cudaMemcpyAsync(d_uv, corners_uv, sizeof(float) * 8 * D, cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) {
    clc::clc_estimate_poses_kernel<<<(unsigned)((n_frames + 63) / 64), 64, 0, st>>>(c, n_frames, d_off, d_ids, d_uv, d_lift, d_pose, d_ok);
    g_launches.fetch_add(1);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaMemcpyAsync(pose_wc, d_pose, sizeof(double) * 7 * n_frames, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaMemcpyAsync(ok, d_ok, sizeof(int) * n_frames, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  void* bufs[] = {d_off, d_ids, d_uv, d_lift, d_pose, d_ok};
  for (void* b : bufs)
    if (b) cudaFreeAsync(b, st);
  cudaStreamSynchronize(st);
  cudaStreamDestroy(st);
  if (e != cudaSuccess) return fail(CLC_ERR_CUDA, cudaGetErrorString(e));
  return CLC_OK;
}

// ---- multi-GPU --------------------------------------------------------------------------------------------------

int clc_shard_range(int64_t n_frames, const int64_t* offsets, int nranks, int rank, int64_t* begin, int64_t* end) {
  if (nranks < 1 || rank < 0 || rank >= nranks || n_frames < 0 || !begin || !end)
    return fail(CLC_ERR_INVALID, "bad shard arguments");
  if (!offsets) {
    *begin = n_frames * rank / nranks;
    *end = n_frames * (rank + 1) / nranks;
    return CLC_OK;
  }
  // contiguous ranges balanced by point count: boundary r is the first frame whose start >= r * P / nranks
  const int64_t P = offsets[n_frames];
  auto boundary = [&](int r) -> int64_t {
    if (r <= 0) return 0;
    if (r >= nranks) return n_frames;
    const int64_t target = (int64_t)((__int128)P * r / nranks);
    return std::lower_bound(offsets, offsets + n_frames + 1, target) - offsets;
  };
  *begin = boundary(rank);
  *end = boundary(rank + 1);
  if (*end < *begin) *end = *begin;
  return CLC_OK;
}

int clc_comm_unique_id(void* id128) {
  if (!id128) return fail(CLC_ERR_INVALID, "NULL id");
  NcclApi* api = nccl_api();
  if (!api->handle) return fail(CLC_ERR_NCCL, api->error);
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
  ncclUniqueId id;
  CLC_NCCL(api->GetUniqueId(&id));
  std::memcpy(id128, &id, sizeof(id));
  return CLC_OK;
}

int clc_comm_create(clc_comm** out, const void* id128, int nranks, int rank, int device) {
  if (!out || !id128 || nranks < 1 || rank < 0 || rank >= nranks) return fail(CLC_ERR_INVALID, "bad comm arguments");
  *out = nullptr;
  NcclApi* api = nccl_api();
  if (!api->handle) return fail(CLC_ERR_NCCL, api->error);
  if (device < 0) CLC_CUDA(cudaGetDevice(&device));
  CLC_CUDA(cudaSetDevice(device));
  ncclUniqueId id;
  std::memcpy(&id, id128, sizeof(id));
  clc_comm* c = new clc_comm();
  c->nranks = nranks;
  c->rank = rank;
  c->device = device;
  ncclResult_t r = api->CommInitRank(&c->comm, nranks, id, rank);
  if (r != ncclSuccess) {
    delete c;
    return fail(CLC_ERR_NCCL, std::string("ncclCommInitRank: ") + api->GetErrorString(r));
  }
  *out = c;
  return CLC_OK;
}

int clc_comm_p2p_export(clc_comm* c, void* handle64) {
  if (!c || !handle64) return fail(CLC_ERR_INVALID, "NULL argument");
  if (c->nranks > clc::kMaxRanks) return fail(CLC_ERR_INVALID, "too many ranks for the peer path");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
  CLC_CUDA(cudaSetDevice(c->device));
  if (!c->p2p_block) {
    CLC_CUDA(cudaMalloc(&c->p2p_block, c->block_bytes()));  // cudaMalloc (not the pool): IPC needs a real allocation
    CLC_CUDA(cudaMemset(c->p2p_block, 0, c->block_bytes()));
  }
  cudaIpcMemHandle_t h;
  CLC_CUDA(cudaIpcGetMemHandle(&h, c->p2p_block));
  std::memcpy(handle64, &h, sizeof(h));
  return CLC_OK;
}

int clc_comm_p2p_import(clc_comm* c, const void* handles) {
  if (!c || !handles) return fail(CLC_ERR_INVALID, "NULL argument");
  if (!c->p2p_block) return fail(CLC_ERR_STATE, "clc_comm_p2p_export must be called first");
  CLC_CUDA(cudaSetDevice(c->device));
  for (int r = 0; r < c->nranks; ++r) {
    if (r == c->rank) {
      c->peer_block[r] = c->p2p_block;
      continue;
    }
    cudaIpcMemHandle_t h;
    std::memcpy(&h, static_cast<const char*>(handles) + 64 * (size_t)r, sizeof(h));
    CLC_CUDA(cudaIpcOpenMemHandle(&c->peer_block[r], h, cudaIpcMemLazyEnablePeerAccess));
  }
  c->p2p_ready = true;
  return CLC_OK;
}

int clc_comm_destroy(clc_comm* c) {
  if (!c) return CLC_OK;
  cudaSetDevice(c->device);
  if (!c->local)
    for (int r = 0; r < c->nranks; ++r)
      if (r != c->rank && c->peer_block[r]) cudaIpcCloseMemHandle(c->peer_block[r]);
  if (c->p2p_block) cudaFree(c->p2p_block);
  if (c->comm && nccl_api()->handle) {
    cudaSetDevice(c->device);
    nccl_api()->CommDestroy(c->comm);
  }
  delete c;
  return CLC_OK;
}

int clc_problem_attach_comm(clc_problem* p, clc_comm* c) {
  if (!p) return fail(CLC_ERR_INVALID, "NULL problem");
  if (!c) {
    p->comm_obj = nullptr;
    p->comm = nullptr;
    p->nranks = 1;
    p->rank = 0;
    p->allreduce_mode = 0;
    return CLC_OK;
  }
  if (c->device != p->device) return fail(CLC_ERR_INVALID, "communicator and problem live on different devices");
  p->comm_obj = c;
  p->comm = c->comm;
  p->nranks = c->nranks;
  p->rank = c->rank;
  p->allreduce_mode = c->p2p_ready ? 1 : 0;
  return CLC_OK;
}

int clc_problem_set_allreduce_mode(clc_problem* p, int mode) {
  if (!p) return fail(CLC_ERR_INVALID, "NULL problem");
  if (mode != 0 && mode != 1) return fail(CLC_ERR_INVALID, "unknown all-reduce mode");
  if (mode == 1 && !(p->comm_obj && p->comm_obj->p2p_ready))
    return fail(CLC_ERR_STATE, "peer exchange not initialised (clc_comm_p2p_export / clc_comm_p2p_import)");
  p->allreduce_mode = mode;
  return CLC_OK;
}

// ---- in-process multi-GPU: one host thread, G devices, the same fused NVLink exchange --------------------------------

struct clc_group {
  std::vector<clc_problem*> problems;
  std::vector<clc_comm*> comms;  // local communicators (empty for a single device)
  int64_t n_frames = 0, n_points = 0;
};

}  // extern "C"
static clc_problem* group_release_single(clc_group* g) {
  clc_problem* p = g->problems.empty() ? nullptr : g->problems[0];
  delete g;
  return p;
}
extern "C" {

namespace {

// mailboxes on every device, peer access between all pairs, plain device pointers instead of IPC handles
int comms_create_local(std::vector<clc_comm*>* out, const int* devices, int n) {
  if (n > clc::kMaxRanks) return fail(CLC_ERR_INVALID, "too many devices for the peer exchange");
  for (int i = 0; i < n; ++i)
    for (int j = 0; j < i; ++j)
      if (devices[i] == devices[j]) return fail(CLC_ERR_INVALID, "a device may appear only once in a group");
  auto cleanup = [&]() {
    for (clc_comm* c : *out) clc_comm_destroy(c);
    out->clear();
  };
  for (int i = 0; i < n; ++i) {
    clc_comm* c = new clc_comm();
    c->nranks = n;
    c->rank = i;
    c->device = devices[i];
    c->local = true;
    out->push_back(c);
    cudaError_t e = cudaSetDevice(devices[i]);
    if (e == cudaSuccess) e = cudaMalloc(&c->p2p_block, c->block_bytes());
    if (e == cudaSuccess) e = cudaMemset(c->p2p_block, 0, c->block_bytes());
    if (e != cudaSuccess) {
      cleanup();
      return fail(CLC_ERR_CUDA, std::string("group mailbox: ") + cudaGetErrorString(e));
    }
  }
  for (int i = 0; i < n; ++i) {
    cudaSetDevice(devices[i]);
    for (int j = 0; j < n; ++j) {
      if (i == j) continue;
      int can = 0;
      cudaError_t e = cudaDeviceCanAccessPeer(&can, devices[i], devices[j]);
      if (e == cudaSuccess && !can) {
        cleanup();
        return fail(CLC_ERR_CUDA, "devices " + std::to_string(devices[i]) + " and " + std::to_string(devices[j]) +
                                      " have no peer access: the fused exchange needs NVLink/PCIe P2P");
      }
      if (e == cudaSuccess) e = cudaDeviceEnablePeerAccess(devices[j], 0);
      if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); e = cudaSuccess; }
      if (e != cudaSuccess) {
        cleanup();
        return fail(CLC_ERR_CUDA, std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e));
      }
    }
  }
  for (int i = 0; i < n; ++i) {
    for (int r = 0; r < n; ++r) (*out)[i]->peer_block[r] = (*out)[r]->p2p_block;
    (*out)[i]->p2p_ready = true;
  }
  return CLC_OK;
}

// The mailboxes of an in-process group outlive the group: cudaMalloc / cudaFree / enabling peer access cost milliseconds,
// and the drop-in builds a group per CamLaserCalibration() call.  One idle set per device list is kept; the exchange's
// sequence counter lives in the mailbox block and simply keeps counting across groups.
std::mutex g_comm_cache_mutex;
std::vector<std::pair<std::vector<int>, std::vector<clc_comm*>>> g_comm_cache;

int comms_acquire_local(std::vector<clc_comm*>* out, const int* devices, int n) {
  const std::vector<int> key(devices, devices + n);
  {
    std::lock_guard<std::mutex> lock(g_comm_cache_mutex);
    for (size_t i = 0; i < g_comm_cache.size(); ++i)
      if (g_comm_cache[i].first == key) {
        *out = g_comm_cache[i].second;
        g_comm_cache.erase(g_comm_cache.begin() + (long)i);
        return CLC_OK;
      }
  }
  return comms_create_local(out, devices, n);
}

void comms_release_local(std::vector<clc_comm*>& comms) {
  if (comms.empty()) return;
  std::vector<int> key;
  for (clc_comm* c : comms) key.push_back(c->device);
  {
    std::lock_guard<std::mutex> lock(g_comm_cache_mutex);
    bool have = false;
    for (auto& e : g_comm_cache) have = have || e.first == key;
    if (!have && g_comm_cache.size() < 8) {
      g_comm_cache.emplace_back(key, comms);
      comms.clear();
      return;
    }
  }
  for (clc_comm* c : comms) clc_comm_destroy(c);
  comms.clear();
}

int group_attach(clc_group* g, const int* devices, int n) {
  if (n <= 1) return CLC_OK;
  int rc = comms_acquire_local(&g->comms, devices, n);
  if (rc != CLC_OK) return rc;
  for (int i = 0; i < n; ++i) {
    rc = clc_problem_attach_comm(g->problems[i], g->comms[i]);
    if (rc != CLC_OK) return rc;
  }
  // warm the peer mappings and the exchange path: a few collective sweeps outside any timed region
  const double ident[7] = {0, 0, 0, 0, 0, 0, 1};
  for (int k = 0; k < 3 && rc == CLC_OK; ++k) rc = eval_all(g->problems.data(), n, ident, 1);
  return rc;
}

int resolve_devices(const int* devices, int n_devices, std::vector<int>* out) {
  int count = 0;
  CLC_CUDA(cudaGetDeviceCount(&count));
  if (count <= 0) return fail(CLC_ERR_CUDA, "no CUDA device");
  if (n_devices < 1 || !devices) return fail(CLC_ERR_INVALID, "need at least one device");
  for (int i = 0; i < n_devices; ++i) {
    int d = devices[i];
    if (d < 0) CLC_CUDA(cudaGetDevice(&d));
    if (d >= count) return fail(CLC_ERR_INVALID, "device ordinal out of range");
    out->push_back(d);
  }
  return CLC_OK;
}

}  // namespace

int clc_group_destroy(clc_group* g) {
  if (!g) return CLC_OK;
  bool clean = true;  // a group whose exchange timed out must not hand its mailboxes to the next one
  if (!g->comms.empty())
  for (clc_problem* p : g->problems) {
    int err = 0;
    if (p->p2p_error && cudaSetDevice(p->device) == cudaSuccess && cudaStreamSynchronize(p->stream) == cudaSuccess &&
        cudaMemcpy(&err, p->p2p_error, sizeof(int), cudaMemcpyDeviceToHost) == cudaSuccess)
      clean = clean && err == 0;
    else
      clean = false;
  }
  for (clc_problem* p : g->problems) clc_problem_destroy(p);
  if (clean) comms_release_local(g->comms);
  for (clc_comm* c : g->comms) clc_comm_destroy(c);
  delete g;
  return CLC_OK;
}

int clc_group_create_gather(clc_group** out, const clc_gather_desc* d, const int* devices, int n_devices) {
  if (!out || !d) return fail(CLC_ERR_INVALID, "NULL argument");
  *out = nullptr;
  const int64_t N = d->n_frames;
  if (N < 0 || (N > 0 && (!d->frame_pose || !d->frame_points || !d->frame_counts)))
    return fail(CLC_ERR_INVALID, "frame_pose/frame_points/frame_counts missing");
  if (!(d->cauchy_a > 0.0)) return fail(CLC_ERR_INVALID, "cauchy_a must be positive");
  if (N >= ((int64_t)1 << 31)) return fail(CLC_ERR_INVALID, "too many frames");
  std::vector<int> devs;
  int rc = resolve_devices(devices, n_devices, &devs);
  if (rc != CLC_OK) return rc;
  const int G = (int)devs.size();
  std::vector<int64_t> prefix((size_t)N + 1, 0);
  for (int64_t f = 0; f < N; ++f) {
    if (d->frame_counts[f] < 0) return fail(CLC_ERR_INVALID, "negative frame count");
    if (d->frame_counts[f] > 0 && !d->frame_points[f]) return fail(CLC_ERR_INVALID, "NULL frame_points entry");
    prefix[f + 1] = prefix[f] + d->frame_counts[f];
  }
  clc_group* g = new clc_group();
  g->n_frames = N;
  g->n_points = prefix[N];
  std::vector<UploadShard> shards((size_t)G);
  std::vector<std::vector<int64_t>> local_offsets((size_t)G);
  for (int i = 0; i < G && rc == CLC_OK; ++i) {
    int64_t fb = 0, fe = N;
    rc = clc_shard_range(N, prefix.data(), G, i, &fb, &fe);  // contiguous frame ranges balanced by point count
    if (rc != CLC_OK) break;
    std::vector<int64_t>& lo = local_offsets[i];
    lo.resize((size_t)(fe - fb) + 1);
    for (int64_t f = fb; f <= fe; ++f) lo[f - fb] = prefix[f] - prefix[fb];
    HostSource src;
    src.n_frames = fe - fb;
    src.frame_pose = d->frame_pose + 7 * fb;
    src.offsets = lo.data();
    src.frame_points = d->frame_points + fb;
    src.edge_points = d->edge_points ? d->edge_points + 6 * fb : nullptr;
    clc_problem* p = nullptr;
    rc = create_shell(&p, src, d->use_loss, d->cauchy_a, devs[i], &shards[i]);
    if (rc == CLC_OK) g->problems.push_back(p);
  }
  if (rc == CLC_OK) {
    shards.resize(g->problems.size());
    rc = upload_and_finish(g->problems, shards);
  }
  if (rc == CLC_OK) rc = group_attach(g, devs.data(), G);
  if (rc != CLC_OK) {
    const std::string msg = g_last_error;
    clc_group_destroy(g);
    g_last_error = msg;
    return rc;
  }
  *out = g;
  return CLC_OK;
}

int clc_group_create_synthetic(clc_group** out, const clc_synthetic_desc* d, const int* devices, int n_devices) {
  if (!out || !d) return fail(CLC_ERR_INVALID, "NULL argument");
  *out = nullptr;
  std::vector<int> devs;
  int rc = resolve_devices(devices, n_devices, &devs);
  if (rc != CLC_OK) return rc;
  const int G = (int)devs.size();
  clc_group* g = new clc_group();
  const int64_t fb0 = d->frame_begin, N = d->frame_end - d->frame_begin;
  for (int i = 0; i < G && rc == CLC_OK; ++i) {
    clc_synthetic_desc di = *d;
    di.frame_begin = fb0 + N * i / G;
    di.frame_end = fb0 + N * (i + 1) / G;
    di.device = devs[i];
    clc_problem* p = nullptr;
    rc = clc_problem_create_synthetic(&p, &di);
    if (rc == CLC_OK) {
      g->problems.push_back(p);
      g->n_frames += p->n_frames;
      g->n_points += p->n_points;
    }
  }
  if (rc == CLC_OK) rc = group_attach(g, devs.data(), G);
  if (rc != CLC_OK) {
    const std::string msg = g_last_error;
    clc_group_destroy(g);
    g_last_error = msg;
    return rc;
  }
  *out = g;
  return CLC_OK;
}

int clc_group_size(const clc_group* g, int* n_devices, int64_t* n_frames, int64_t* n_points) {
  if (!g) return fail(CLC_ERR_INVALID, "NULL group");
  if (n_devices) *n_devices = (int)g->problems.size();
  if (n_frames) *n_frames = g->n_frames;
  if (n_points) *n_points = g->n_points;
  return CLC_OK;
}

int clc_group_problem(clc_group* g, int index, clc_problem** out) {
  if (!g || !out || index < 0 || index >= (int)g->problems.size()) return fail(CLC_ERR_INVALID, "bad group index");
  *out = g->problems[index];
  return CLC_OK;
}

int clc_group_eval(clc_group* g, const double pose7[7], double H36[36], double g6[6], double* cost) {
  if (!g || g->problems.empty()) return fail(CLC_ERR_INVALID, "NULL group");
  int rc = eval_all(g->problems.data(), (int)g->problems.size(), pose7, 0);
  if (rc != CLC_OK) return rc;
  eval_post(g->problems[0]->h_sums, H36, g6, cost);
  return CLC_OK;
}

int clc_group_information(clc_group* g, const double pose7[7], double H36[36], double b6[6], double* chi, double sv6[6],
                          double V36[36]) {
  if (!g || g->problems.empty()) return fail(CLC_ERR_INVALID, "NULL group");
  int rc = eval_all(g->problems.data(), (int)g->problems.size(), pose7, 1);
  if (rc != CLC_OK) return rc;
  information_post(g->problems[0]->h_sums, H36, b6, chi, sv6, V36);
  return CLC_OK;
}

int clc_group_closed_form(clc_group* g, double Tlc16[16], int* unobservable, double AtA81[81], double Atb9[9]) {
  if (!g || g->problems.empty() || !Tlc16) return fail(CLC_ERR_INVALID, "NULL argument");
  int rc = eval_all(g->problems.data(), (int)g->problems.size(), nullptr, 2);
  if (rc != CLC_OK) return rc;
  closed_form_post(g->problems[0]->h_sums, Tlc16, unobservable, AtA81, Atb9);
  return CLC_OK;
}

int clc_group_solve_lm(clc_group* g, double pose7[7], const clc_lm_options* opt, clc_lm_summary* summary,
                       clc_lm_iteration* trace, int trace_cap) {
  if (!g || g->problems.empty() || !pose7) return fail(CLC_ERR_INVALID, "NULL argument");
  return solve_all(g->problems.data(), (int)g->problems.size(), pose7, opt, summary, trace, trace_cap);
}

// Devices the reference-facing drop-in uses (its signatures have no device argument): the environment variable
// CLC_DEVICES = "0,1,2,3" | "all" | unset (the current device).
int clc_default_devices(int* devices, int cap, int* n) {
  if (!devices || !n || cap < 1) return fail(CLC_ERR_INVALID, "bad device list arguments");
  int count = 0;
  CLC_CUDA(cudaGetDeviceCount(&count));
  if (count <= 0) return fail(CLC_ERR_CUDA, "no CUDA device");
  *n = 0;
  const char* env = std::getenv("CLC_DEVICES");
  if (!env || !*env) {
    int cur = 0;
    CLC_CUDA(cudaGetDevice(&cur));
    devices[(*n)++] = cur;
    return CLC_OK;
  }
  if (std::strcmp(env, "all") == 0) {
    for (int d = 0; d < count && *n < cap; ++d) devices[(*n)++] = d;
    return CLC_OK;
  }
  const char* s = env;
  while (*s) {
    char* endp = nullptr;
    const long v = std::strtol(s, &endp, 10);
    if (endp == s) return fail(CLC_ERR_INVALID, std::string("cannot parse CLC_DEVICES=") + env);
    if (v < 0 || v >= count) return fail(CLC_ERR_INVALID, std::string("CLC_DEVICES names a device that does not exist: ") + env);
    if (*n < cap) devices[(*n)++] = (int)v;
    s = endp;
    while (*s == ',' || *s == ' ') ++s;
  }
  if (*n == 0) return fail(CLC_ERR_INVALID, "CLC_DEVICES is empty");
  return CLC_OK;
}

// test hook (no CUDA involved): what the pack threads would write for the local point range [a, b) of a gathered shard.
// xy != 0: packed x,y pairs, *nonplanar receives whether a z != 0 was met; xy == 0: packed xyz.
int clc_debug_pack(int64_t n_frames, const double* const* frame_points, const int64_t* frame_counts, int64_t a, int64_t b,
                   int xy, double* out, int* nonplanar) {
  if (n_frames < 0 || !frame_points || !frame_counts || !out || a < 0 || b < a) return fail(CLC_ERR_INVALID, "bad pack arguments");
  std::vector<int64_t> prefix((size_t)n_frames + 1, 0);
  for (int64_t f = 0; f < n_frames; ++f) prefix[f + 1] = prefix[f] + frame_counts[f];
  if (b > prefix[n_frames]) return fail(CLC_ERR_INVALID, "pack range beyond the last point");
  UploadShard s;
  s.frame_points = frame_points;
  s.offsets = prefix.data();
  s.n_frames = n_frames;
  if (xy) {
    const bool np = pack_xy(s, a, b, out);
    if (nonplanar) *nonplanar = np ? 1 : 0;
  } else {
    pack_xyz(s, a, b, out);
  }
  return CLC_OK;
}

// statistics of the most recent host -> HBM upload of this process (measurement hook)
int clc_upload_last_stats(double* total_ms, double* pack_wait_ms, int64_t* bytes_h2d, int* chunks, int* pack_threads,
                          int* direct) {
  if (total_ms) *total_ms = g_last_upload.total_ms;
  if (pack_wait_ms) *pack_wait_ms = g_last_upload.pack_wait_ms;
  if (bytes_h2d) *bytes_h2d = g_last_upload.bytes_h2d;
  if (chunks) *chunks = g_last_upload.chunks;
  if (pack_threads) *pack_threads = g_last_upload.threads;
  if (direct) *direct = g_last_upload.direct;
  return CLC_OK;
}

// ---- measurement hooks -------------------------------------------------------------------------------------------

int clc_bench_eval(clc_problem* p, const double pose7[7], int n, int flush_l2, float* ms_each) {
  if (!p || !pose7 || n < 1 || !ms_each) return fail(CLC_ERR_INVALID, "bad bench arguments");
  int rc = set_device(p);
  if (rc != CLC_OK) return rc;
  if (flush_l2 && !p->flush_buf) {
    p->flush_n = ((int64_t)256 << 20) / sizeof(double);  // 256 MiB > 126 MB of L2
    CLC_CUDA(cudaMallocAsync(&p->flush_buf, sizeof(double) * p->flush_n, p->stream));
  }
  CLC_CUDA(cudaMemcpyAsync(p->pose, pose7, sizeof(double) * 7, cudaMemcpyHostToDevice, p->stream));
  std::vector<cudaEvent_t> ev(2 * (size_t)n);
  for (auto& e : ev) CLC_CUDA(cudaEventCreate(&e));
  const bool loss = p->use_loss != 0, edges = p->n_edges > 0;
  // The flush kernels run with the sweep kernel's shared-memory carve-out (CLC_FLUSH_SMEM=0 disables): an SM that has to
  // switch its L1/shared split between two kernels drains first, and in the LM loop the sweeps follow each other with
  // the same split -- the timed launch should not pay a reconfiguration the product never sees.
  int flush_smem = clc::dyn_smem_bytes(p->planar);
  if (const char* env = std::getenv("CLC_FLUSH_SMEM")) {
    if (std::atoi(env) == 0) flush_smem = 0;
  }
  if (flush_l2 && flush_smem > 0) {
    CLC_CUDA(cudaFuncSetAttribute(clc::clc_flush_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, flush_smem));
    CLC_CUDA(cudaFuncSetAttribute(clc::clc_flush_read_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, flush_smem));
  }
  for (int i = 0; i < n; ++i) {
    if (flush_l2) {
      clc::clc_flush_kernel<<<p->num_sms, 1024, flush_smem, p->stream>>>(p->flush_buf, p->flush_n, (double)i);
      CLC_LAUNCH_CHECK();
      clc::clc_flush_read_kernel<<<p->num_sms, 1024, flush_smem, p->stream>>>(p->flush_buf, p->flush_n, p->flush_buf);
      CLC_LAUNCH_CHECK();
    }
    CLC_CUDA(cudaEventRecord(ev[2 * i], p->stream));
    rc = launch_sweep(p, clc::kModeLM, loss, edges, p->pose, nullptr, nullptr, /*collective=*/false);
    if (rc != CLC_OK) return rc;
    CLC_CUDA(cudaEventRecord(ev[2 * i + 1], p->stream));
  }
  CLC_CUDA(cudaStreamSynchronize(p->stream));
  for (int i = 0; i < n; ++i) CLC_CUDA(cudaEventElapsedTime(&ms_each[i], ev[2 * i], ev[2 * i + 1]));
  for (auto& e : ev) cudaEventDestroy(e);
  return CLC_OK;
}

// Profiling hook (not part of the reference-facing surface): one sweep with per-block globaltimer stamps.
// stamps[grid*8]: 0 block start, 1 stream done, 2 tile flushed, 3 block partial written, 4 (last block) final sums,
// 5 (last block) after the LM update.  with_lm != 0 runs the fused LM update of a fresh LM state at pose7.
// warp_stamps (optional, [grid * 16]): the time every warp finished its stream.
int clc_debug_sweep_timing(clc_problem* p, const double pose7[7], int with_lm, int flush_l2, unsigned long long* stamps,
                           int* grid_out, unsigned long long* warp_stamps) {
  if (!p || !pose7 || !stamps) return fail(CLC_ERR_INVALID, "bad timing arguments");
  int rc = set_device(p);
  if (rc != CLC_OK) return rc;
  if (grid_out) *grid_out = p->grid;
  const size_t bytes = sizeof(unsigned long long) * 8 * (size_t)p->grid;
  const size_t wbytes = sizeof(unsigned long long) * clc::kWarps * (size_t)p->grid;
  CLC_CUDA(cudaMallocAsync(&p->timing, bytes + wbytes, p->stream));
  CLC_CUDA(cudaMemsetAsync(p->timing, 0, bytes + wbytes, p->stream));
  if (flush_l2) {
    if (!p->flush_buf) {
      p->flush_n = ((int64_t)256 << 20) / sizeof(double);
      CLC_CUDA(cudaMallocAsync(&p->flush_buf, sizeof(double) * p->flush_n, p->stream));
    }
    clc::clc_flush_kernel<<<p->num_sms * 4, 256, 0, p->stream>>>(p->flush_buf, p->flush_n, 1.0);
    CLC_LAUNCH_CHECK();
    clc::clc_flush_read_kernel<<<p->num_sms * 4, 256, 0, p->stream>>>(p->flush_buf, p->flush_n, p->flush_buf);
    CLC_LAUNCH_CHECK();
  }
  clc_lm_options opt;
  clc_lm_default_options(&opt);
  clc::lm_init(&p->h_lm->core, pose7, opt);
  CLC_CUDA(cudaMemcpyAsync(p->lm, p->h_lm, sizeof(clc::LmState), cudaMemcpyHostToDevice, p->stream));
  CLC_CUDA(cudaMemcpyAsync(p->pose, pose7, sizeof(double) * 7, cudaMemcpyHostToDevice, p->stream));
  rc = launch_sweep(p, clc::kModeLM, p->use_loss != 0, p->n_edges > 0, p->pose, nullptr, with_lm ? p->lm : nullptr, /*collective=*/false);
  cudaError_t e = cudaMemcpyAsync(stamps, p->timing, bytes, cudaMemcpyDeviceToHost, p->stream);
  if (e == cudaSuccess && warp_stamps)
    e = cudaMemcpyAsync(warp_stamps, p->timing + 8 * (size_t)p->grid, wbytes, cudaMemcpyDeviceToHost, p->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(p->stream);
  cudaFreeAsync(p->timing, p->stream);
  p->timing = nullptr;
  if (rc != CLC_OK) return rc;
  if (e != cudaSuccess) return fail(CLC_ERR_CUDA, cudaGetErrorString(e));
  return CLC_OK;
}

// experiment builds (-DCLC_LM_PROFILE): clock stamps of the last on-device lm_update (see clc_lm.cuh); zeros otherwise
int clc_debug_lm_profile(long long out[16]) {
  if (!out) return fail(CLC_ERR_INVALID, "NULL argument");
  for (int i = 0; i < 16; ++i) out[i] = 0;
#ifdef CLC_LM_PROFILE
  CLC_CUDA(cudaMemcpyFromSymbol(out, clc::g_lm_profile, sizeof(long long) * 16));
#endif
  return CLC_OK;
}

int clc_bench_h2d(int64_t bytes, int device, int reps, float* ms_each) {
  if (bytes < 1 || reps < 1 || !ms_each) return fail(CLC_ERR_INVALID, "bad h2d bench arguments");
  if (device >= 0) CLC_CUDA(cudaSetDevice(device));
  void *h = nullptr, *d = nullptr;
  cudaStream_t st = nullptr;
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  cudaError_t e = cudaHostAlloc(&h, (size_t)bytes, cudaHostAllocDefault);
  if (e == cudaSuccess) { std::memset(h, 0, (size_t)bytes); e = cudaMalloc(&d, (size_t)bytes); }
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaEventCreate(&e0);
  if (e == cudaSuccess) e = cudaEventCreate(&e1);
  for (int i = -1; i < reps && e == cudaSuccess; ++i) {  // one untimed copy first
    e = cudaEventRecord(e0, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d, h, (size_t)bytes, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaEventRecord(e1, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e == cudaSuccess && i >= 0) e = cudaEventElapsedTime(&ms_each[i], e0, e1);
  }
  if (e0) cudaEventDestroy(e0);
  if (e1) cudaEventDestroy(e1);
  if (st) cudaStreamDestroy(st);
  if (d) cudaFree(d);
  if (h) cudaFreeHost(h);
  if (e != cudaSuccess) return fail(CLC_ERR_CUDA, std::string("h2d bench: ") + cudaGetErrorString(e));
  return CLC_OK;
}

int64_t clc_solve_readback_bytes(void) { return (int64_t)sizeof(clc::LmState) + (int64_t)sizeof(int); }

int clc_host_alloc(void** ptr, int64_t bytes) {
  if (!ptr || bytes < 0) return fail(CLC_ERR_INVALID, "bad host alloc arguments");
  CLC_CUDA(cudaMallocHost(ptr, (size_t)std::max<int64_t>(bytes, 1)));
  return CLC_OK;
}

int clc_host_free(void* ptr) {
  if (ptr) CLC_CUDA(cudaFreeHost(ptr));
  return CLC_OK;
}

}  // extern "C"
