// ba_host.cu -- host side of the BA path: problem regrouping, symbolic analysis of the reduced
// camera system, the Levenberg-Marquardt driver and the C ABI (include/svs_b200.h).
//
// Mirrors SlamGraph::optimize (slam_graph.cpp:319-355): copyDataToG2o -> optimizer.optimize(n)
// -> restoreDataFromG2o, with g2o's numerics replaced by the kernels in ba_kernels.cu.
// There is no CPU fallback: every entry point fails with SVS_ERR_NOGPU / SVS_ERR_CUDA
// when the device path is unavailable.
#include <algorithm>
#include <atomic>
#include <cstdio>
#include <chrono>
#include <cstdlib>
#include <condition_variable>
#include <cstring>
#include <functional>
#include <mutex>
#include <numeric>
#include <set>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include "../../include/svs_b200.h"
#include "ba_kernels.cuh"
#include "nccl_dyn.cuh"
#include "host_pool.hpp"
#include "svs_nvtx.hpp"

using namespace svs;

// One helper thread per handle (started on first use, parked on a condition variable in between): stages the
// observation arrays in pinned memory and enqueues their DMA while the calling thread analyses the structure.
struct Worker {
  std::thread th;
  std::mutex m;
  std::condition_variable cv;
  std::function<void()> job;
  bool busy = false, quit = false;
  void run() {
    std::unique_lock<std::mutex> lk(m);
    for (;;) {
      cv.wait(lk, [&] { return quit || job; });
      if (quit) return;
      std::function<void()> f = std::move(job);
      job = nullptr;
      lk.unlock();
      f();
      lk.lock();
      busy = false;
      cv.notify_all();
    }
  }
  void post(std::function<void()> f) {
    std::unique_lock<std::mutex> lk(m);
    if (!th.joinable()) th = std::thread([this] { run(); });
    cv.wait(lk, [&] { return !busy; });
    busy = true;
    job = std::move(f);
    cv.notify_all();
  }
  void wait() {
    std::unique_lock<std::mutex> lk(m);
    cv.wait(lk, [&] { return !busy; });
  }
  ~Worker() {
    {
      std::unique_lock<std::mutex> lk(m);
      cv.wait(lk, [&] { return !busy; });
      quit = true;
      cv.notify_all();
    }
    if (th.joinable()) th.join();
  }
};

// Symbolic analysis of the reduced camera system (see analyse() below)
struct Symbolic {
  std::vector<int> perm, pos, col_ptr, row_idx, upd_ptr, upd_dst, upd_ab, urg_dst, tbl, branch_ptr;
  std::vector<int> rptr, rowpos, rcol;   // row-major index of the off-diagonal factor blocks (backward pass)
  int max_col_branch = 0, max_col_sep = 0, max_row = 0;
  int nblk = 0;
};

struct svs_ba {
  int device = 0;
  int flags = 0;
  cudaStream_t stream = nullptr;
  std::string err;
  bool has_problem = false;
  double* d_raw = nullptr; double* h_raw = nullptr; size_t raw_cap = 0;   // user-order observations + weights (6 doubles per edge)
  Worker worker;
  SpinPool pool;   // the per-landmark / per-edge host loops of set_problem
  int host_threads = 8;  // threads of the per-landmark / per-edge host loops of set_problem (SVS_HOST_THREADS)
  int cur_known = -1;   // host mirror of LmCtl::cur (index of the accepted state buffers), -1 = ask the device
  BaDev d{};
  // one device arena + one pinned staging arena, grown on demand and reused across set_problem calls
  char* arena = nullptr; size_t arena_cap = 0, arena_off = 0;
  char* stage = nullptr; size_t stage_cap = 0;
  bool measuring = false;
  LmCtl* h_ctl = nullptr;  // pinned
  double* d_pose0 = nullptr;
  double* d_psi0 = nullptr;
  std::vector<int> lm_to_user;  // internal landmark -> caller's index
  int Kmax = 1;
  int Kmax_gen = 1;
  int nnzb_S = 0;
  int C_edges = 0;
  int max_col_blocks = 0, max_col_branch = 0, nbranch = 1, nsep_blk = 0, max_row_blocks = 0;
  std::vector<int> extra_pairs;   // svs_ba_set_structure: pose pairs added to the block pattern
  bool extra_pairs_from_caller = false;   // set by svs_ba_set_structure (not by the in-library sharded window)
  // one window sharded by landmarks across ranks (SURVEY.md 8e): NCCL communicator of this handle
  NcclComm comm = nullptr; int comm_rank = 0, comm_size = 1;
  size_t sys_count = 0;            // doubles of the packed S | bp | bc buffer (one all-reduce per trial)
  int L_full = 0;                  // svs_ba_set_problem_sharded: landmarks of the whole window, 0 = not sharded
  // the loaded problem is this rank's share of a sharded window: optimize() sums across the communicator only then (a
  // whole window loaded by svs_ba_set_problem or the one-call API on a handle that has a communicator is solved alone)
  bool sharded = false;
  double* d_psi_all = nullptr; size_t psi_all_cap = 0;
  double* d_out = nullptr; double* h_out = nullptr; size_t out_cap = 0;   // accepted state in the caller's order (one-call API)
  bool export_next = false;
  // host scratch of set_problem, kept across calls (fresh multi-MB vectors page-fault every time)
  std::vector<std::pair<unsigned long long, int>> w_ko;
  std::vector<int> w_cnt, w_eptr, w_eord, w_fill, w_anchor, w_K, w_order, w_lm_eptr, w_lm_sptr, w_lm_anchor, w_ie_pose, w_bucket;
  std::vector<unsigned char> w_self, w_lm_self, w_adj, w_npad;
  std::vector<unsigned long long> w_key;
  std::vector<double> w_psi;
  std::vector<int> w_edge_src;
  cudaEvent_t ev[8] = {};
  // structure of the last problem (index arrays as the caller passed them): a call with the same structure --
  // the second optimize() of a back-end tick (backend.cpp:186-197), repeated measurement -- skips the structure
  // analysis and re-sends only the numbers
  std::vector<int> k_epoint, k_epose, k_eanchor, k_ci, k_cj, k_extra;
  std::vector<unsigned char> k_fixed;
  int k_P = -1, k_L = -1, k_E = -1, k_C = -1, k_flags = 0;
  size_t off_num = 0, off_cT = 0, off_cLam = 0, off_pose0 = 0, off_psi0 = 0, upload_bytes = 0;
  int reuse_hits = 0;
  // symbolic factorisation of the last pose graph: reused while the co-visibility pattern (P x P) stays the same,
  // which it does from tick to tick unless a keyframe enters or leaves the double window
  Symbolic k_sy; std::vector<unsigned char> k_adj; int k_adjP = -1, k_nbranch = 1, k_nsep = 0, k_nnzb = 0; bool k_natural = false;
  int symbolic_hits = 0;
  std::vector<cudaEvent_t> tev;   // per-trial timing events
  // last optimize() settings
};

namespace {

struct CudaErr {
  cudaError_t e;
  const char* what;
};

#define CK(call)                                                        \
  do {                                                                  \
    cudaError_t e_ = (call);                                            \
    if (e_ != cudaSuccess) {                                            \
      h->err = std::string(#call) + ": " + cudaGetErrorString(e_);      \
      return SVS_ERR_CUDA;                                              \
    }                                                                   \
  } while (0)

constexpr size_t kAlign = 256;

template <typename T>
int dev_alloc(svs_ba* h, T** p, size_t n) {
  const size_t bytes = ((std::max<size_t>(n, 1) * sizeof(T) + kAlign - 1) / kAlign) * kAlign;
  if (!h->measuring) *p = reinterpret_cast<T*>(h->arena + h->arena_off);
  h->arena_off += bytes;
  return SVS_OK;
}

// Uploads are laid out at the front of the arena, mirrored in the pinned staging buffer, and
// shipped with a single H2D copy (finish_upload).
template <typename T>
int dev_upload(svs_ba* h, const T** p, const T* src, size_t n) {
  const size_t off = h->arena_off;
  T* q = nullptr;
  dev_alloc(h, &q, n);
  if (!h->measuring) {
    if (n) {
      const size_t bytes = n * sizeof(T);
      if (bytes >= (1u << 20)) {   // multi-MB arrays (observations, weights): split the copy over a few threads
        const int parts = 4;
        h->pool.parallel_for(parts, [&](int q) {
          const size_t b0 = bytes * q / parts, b1 = bytes * (q + 1) / parts;
          memcpy(h->stage + off + b0, reinterpret_cast<const char*>(src) + b0, b1 - b0);
        });
      } else {
        memcpy(h->stage + off, src, bytes);
      }
    }
    *p = q;
  }
  return SVS_OK;
}
template <typename T>
int dev_upload(svs_ba* h, const T** p, const std::vector<T>& v) { return dev_upload(h, p, v.data(), v.size()); }

int arena_reserve(svs_ba* h, size_t total, size_t upload) {
  if (total > h->arena_cap) {
    if (h->arena) cudaFree(h->arena);
    h->arena = nullptr; h->arena_cap = 0;
    const size_t want = total + total / 4;
    CK(cudaMalloc((void**)&h->arena, want));
    h->arena_cap = want;
  }
  if (upload > h->stage_cap) {
    if (h->stage) cudaFreeHost(h->stage);
    h->stage = nullptr; h->stage_cap = 0;
    const size_t want = upload + upload / 4;
    CK(cudaMallocHost((void**)&h->stage, want));
    h->stage_cap = want;
  }
  return SVS_OK;
}

// Observations and weights in the caller's edge order, 6 doubles per edge: pinned staging + device copy, grown on
// demand.  A window assembled on the device (svs_ba_set_problem_from_map) never needs them, so a later host call
// with the same structure may find them missing or too small.
int raw_reserve(svs_ba* h, int E) {
  const size_t need = 6 * (size_t)E;
  if (need <= h->raw_cap) return SVS_OK;
  if (h->d_raw) cudaFree(h->d_raw);
  if (h->h_raw) cudaFreeHost(h->h_raw);
  h->d_raw = h->h_raw = nullptr; h->raw_cap = 0;
  const size_t want = need + need / 4;
  CK(cudaMalloc((void**)&h->d_raw, want * sizeof(double)));
  CK(cudaMallocHost((void**)&h->h_raw, want * sizeof(double)));
  h->raw_cap = want;
  return SVS_OK;
}

void free_problem(svs_ba* h) {
  h->has_problem = false;
  h->d = BaDev{};
}

void free_arena(svs_ba* h) {
  if (h->arena) cudaFree(h->arena);
  if (h->stage) cudaFreeHost(h->stage);
  if (h->d_raw) cudaFree(h->d_raw);
  if (h->h_raw) cudaFreeHost(h->h_raw);
  h->d_raw = h->h_raw = nullptr; h->raw_cap = 0;
  h->arena = nullptr; h->stage = nullptr; h->arena_cap = h->stage_cap = 0;
}

// Symbolic analysis of the reduced camera system: elimination order (greedy minimum degree on
// the pose graph, the role AMD plays inside LinearSolverCSparse), block fill, and the update
// lists of the right-looking block Cholesky.

// `order`: empty = greedy minimum degree (or the caller's order when `natural`), else the elimination
// order to use (nested dissection, see choose_branches).
void analyse(int P, const std::vector<std::vector<int>>& adj_in, bool natural, const std::vector<int>& order, Symbolic& sy) {
  // elimination graph as a byte matrix: P is a window of poses (hundreds to a few thousand)
  std::vector<unsigned char> G((size_t)P * P, 0);
  std::vector<int> deg(P, 0);
  for (int i = 0; i < P; ++i)
    for (int j : adj_in[i])
      if (j != i && !G[(size_t)i * P + j]) { G[(size_t)i * P + j] = 1; ++deg[i]; }
  sy.perm.assign(P, 0);
  sy.pos.assign(P, 0);
  std::vector<std::vector<int>> cols(P);  // by position: neighbours still alive when eliminated (as poses)
  std::vector<char> done(P, 0);
  std::vector<int> nb;
  for (int step = 0; step < P; ++step) {
    int v = step;
    if (!order.empty()) {
      v = order[step];
    } else if (!natural) {   // greedy minimum degree, ties to the lowest index
      int best = 1 << 30;
      for (int i = 0; i < P; ++i)
        if (!done[i] && deg[i] < best) { best = deg[i]; v = i; }
    }
    done[v] = 1;
    sy.perm[step] = v;
    sy.pos[v] = step;
    nb.clear();
    const unsigned char* row = G.data() + (size_t)v * P;
    for (int j = 0; j < P; ++j)
      if (row[j] && !done[j]) nb.push_back(j);
    cols[step] = nb;
    for (int a : nb) { G[(size_t)a * P + v] = 0; --deg[a]; }
    for (size_t x = 0; x < nb.size(); ++x)
      for (size_t y = x + 1; y < nb.size(); ++y) {
        const int p = nb[x], q = nb[y];
        if (!G[(size_t)p * P + q]) { G[(size_t)p * P + q] = 1; G[(size_t)q * P + p] = 1; ++deg[p]; ++deg[q]; }
      }
  }
  // column structures by position
  sy.col_ptr.assign(P + 1, 0);
  sy.row_idx.clear();
  for (int j = 0; j < P; ++j) {
    std::vector<int> rows;
    for (int a : cols[j]) rows.push_back(sy.pos[a]);
    std::sort(rows.begin(), rows.end());
    sy.col_ptr[j] = (int)sy.row_idx.size();
    sy.row_idx.push_back(j);
    for (int r : rows) sy.row_idx.push_back(r);
  }
  sy.col_ptr[P] = (int)sy.row_idx.size();
  sy.nblk = (int)sy.row_idx.size();
  // table (row pose, col pose) -> block<<1 | transpose.  Block (i,j), i >= j in position, stores rows <-> i.
  sy.tbl.assign((size_t)P * P, -1);
  for (int j = 0; j < P; ++j)
    for (int b = sy.col_ptr[j]; b < sy.col_ptr[j + 1]; ++b) {
      const int i = sy.row_idx[b];
      const int pi = sy.perm[i], pj = sy.perm[j];
      sy.tbl[(size_t)pi * P + pj] = b << 1;             // rows <-> pi: as stored
      if (i != j) sy.tbl[(size_t)pj * P + pi] = (b << 1) | 1;  // rows <-> pj: transpose on write
    }
  // update lists
  sy.upd_ptr.assign(P + 1, 0);
  sy.upd_dst.clear();
  sy.upd_ab.clear();
  for (int j = 0; j < P; ++j) {
    sy.upd_ptr[j] = (int)sy.upd_dst.size();
    const int base = sy.col_ptr[j] + 1, nb = sy.col_ptr[j + 1] - base;
    // b-major: the pairs (a, 0) that land in the next column to be factored come first
    for (int b = 0; b < nb; ++b)
      for (int a = b; a < nb; ++a) {
        const int ia = sy.row_idx[base + a], ib = sy.row_idx[base + b];  // ia >= ib
        const int t = sy.tbl[(size_t)sy.perm[ia] * P + sy.perm[ib]];
        sy.upd_dst.push_back(t >> 1);
        sy.upd_ab.push_back((a << 16) | b);
      }
  }
  sy.upd_ptr[P] = (int)sy.upd_dst.size();
  // row-major index of the off-diagonal blocks, columns descending inside a row: the backward pass walks the
  // rows from the last to the first and scatters x_i into the columns of row i
  {
    sy.rptr.assign(P + 1, 0);
    for (int j = 0; j < P; ++j)
      for (int b = sy.col_ptr[j] + 1; b < sy.col_ptr[j + 1]; ++b) sy.rptr[sy.row_idx[b] + 1]++;
    sy.max_row = 0;
    for (int i = 0; i < P; ++i) { sy.max_row = std::max(sy.max_row, sy.rptr[i + 1]); sy.rptr[i + 1] += sy.rptr[i]; }
    std::vector<int> fill(sy.rptr.begin(), sy.rptr.end() - 1);
    sy.rowpos.assign(sy.nblk, -1);
    sy.rcol.assign(sy.nblk - P > 0 ? sy.nblk - P : 0, 0);
    for (int j = P - 1; j >= 0; --j)
      for (int b = sy.col_ptr[j] + 1; b < sy.col_ptr[j + 1]; ++b) {
        const int at = fill[sy.row_idx[b]]++;
        sy.rowpos[b] = at;
        sy.rcol[at] = j;
      }
  }
  // urg_dst[col_ptr[j] + 1 + a] = destination of pair (a, 0) of column j
  sy.urg_dst.assign(sy.nblk, 0);
  for (int j = 0; j < P; ++j) {
    const int base = sy.col_ptr[j] + 1, nb = sy.col_ptr[j + 1] - base;
    for (int a = 0; a < nb; ++a) sy.urg_dst[base + a] = sy.upd_dst[sy.upd_ptr[j] + a];
  }
}

// Two-ended elimination for window-shaped pose graphs ("burn at both ends"): keyframes are
// temporal, so in the caller's order the co-visibility graph is banded (bandwidth w).  Team 0
// eliminates poses 0, 1, 2, ... and team 1 eliminates P-1, P-2, ... concurrently; they meet at a
// separator of w poses in the middle that is factored last.  Neither chain starts next to a
// separator, so no separator rows are dragged through the columns: the factor has the fill of the
// plain band, and the pivot chain is P/2 + w columns instead of P.  (A k-way dissection with k > 2
// was measured: interior parts drag their first separator through every column, the wider columns
// saturate the shared-memory pipe of the one SM that runs the factorisation, and nothing is gained.)
// Returns the number of branches (1 when the graph is not banded enough).
int choose_branches(int P, const std::vector<std::vector<int>>& adj, std::vector<int>& order,
                    std::vector<int>& branch_ptr) {
  order.clear();
  branch_ptr.clear();
  if (P < 8) return 1;
  // band width of the window WITHOUT its few long-range edges (loop closures, prepareForOptimization(root, loop_id)):
  // the smallest w that leaves at most kMaxLong edges longer than w
  constexpr int kMaxLong = 24;
  std::vector<int> hist(P, 0);
  for (int i = 0; i < P; ++i)
    for (int j : adj[i])
      if (j > i) hist[j - i]++;
  int w = P - 1, longer = 0;
  while (w > 0 && longer + hist[w] <= kMaxLong) { longer += hist[w]; --w; }
  if (w == 0 || (P - w) / 2 < 3 * w) return 1;
  const int left = (P - w) / 2;             // poses [0, left) | separator [left, left + w) | [left + w, P)
  auto side = [&](int p) { return p < left ? 0 : (p >= left + w ? 1 : 2); };
  // a long edge between the two ends would couple the concurrent eliminations: one of its poses joins the separator
  std::vector<char> in_sep(P, 0);
  for (int i = 0; i < P; ++i)
    for (int j : adj[i])
      if (j - i > w && side(i) + side(j) == 1 && !in_sep[i] && !in_sep[j]) in_sep[j] = 1;
  branch_ptr.push_back(0);
  for (int i = 0; i < left; ++i)
    if (!in_sep[i]) order.push_back(i);
  branch_ptr.push_back((int)order.size());
  for (int i = P - 1; i >= left + w; --i)
    if (!in_sep[i]) order.push_back(i);
  branch_ptr.push_back((int)order.size());
  for (int i = 0; i < P; ++i)
    if (in_sep[i]) order.push_back(i);
  for (int i = left; i < left + w; ++i) order.push_back(i);
  return 2;
}

// Track padding rule (set_problem_impl, 'Track padding'): a track of m >= 2 non-anchor observers lo..hi is completed
// with zero-weight edges to the np frames of lo..hi it skips (the anchor frame is never one of them) when the completed
// track has at most 8 slots and np <= max(1, m / 2).  Returns np (0: leave the track as it is).  The sharded window
// uses the same rule for the block pattern every rank must agree on.
inline int track_padding(int m, int lo, int hi, int anchor) {
  if (m < 2) return 0;
  const int span = hi - lo + 1 - ((anchor > lo && anchor < hi) ? 1 : 0);   // frames lo..hi without the anchor
  const int np = span - m;
  return (np > 0 && 1 + span <= 8 && np <= std::max(1, m / 2)) ? np : 0;
}

int fail(svs_ba* h, int code, const std::string& msg) {
  h->err = msg;
  return code;
}

}  // namespace

extern "C" {

int svs_device_info(char* buf, int buflen) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
    snprintf(buf, buflen, "no CUDA device");
    return SVS_ERR_NOGPU;
  }
  int dev = 0;
  cudaGetDevice(&dev);
  cudaDeviceProp pr;
  cudaGetDeviceProperties(&pr, dev);
  snprintf(buf, buflen, "%s;sm_%d%d;SMs=%d;smem_optin=%zu;l2=%d", pr.name, pr.major, pr.minor,
           pr.multiProcessorCount, pr.sharedMemPerBlockOptin, pr.l2CacheSize);
  return SVS_OK;
}

int svs_ba_create(const svs_ba_opts* opts, svs_ba** out) {
  if (!out) return SVS_ERR_INVALID;
  *out = nullptr;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) return SVS_ERR_NOGPU;
  svs_ba* h = new svs_ba();
  h->flags = opts ? opts->flags : 0;
  {   // threads of the per-landmark host loops of set_problem: a few, never more than half the machine
    const int hw = (int)std::thread::hardware_concurrency();
    h->host_threads = std::max(1, std::min(8, hw / 2));
  }
  if (const char* ht = getenv("SVS_HOST_THREADS")) h->host_threads = std::max(1, atoi(ht));
  h->pool.set_threads(h->host_threads);
  int dev = opts ? opts->device : -1;
  if (dev < 0) cudaGetDevice(&dev);
  h->device = dev;
  if (cudaSetDevice(dev) != cudaSuccess || cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaMallocHost(&h->h_ctl, sizeof(LmCtl)) != cudaSuccess) {
    delete h;
    return SVS_ERR_CUDA;
  }
  for (auto& e : h->ev) cudaEventCreate(&e);
  *out = h;
  return SVS_OK;
}

void svs_ba_destroy(svs_ba* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  cudaStreamSynchronize(h->stream);
  free_problem(h);
  free_arena(h);
  if (h->comm) { if (const NcclApi* nc = nccl_api()) nc->CommDestroy(h->comm); }
  if (h->d_psi_all) cudaFree(h->d_psi_all);
  if (h->d_out) cudaFree(h->d_out);
  if (h->h_out) cudaFreeHost(h->h_out);
  for (auto& e : h->ev) cudaEventDestroy(e);
  for (auto& e : h->tev) cudaEventDestroy(e);
  if (h->h_ctl) cudaFreeHost(h->h_ctl);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
}

const char* svs_last_error(const svs_ba* h) { return h ? h->err.c_str() : "null handle"; }

// d_obs_info != nullptr: the observations [E][3] followed by the weights [E][3] already lie on this device in
// the caller's edge order (assembled there, svs_ba_set_problem_from_map) and e_obs / e_info are not read.
static int set_problem_impl(svs_ba* h, int P, const double* T_qt, const unsigned char* fixed, int L, const double* psi,
                            int E, const int* e_point, const int* e_pose, const int* e_anchor, const double* e_obs,
                            const double* e_info, int C, const int* c_i, const int* c_j, const double* c_T,
                            const double* c_Lambda, const svs_cam* cam, const double* d_obs_info) {
  if (!h) return SVS_ERR_INVALID;
  if (P < 0 || L < 0 || E < 0 || C < 0 || !cam) return fail(h, SVS_ERR_INVALID, "negative size or null camera");
  if ((P && !T_qt) || (L && !psi) || (E && (!e_point || !e_pose || !e_anchor || (!d_obs_info && (!e_obs || !e_info)))) ||
      (C && (!c_i || !c_j || !c_T || !c_Lambda)))
    return fail(h, SVS_ERR_INVALID, "null array");
  // (the observation edges are range-checked inside the grouping pass below, which reads them anyway; the
  //  same-structure path compares them with an already validated list)
  for (int c = 0; c < C; ++c)
    if (c_i[c] < 0 || c_i[c] >= P || c_j[c] < 0 || c_j[c] >= P || c_i[c] == c_j[c])
      return fail(h, SVS_ERR_INVALID, "pose-pose edge index out of range");
  cudaSetDevice(h->device);
  h->pool.begin();   // the host loops below run on a few spinning threads until this call returns
  struct PoolEnd { SpinPool* p; ~PoolEnd() { p->end(); } } pool_end{&h->pool};
  CK(cudaStreamSynchronize(h->stream));   // the arena and the staging buffer are about to be reused
  const bool host_timing = getenv("SVS_HOST_TIMING") != nullptr;
  // ---- same structure as the problem on the device: only the numbers travel
  if (h->has_problem && !getenv("SVS_NO_STRUCT_REUSE") && P == h->k_P && L == h->k_L && E == h->k_E && C == h->k_C &&
      h->flags == h->k_flags && h->extra_pairs == h->k_extra &&
      (E == 0 || (memcmp(e_point, h->k_epoint.data(), sizeof(int) * E) == 0 && memcmp(e_pose, h->k_epose.data(), sizeof(int) * E) == 0 &&
                  memcmp(e_anchor, h->k_eanchor.data(), sizeof(int) * E) == 0)) &&
      (C == 0 || (memcmp(c_i, h->k_ci.data(), sizeof(int) * C) == 0 && memcmp(c_j, h->k_cj.data(), sizeof(int) * C) == 0))) {
    bool same_fixed = true;
    for (int p = 0; p < P && same_fixed; ++p) same_fixed = (fixed ? fixed[p] : 0) == h->k_fixed[p];
    if (same_fixed) {
      BaDev& d = h->d;
      d.f = cam->f; d.px = cam->px; d.py = cam->py; d.b = cam->b;
      if (E > 0 && !d_obs_info) {
        // staged in pinned memory and sent in two pieces, so that the first DMA runs under the second copy
        if (const int rc = raw_reserve(h, E)) return rc;
        const size_t bytes = 3 * (size_t)E * sizeof(double);
        const int parts = 4;
        for (int half = 0; half < 2; ++half) {
          const char* src = reinterpret_cast<const char*>(half ? e_info : e_obs);
          char* dst = reinterpret_cast<char*>(h->h_raw) + (half ? bytes : 0);
          h->pool.parallel_for(parts, [&](int q) {
            const size_t b0 = bytes * q / parts, b1 = bytes * (q + 1) / parts;
            memcpy(dst + b0, src + b0, b1 - b0);
          });
          CK(cudaMemcpyAsync(reinterpret_cast<char*>(h->d_raw) + (half ? bytes : 0), dst, bytes, cudaMemcpyHostToDevice, h->stream));
        }
      }
      if (C) {
        memcpy(h->stage + h->off_cT, c_T, 7 * (size_t)C * sizeof(double));
        memcpy(h->stage + h->off_cLam, c_Lambda, 36 * (size_t)C * sizeof(double));
      }
      if (P) memcpy(h->stage + h->off_pose0, T_qt, 7 * (size_t)P * sizeof(double));
      double* sp = reinterpret_cast<double*>(h->stage + h->off_psi0);
      for (int li = 0; li < L; ++li) {
        const double* src = psi + 3 * (size_t)h->lm_to_user[li];
        sp[3 * (size_t)li] = src[0]; sp[3 * (size_t)li + 1] = src[1]; sp[3 * (size_t)li + 2] = src[2];
      }
      CK(cudaMemcpyAsync(h->arena + h->off_num, h->stage + h->off_num, h->upload_bytes - h->off_num, cudaMemcpyHostToDevice,
                         h->stream));
      launch_regroup(d, d_obs_info ? d_obs_info : h->d_raw, h->stream);
      CK(cudaMemsetAsync(d.ticket, 0, 4 * sizeof(unsigned), h->stream));   // k_update's ticket, k_build_wave's task counter pair
      CK(cudaMemsetAsync(d.chi_c, 0, std::max(C, 1) * sizeof(double), h->stream));
      CK(cudaMemsetAsync(d.chi_c_new, 0, std::max(C, 1) * sizeof(double), h->stream));
      ++h->reuse_hits;
      if (host_timing) fprintf(stderr, "set_problem: structure reused (%d)\n", h->reuse_hits);
      return svs_ba_reset_state(h);
    }
  }
  free_problem(h);
  const int nthr = h->host_threads;
  (void)nthr;
  auto tp0 = std::chrono::steady_clock::now();
  auto lap = [&](const char* what) {
    if (!host_timing) return;
    auto now = std::chrono::steady_clock::now();
    fprintf(stderr, "set_problem %-12s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(now - tp0).count());
    tp0 = now;
  };

  // ---- observations and weights go to the device in the caller's edge order NOW: a helper thread stages them in
  //      pinned memory and enqueues the DMA (observations, then weights) while this thread analyses the structure; a
  //      gather kernel brings them into the internal order afterwards.  The helper also keeps the copy of the index
  //      arrays that the same-structure test of the next call compares against.
  if (E > 0 && !d_obs_info)
    if (const int rc = raw_reserve(h, E)) return rc;
  struct Side {   // (every return below waits for the helper: it reads the caller's arrays)
    Worker* w;
    cudaError_t err = cudaSuccess;
    ~Side() { w->wait(); }
  } side{&h->worker};
  {
    cudaError_t* perr = &side.err;
    h->worker.post([=]() {
      cudaSetDevice(h->device);
      if (E > 0 && !d_obs_info) {
        const size_t bytes = 3 * (size_t)E * sizeof(double);
        char* hr = reinterpret_cast<char*>(h->h_raw);
        char* dr = reinterpret_cast<char*>(h->d_raw);
        memcpy(hr, e_obs, bytes);
        const cudaError_t e1 = cudaMemcpyAsync(dr, hr, bytes, cudaMemcpyHostToDevice, h->stream);
        memcpy(hr + bytes, e_info, bytes);
        const cudaError_t e2 = cudaMemcpyAsync(dr + bytes, hr + bytes, bytes, cudaMemcpyHostToDevice, h->stream);
        *perr = e1 != cudaSuccess ? e1 : e2;
      }
      h->k_epoint.assign(e_point, e_point + E); h->k_epose.assign(e_pose, e_pose + E); h->k_eanchor.assign(e_anchor, e_anchor + E);
    });
  }
  lap("raw enqueue");
  // ---- group edges per landmark (counting sort), flat arrays only: this runs on the caller's
  //      thread inside the end-to-end time, like g2o's buildStructure does in the reference.
  //      Scratch lives in the handle; the per-landmark and per-edge loops use a few host threads.
  auto& eptr = h->w_eptr; auto& eord = h->w_eord; auto& fillp = h->w_fill;
  eptr.assign(L + 1, 0);
  eord.resize(E);
  {
    // stable counting sort by landmark on `nt` threads: per-thread histograms over contiguous edge ranges, one
    // prefix over (landmark, thread), per-thread scatter.  The index ranges are checked in the counting pass.
    const int nt = (E > 32768 && L > 0) ? nthr : 1;
    auto& cnt = h->w_cnt;
    cnt.resize((size_t)nt * (L + 1));
    std::atomic<int> out_of_range{0};
    h->pool.parallel_for(nt, [&](int t) {
      int* c = cnt.data() + (size_t)t * (L + 1);
      memset(c, 0, sizeof(int) * (size_t)(L + 1));   // every thread clears its own histogram
      const int e0 = (int)((long long)E * t / nt), e1 = (int)((long long)E * (t + 1) / nt);
      for (int e = e0; e < e1; ++e) {
        const int l = e_point[e];
        if (l < 0 || l >= L || e_pose[e] < 0 || e_pose[e] >= P || e_anchor[e] < 0 || e_anchor[e] >= P) { out_of_range.store(1); continue; }
        c[l]++;
      }
    });
    if (out_of_range.load()) return fail(h, SVS_ERR_INVALID, "observation edge index out of range");
    // prefix over (landmark, thread).  Only the prefix over the L landmark totals is serial; the totals and the
    // per-thread start offsets are computed on the pool over landmark ranges (the flat double loop was nt x L serial
    // steps and grew with the thread count: measured 0.26 ms of the grouping phase at 8 threads, 0.50 at 24)
    if (nt == 1) {
      int run = 0;
      for (int l = 0; l < L; ++l) { int& c = cnt[l]; const int n = c; eptr[l] = run; c = run; run += n; }
      eptr[L] = run;
    } else {
      h->pool.parallel_for(nt, [&](int r) {
        const int l0 = (int)((long long)L * r / nt), l1 = (int)((long long)L * (r + 1) / nt);
        for (int l = l0; l < l1; ++l) {
          int tot = 0;
          for (int t = 0; t < nt; ++t) tot += cnt[(size_t)t * (L + 1) + l];
          eptr[l + 1] = tot;   // totals first, turned into the prefix below
        }
      });
      eptr[0] = 0;
      for (int l = 0; l < L; ++l) eptr[l + 1] += eptr[l];
      h->pool.parallel_for(nt, [&](int r) {
        const int l0 = (int)((long long)L * r / nt), l1 = (int)((long long)L * (r + 1) / nt);
        for (int l = l0; l < l1; ++l) {
          int run = eptr[l];
          for (int t = 0; t < nt; ++t) { int& c = cnt[(size_t)t * (L + 1) + l]; const int n = c; c = run; run += n; }
        }
      });
    }
    h->pool.parallel_for(nt, [&](int t) {
      int* c = cnt.data() + (size_t)t * (L + 1);
      const int e0 = (int)((long long)E * t / nt), e1 = (int)((long long)E * (t + 1) / nt);
      for (int e = e0; e < e1; ++e) eord[c[e_point[e]]++] = e;
    });
  }
  // per landmark: anchor, self-observation flag, observer edges sorted by pose index (in place in eord)
  auto& l_anchor = h->w_anchor; auto& l_K = h->w_K; auto& l_self = h->w_self; auto& key = h->w_key;
  l_anchor.assign(L, -1); l_K.assign(L, 0); l_self.assign(L, 0); key.resize(L);
  // Track padding (SVS_BUILD_NO_PAD=1 switches it off): a track with a few visibility drop-outs -- observers
  // lo..hi with gaps -- is completed with ZERO-WEIGHT edges to the frames it skips, when the completed track still
  // fits the fused kernel (<= 8 slots) and at most half as many edges are added as there are.  A zero-weight edge
  // adds exactly 0 to every sum (linearize_edge / edge_cost return zeros for it without touching the projection),
  // so the reduced system, the update and chi2 are unchanged; what changes is that the landmark now has the slot
  // list of its undamaged neighbours and joins their run, instead of being a task of its own (20 % drop-outs on
  // the 200-keyframe window: 9 700 runs of 2 landmarks -> 3 600 runs of 6).
  auto& l_npad = h->w_npad;
  l_npad.assign(L, 0);
  const bool pad_tracks = getenv("SVS_BUILD_NO_PAD") == nullptr && !h->extra_pairs_from_caller;
  int Kmax = 1;
  int bad = 0;
  const int nchunk = L > 4096 ? 4 * nthr : 1;   // contiguous landmark ranges, handed out dynamically
  std::vector<int> c_kmax(nchunk, 1), c_bad(nchunk, 0);
  h->pool.parallel_for(nchunk, [&](int ck) {
    int Kmax = 1, bad = 0;
    for (int l = (int)((long long)L * ck / nchunk), l_end = (int)((long long)L * (ck + 1) / nchunk); l < l_end; ++l) {
      const int b = eptr[l], en = eptr[l + 1];
      key[l] = ~0ull;   // landmarks without observations go last
      if (b == en) continue;
      const int anchor = e_anchor[eord[b]];
      int nself = 0;
      for (int k = b; k < en; ++k) {
        const int e = eord[k];
        if (e_anchor[e] != anchor) bad = std::max(bad, 1);
        if (e_pose[e] == anchor) ++nself;
      }
      // insertion sort by (is-not-self, pose): the self edge first, then ascending pose index
      for (int k = b + 1; k < en; ++k) {
        const int e = eord[k];
        const int ke = e_pose[e] == anchor ? -1 : e_pose[e];
        int q = k - 1;
        while (q >= b) {
          const int f = eord[q];
          const int kf = e_pose[f] == anchor ? -1 : e_pose[f];
          if (kf <= ke) break;
          eord[q + 1] = f;
          --q;
        }
        eord[q + 1] = e;
      }
      for (int k = b + 1; k < en; ++k)
        if (e_pose[eord[k]] == e_pose[eord[k - 1]]) bad = std::max(bad, 2);
      int K = 1 + (en - b) - nself;
      if (pad_tracks && bad == 0 && nself <= 1 && en - b - nself >= 2) {
        const int np = track_padding(en - b - nself, e_pose[eord[b + nself]], e_pose[eord[en - 1]], anchor);
        if (np > 0) { l_npad[l] = (unsigned char)np; K += np; }
      }
      l_anchor[l] = anchor; l_self[l] = (unsigned char)nself; l_K[l] = K;
      Kmax = std::max(Kmax, K);
      // locality key: track shape (self flag, length, first and last observer) inside an anchor, so that
      // neighbouring warps of the fused kernel scatter into the same blocks of the reduced system
      const unsigned long long first = (unsigned long long)(e_pose[eord[b + (nself ? 1 : 0) < en ? b + (nself ? 1 : 0) : b]] & 0xfffff);
      const unsigned long long last = (unsigned long long)(e_pose[eord[en - 1]] & 0xfffff);
      key[l] = ((unsigned long long)(nself ? 0 : 1) << 61) | ((unsigned long long)(K & 0xfffff) << 40) | (first << 20) | last;
    }
    c_kmax[ck] = Kmax; c_bad[ck] = bad;
  });
  for (int ck = 0; ck < nchunk; ++ck) { Kmax = std::max(Kmax, c_kmax[ck]); bad = std::max(bad, c_bad[ck]); }
  if (bad == 1) return fail(h, SVS_ERR_UNSUPPORTED, "edges of one point name different anchor frames");
  if (bad == 2) return fail(h, SVS_ERR_UNSUPPORTED, "a point is observed twice by the same frame");
  lap("group");
  // internal landmark order: bucket by anchor (counting sort), then by track shape inside a bucket
  auto& order = h->w_order; auto& bucket = h->w_bucket;
  order.resize(L);
  bucket.assign(P + 2, 0);
  for (int l = 0; l < L; ++l) bucket[(l_anchor[l] < 0 ? P : l_anchor[l]) + 1]++;
  for (int a = 0; a <= P; ++a) bucket[a + 1] += bucket[a];
  {
    // (key, landmark) pairs side by side: the comparisons of the per-anchor sorts touch no other array
    auto& cur = fillp;
    cur.assign(bucket.begin(), bucket.end() - 1);
    auto& ko = h->w_ko;
    ko.resize(L);
    for (int l = 0; l < L; ++l) ko[cur[l_anchor[l] < 0 ? P : l_anchor[l]]++] = std::make_pair(key[l], l);
    h->pool.parallel_for((P + 1 + 7) / 8, [&](int ck) {
      for (int a = 8 * ck; a <= P && a < 8 * ck + 8; ++a) {
        std::sort(ko.begin() + bucket[a], ko.begin() + bucket[a + 1]);
        for (int i = bucket[a]; i < bucket[a + 1]; ++i) order[i] = ko[i].second;
      }
    });
  }
  h->lm_to_user = order;
  lap("order");
  auto& lm_eptr = h->w_lm_eptr; auto& lm_sptr = h->w_lm_sptr; auto& lm_anchor = h->w_lm_anchor; auto& ie_pose = h->w_ie_pose;
  auto& lm_self = h->w_lm_self; auto& edge_src = h->w_edge_src; auto& ipsi = h->w_psi;
  lm_eptr.assign(L + 1, 0); lm_sptr.assign(L + 1, 0); lm_anchor.assign(L, 0);
  lm_self.assign(L, 0); ipsi.resize(3 * (size_t)L);
  for (int li = 0; li < L; ++li) {
    const int l = order[li];
    lm_eptr[li + 1] = lm_eptr[li] + (eptr[l + 1] - eptr[l]) + l_npad[l];
    lm_sptr[li + 1] = lm_sptr[li] + l_K[l];
  }
  const int ne = lm_eptr[L], ns = lm_sptr[L];   // ne = E + padding edges: the internal edge count
  ie_pose.resize(ne); edge_src.resize(ne);
  h->pool.parallel_for(nchunk, [&](int ck) {
    for (int li = (int)((long long)L * ck / nchunk), li_end = (int)((long long)L * (ck + 1) / nchunk); li < li_end; ++li) {
      const int l = order[li];
      for (int q = 0; q < 3; ++q) ipsi[3 * (size_t)li + q] = psi[3 * (size_t)l + q];
      if (l_anchor[l] < 0) continue;
      lm_anchor[li] = l_anchor[l]; lm_self[li] = l_self[l];
      int at = lm_eptr[li];
      if (l_npad[l] == 0) {
        for (int k = eptr[l]; k < eptr[l + 1]; ++k, ++at) {
          const int e = eord[k];
          ie_pose[at] = e_pose[e];
          edge_src[at] = e;   // the doubles follow on the device (k_regroup)
        }
      } else {   // completed track: the self edge, then every frame lo..hi but the anchor; -1 = zero-weight padding edge
        int k = eptr[l];
        const int en = eptr[l + 1], anchor = l_anchor[l];
        if (l_self[l]) { ie_pose[at] = anchor; edge_src[at++] = eord[k++]; }
        const int lo = e_pose[eord[k]], hi = e_pose[eord[en - 1]];
        for (int p = lo; p <= hi; ++p) {
          if (p == anchor) continue;
          ie_pose[at] = p;
          if (k < en && e_pose[eord[k]] == p) edge_src[at++] = eord[k++];
          else edge_src[at++] = -1;
        }
      }
    }
  });
  lap("fill");
  // ---- work lists of the fused kernel: runs of landmarks with identical slot lists (<= 8 frames)
  std::vector<int> task_lm, task_cnt, gen_lm, long_lm;   // long_lm: more than kMaxTrack slots (streaming kernel, any length)
  int Kmax_gen = 1;
  {
    // landmarks per task.  Measured on B200 with the persistent grid (1 184 resident warps), build kernel per trial on
    // the 200-keyframe window / with 20 % drop-outs: chunk 8: 0.100 / 0.116 ms, 12: 0.095 / 0.113, 16: 0.097 / 0.110,
    // 20: 0.108 / 0.113, 24: 0.125 / 0.127, 32: 0.156 / 0.159 (fewer flushes against a coarser tail); the
    // 1 000-keyframe window is flat from 32 up
    int chunk = L / (148 * 11);
    chunk = chunk < 4 ? 4 : (chunk > 32 ? 32 : chunk);
    if (const char* cs = getenv("SVS_BUILD_CHUNK")) chunk = atoi(cs);   // tuning knob
    if (getenv("SVS_BUILD_V1")) chunk = 0;   // A/B switch: everything through the one-warp-per-landmark kernel
    auto same_slots = [&](int la, int lb) {   // internal indices
      const int ka = lm_eptr[la + 1] - lm_eptr[la], kb = lm_eptr[lb + 1] - lm_eptr[lb];
      if (ka != kb || lm_anchor[la] != lm_anchor[lb] || lm_self[la] != lm_self[lb]) return false;
      for (int i = 0; i < ka; ++i)
        if (ie_pose[lm_eptr[la] + i] != ie_pose[lm_eptr[lb] + i]) return false;
      return true;
    };
    // built on `nt` threads over contiguous landmark ranges (a run never spans two ranges), concatenated in order
    const int nt = L > 4096 ? nthr : 1;
    std::vector<std::vector<int>> t_lm(nt), t_cnt(nt), t_gen(nt), t_long(nt);
    std::vector<int> t_kmax(nt, 1);
    h->pool.parallel_for(nt, [&](int t) {
      auto& tl = t_lm[t]; auto& tc = t_cnt[t];
      const int l0 = (int)((long long)L * t / nt), l1 = (int)((long long)L * (t + 1) / nt);
      for (int li = l0; li < l1; ++li) {
        const int kk = lm_eptr[li + 1] - lm_eptr[li], KK = lm_sptr[li + 1] - lm_sptr[li];
        if (kk > 0 && KK > kMaxTrack) { t_long[t].push_back(li); continue; }
        if (chunk == 0 || kk == 0 || KK > 8) {
          t_gen[t].push_back(li);
          t_kmax[t] = std::max(t_kmax[t], KK);
          continue;
        }
        // (rounding the limit to whole 32-edge waves of the track shape was measured: no difference)
        if (!tl.empty() && tl.back() + tc.back() == li && tc.back() < chunk && same_slots(tl.back(), li))
          tc.back()++;
        else { tl.push_back(li); tc.push_back(1); }
      }
    });
    for (int t = 0; t < nt; ++t) {
      task_lm.insert(task_lm.end(), t_lm[t].begin(), t_lm[t].end());
      task_cnt.insert(task_cnt.end(), t_cnt[t].begin(), t_cnt[t].end());
      gen_lm.insert(gen_lm.end(), t_gen[t].begin(), t_gen[t].end());
      long_lm.insert(long_lm.end(), t_long[t].begin(), t_long[t].end());
      Kmax_gen = std::max(Kmax_gen, t_kmax[t]);
    }
    // longest tasks first: the warps of the persistent k_build_wave draw tasks from one counter, so the short
    // tasks fill the end of the launch.  Cost = waves (<= 32 edges, 40 slots, 8 landmarks each); a stable counting
    // sort by waves, descending (landmark order inside a class is kept for the locality of the scatter)
    if (!getenv("SVS_BUILD_NO_LPT") && task_lm.size() > 1) {
      const size_t nt_all = task_lm.size();
      constexpr int kMaxWaves = 64;
      std::vector<unsigned char> wv(nt_all);
      int hist[kMaxWaves + 1] = {};
      for (size_t t = 0; t < nt_all; ++t) {
        const int li = task_lm[t], cnt = task_cnt[t];
        const int kk = lm_eptr[li + 1] - lm_eptr[li], KK = lm_sptr[li + 1] - lm_sptr[li];
        const int nw_max = std::max(1, std::min(std::min(32 / std::max(kk, 1), 40 / std::max(KK, 1)), 8));
        const int waves = std::min((cnt + nw_max - 1) / nw_max, kMaxWaves);
        wv[t] = (unsigned char)waves;
        hist[waves]++;
      }
      int start[kMaxWaves + 1];
      for (int w = kMaxWaves, at = 0; w >= 0; --w) { start[w] = at; at += hist[w]; }
      std::vector<int> lm2(nt_all), cnt2(nt_all);
      for (size_t t = 0; t < nt_all; ++t) { const int at = start[wv[t]]++; lm2[at] = task_lm[t]; cnt2[at] = task_cnt[t]; }
      task_lm.swap(lm2); task_cnt.swap(cnt2);
    }
  }

  lap("tasks");
  // ---- pose graph of the reduced system: co-visibility (all pairs inside a track) + constraints
  std::vector<std::vector<int>> adj(P);
  {
    auto& A = h->w_adj;
    A.assign((size_t)P * P, 0);
    // one representative per task (its landmarks share one slot list) + the landmarks outside the task lists; a
    // track has no length limit (slam_graph.cpp:1001-1027)
    auto mark = [&](int li) {   // internal landmark index
      const int b = lm_eptr[li] + lm_self[li], en = lm_eptr[li + 1], a = lm_anchor[li];
      for (int x = b; x < en; ++x) {
        const int px = ie_pose[x];
        A[(size_t)a * P + px] = 1; A[(size_t)px * P + a] = 1;
        for (int y = x + 1; y < en; ++y) { const int py = ie_pose[y]; A[(size_t)px * P + py] = 1; A[(size_t)py * P + px] = 1; }
      }
    };
    for (int li : task_lm) mark(li);
    for (int li : gen_lm)
      if (lm_eptr[li + 1] > lm_eptr[li]) mark(li);
    for (int li : long_lm) mark(li);
    for (int c = 0; c < C; ++c) { A[(size_t)c_i[c] * P + c_j[c]] = 1; A[(size_t)c_j[c] * P + c_i[c]] = 1; }
    for (size_t q = 0; q + 1 < h->extra_pairs.size(); q += 2) {   // svs_ba_set_structure
      const int a = h->extra_pairs[q], b = h->extra_pairs[q + 1];
      if (a < 0 || b < 0 || a >= P || b >= P) return fail(h, SVS_ERR_INVALID, "structure pair out of range");
      if (a != b) { A[(size_t)a * P + b] = 1; A[(size_t)b * P + a] = 1; }
    }
    int nnz = 0;
    for (int i = 0; i < P; ++i) {
      const unsigned char* row = A.data() + (size_t)i * P;
      for (int j = 0; j < P; ++j)
        if (row[j] && j != i) adj[i].push_back(j);
      nnz += (int)adj[i].size();
    }
    h->nnzb_S = nnz / 2 + P;
  }
  lap("adjacency");
  Symbolic sy;
  const bool natural_order = (h->flags & SVS_BA_NATURAL_ORDER) != 0;
  const bool chain_only = getenv("SVS_SOLVE_CHAIN") != nullptr;
  if (h->k_adjP == P && h->k_natural == natural_order && !chain_only && !getenv("SVS_NO_STRUCT_REUSE") &&
      h->k_adj.size() == h->w_adj.size() && memcmp(h->k_adj.data(), h->w_adj.data(), h->w_adj.size()) == 0) {
    sy = h->k_sy;
    h->nbranch = h->k_nbranch; h->nsep_blk = h->k_nsep;
    ++h->symbolic_hits;
    if (host_timing) fprintf(stderr, "set_problem: symbolic factorisation reused (%d)\n", h->symbolic_hits);
  } else {
    // two concurrent branches when the window is banded and each team's share of k_solve's
    // shared-memory ring holds its widest columns, else a single chain (minimum degree order)
    const bool natural = natural_order;
    int G = (natural || getenv("SVS_SOLVE_CHAIN")) ? 1 : 2;
    for (;;) {
      std::vector<int> order, bptr;
      G = G > 1 ? choose_branches(P, adj, order, bptr) : 1;
      analyse(P, adj, natural, order, sy);
      if (G == 1) { sy.branch_ptr = {0, P}; h->nsep_blk = 0; }
      else sy.branch_ptr = bptr;
      const int sep0 = sy.branch_ptr[G];
      sy.max_col_branch = sy.max_col_sep = 0;
      for (int j = 0; j < P; ++j) {
        const int nb = sy.col_ptr[j + 1] - sy.col_ptr[j] - 1;
        if (G > 1 && j < sep0) sy.max_col_branch = std::max(sy.max_col_branch, nb);
        else sy.max_col_sep = std::max(sy.max_col_sep, nb);
      }
      if (G == 1) break;
      // each end of the window is factored by its own CTA: its ring must hold four of the widest columns
      const int nsep = sy.nblk - sy.col_ptr[sep0];
      const int cap = solve_ring_capacity(P, sy.nblk, nsep);
      if (cap >= 4 * (sy.max_col_branch + 1) && cap / 2 >= sy.max_col_sep + 2) { h->nsep_blk = nsep; break; }
      G /= 2;
    }
    h->nbranch = (int)sy.branch_ptr.size() - 1;
    if (!chain_only) { h->k_sy = sy; h->k_adj = h->w_adj; h->k_adjP = P; h->k_natural = natural_order; h->k_nbranch = h->nbranch; h->k_nsep = h->nsep_blk; }
  }
  if (sy.nblk >= (1 << 20)) return fail(h, SVS_ERR_UNSUPPORTED, "reduced system factor has more than 2^20 blocks");

  lap("analyse");
  // ---- device image: constant arrays (uploaded in one copy) followed by work buffers
  BaDev& d = h->d;
  d.P = P; d.L = L; d.E = ne; d.E_user = E; d.C = C; d.nslots = ns; d.nblk = sy.nblk; d.flags = h->flags;
  d.f = cam->f; d.px = cam->px; d.py = cam->py; d.b = cam->b;
  std::vector<unsigned char> fx(P, 0);
  if (fixed) fx.assign(fixed, fixed + P);
  const double* d_pose0c = nullptr;
  const double* d_psi0c = nullptr;
  size_t upload_bytes = 0;
  auto lay = [&]() {
    h->arena_off = 0;
#define UP(field, vec) dev_upload(h, &d.field, vec)
    UP(fixed, fx); UP(lm_eptr, lm_eptr); UP(lm_sptr, lm_sptr); UP(lm_anchor, lm_anchor); UP(lm_self, lm_self); UP(lm_user, h->lm_to_user);
    UP(e_pose, ie_pose); UP(edge_src, edge_src);
    UP(task_lm, task_lm); UP(task_cnt, task_cnt); UP(gen_lm, gen_lm); UP(long_lm, long_lm);
    UP(tbl, sy.tbl); UP(perm, sy.perm); UP(pos, sy.pos); UP(col_ptr, sy.col_ptr); UP(row_idx, sy.row_idx);
    UP(upd_ptr, sy.upd_ptr); UP(upd_dst, sy.upd_dst); UP(upd_ab, sy.upd_ab); UP(urg_dst, sy.urg_dst);
    UP(branch_ptr, sy.branch_ptr); UP(rptr, sy.rptr); UP(rowpos, sy.rowpos); UP(rcol, sy.rcol);
    dev_upload(h, &d.c_i, c_i, (size_t)C); dev_upload(h, &d.c_j, c_j, (size_t)C);
    h->off_num = h->off_cT = h->arena_off;   // the numbers (everything a same-structure call re-sends) lie last
    dev_upload(h, &d.c_T, c_T, 7 * (size_t)C);
    h->off_cLam = h->arena_off;
    dev_upload(h, &d.c_Lam, c_Lambda, 36 * (size_t)C);
    h->off_pose0 = h->arena_off;
    dev_upload(h, &d_pose0c, T_qt, 7 * (size_t)P);
    h->off_psi0 = h->arena_off;
    dev_upload(h, &d_psi0c, ipsi.data(), 3 * (size_t)L);
#undef UP
    upload_bytes = h->arena_off;
    h->upload_bytes = upload_bytes;
#define AL(field, n) dev_alloc(h, &d.field, (size_t)(n))
    for (int b = 0; b < 2; ++b) { AL(pose[b], 7 * (size_t)P); AL(Rt[b], 12 * (size_t)P); AL(psi[b], 3 * (size_t)L); }
    AL(e_obs_w, 3 * (size_t)ne); AL(e_w_w, 3 * (size_t)ne);
    AL(W, 18 * (size_t)ns); AL(Dbl, 12 * (size_t)L); AL(chi_l, L); AL(chi_new_l, L); AL(scale_l, L);
    {   // reduced system S | bp | bc | totals in ONE buffer: a sharded window sums it with a single all-reduce
      double* sys = nullptr;
      dev_alloc(h, &sys, 36 * (size_t)sy.nblk + 12 * (size_t)P + 4);
      if (!h->measuring) { d.S = sys; d.bp = sys + 36 * (size_t)sy.nblk; d.bc = d.bp + 6 * (size_t)P; d.totals = d.bc + 6 * (size_t)P; }
      h->sys_count = 36 * (size_t)sy.nblk + 12 * (size_t)P;
    }
    AL(x, 6 * (size_t)P); AL(Nrow, 36 * (size_t)std::max(sy.nblk - P, 1));
    AL(chi_c, C); AL(chi_c_new, C); AL(Linv, 36 * (size_t)P); AL(ywork, 6 * (size_t)P);
    AL(ctl, 1);
    AL(part, 3 * (size_t)update_grid_blocks(L, C)); AL(ticket, 4); AL(dbg, 160);
#undef AL
  };
  h->measuring = true;
  lay();
  h->measuring = false;
  int rc;
  if ((rc = arena_reserve(h, h->arena_off, upload_bytes))) return rc;
  lay();
  lap("stage");
  h->worker.wait();   // its DMA is in the stream ahead of everything enqueued below
  if (side.err != cudaSuccess) return fail(h, SVS_ERR_CUDA, cudaGetErrorString(side.err));
  h->d_pose0 = const_cast<double*>(d_pose0c);
  h->d_psi0 = const_cast<double*>(d_psi0c);
  CK(cudaMemcpyAsync(h->arena, h->stage, upload_bytes, cudaMemcpyHostToDevice, h->stream));
  d.e_obs = d.e_obs_w; d.e_w = d.e_w_w;
  launch_regroup(d, d_obs_info ? d_obs_info : h->d_raw, h->stream);   // [3][E] internal order <- [E][3] user order
  CK(cudaMemsetAsync(d.ticket, 0, 4 * sizeof(unsigned), h->stream));   // k_update's ticket, k_build_wave's task counter pair
  CK(cudaMemsetAsync(d.dbg, 0, 160 * sizeof(long long), h->stream));
  h->max_col_blocks = sy.max_col_sep; h->max_col_branch = sy.max_col_branch; h->max_row_blocks = sy.max_row;
  d.nbranch = h->nbranch;
  CK(cudaMemsetAsync(d.chi_c, 0, std::max(C, 1) * sizeof(double), h->stream));
  CK(cudaMemsetAsync(d.chi_c_new, 0, std::max(C, 1) * sizeof(double), h->stream));
  h->Kmax = Kmax;
  h->Kmax_gen = Kmax_gen;
  d.ntasks = (int)task_lm.size(); d.ngen = (int)gen_lm.size(); d.nlong = (int)long_lm.size();
  h->C_edges = C;
  h->has_problem = true;
  h->k_P = P; h->k_L = L; h->k_E = E; h->k_C = C; h->k_flags = h->flags; h->k_extra = h->extra_pairs;
  h->k_ci.assign(c_i, c_i + C); h->k_cj.assign(c_j, c_j + C);
  h->k_fixed = fx;
  return svs_ba_reset_state(h);
}

int svs_ba_set_problem(svs_ba* h, int P, const double* T_qt, const unsigned char* fixed, int L, const double* psi,
                       int E, const int* e_point, const int* e_pose, const int* e_anchor, const double* e_obs,
                       const double* e_info, int C, const int* c_i, const int* c_j, const double* c_T,
                       const double* c_Lambda, const svs_cam* cam) {
  svs::NvtxRange nvtx_("copyDataToG2o");
  if (h) { h->L_full = 0; h->sharded = false; }
  return set_problem_impl(h, P, T_qt, fixed, L, psi, E, e_point, e_pose, e_anchor, e_obs, e_info, C, c_i, c_j, c_T, c_Lambda,
                          cam, nullptr);
}

int svs_ba_reset_state(svs_ba* h) {
  if (!h || !h->has_problem) return h ? fail(h, SVS_ERR_STATE, "no problem set") : SVS_ERR_INVALID;
  cudaSetDevice(h->device);
  BaDev& d = h->d;
  CK(cudaMemcpyAsync(d.pose[0], h->d_pose0, 7 * (size_t)d.P * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
  CK(cudaMemcpyAsync(d.psi[0], h->d_psi0, 3 * (size_t)d.L * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
  LmCtl z{};
  *h->h_ctl = z;
  h->cur_known = 0;
  CK(cudaMemcpyAsync(d.ctl, h->h_ctl, sizeof(LmCtl), cudaMemcpyHostToDevice, h->stream));
  launch_prep(d, 0, h->stream);
  CK(cudaGetLastError());
  return SVS_OK;
}

static int clear_system(svs_ba* h) {
  BaDev& d = h->d;
  CK(cudaMemsetAsync(d.S, 0, 36 * (size_t)d.nblk * sizeof(double), h->stream));
  CK(cudaMemsetAsync(d.bp, 0, 6 * (size_t)std::max(d.P, 1) * sizeof(double), h->stream));
  CK(cudaMemsetAsync(d.bc, 0, 6 * (size_t)std::max(d.P, 1) * sizeof(double), h->stream));
  return SVS_OK;
}

int svs_ba_optimize(svs_ba* h, int num_iters, int robust, double huber_delta, double lambda_init, int max_trials,
                    svs_ba_stats* st) {
  svs::NvtxRange nvtx_("optimize");
  if (!h) return -100 + SVS_ERR_INVALID;
  if (!h->has_problem) { h->err = "no problem set"; return -100 + SVS_ERR_STATE; }
  if (st) memset(st, 0, sizeof *st);
  BaDev& d = h->d;
  if (d.P == 0) return -1;   // g2o: "0 vertices to optimize"
  cudaSetDevice(h->device);
  int rc;
  int trials_seen = 0;
#define CKO(call)                                                       \
  do {                                                                  \
    cudaError_t e_ = (call);                                            \
    if (e_ != cudaSuccess) {                                            \
      h->err = std::string(#call) + ": " + cudaGetErrorString(e_);      \
      return -100 + SVS_ERR_CUDA;                                       \
    }                                                                   \
  } while (0)
  // LM state is not carried across calls (slam_graph.cpp:338-342, SURVEY B3); the accepted
  // state stays where the previous call (or set_problem) left it.
  if (h->cur_known < 0) {   // someone else may have flipped the state buffers: ask the device
    CKO(cudaMemcpyAsync(h->h_ctl, d.ctl, sizeof(LmCtl), cudaMemcpyDeviceToHost, h->stream));
    CKO(cudaStreamSynchronize(h->stream));
    h->cur_known = h->h_ctl->cur;
  }
  {
    const int cur = h->cur_known;   // known on the host: no round trip while the upload is still in flight
    h->cur_known = -1;
    LmCtl z{};
    z.cur = cur; z.lambda = lambda_init; z.ni = 2; z.max_trials = max_trials; z.max_iters = num_iters;
    *h->h_ctl = z;
    CKO(cudaMemcpyAsync(d.ctl, h->h_ctl, sizeof(LmCtl), cudaMemcpyHostToDevice, h->stream));
  }
  if ((rc = clear_system(h))) return -100 + rc;
  float ms[4] = {0, 0, 0, 0};  // build, solve, update(+decision), collectives
  int launches = 0;
  CKO(cudaEventRecord(h->ev[0], h->stream));
  int it = 0;
  const NcclApi* nc = h->comm && h->sharded ? nccl_api() : nullptr;   // sharded window: sums across ranks on this stream
  if (h->comm && h->sharded && !nc) { h->err = "NCCL library not loadable"; return -100 + SVS_ERR_STATE; }
  const int per_trial = 2 + ((d.ntasks > 0 || d.C > 0) ? 1 : 0) + (d.ngen > 0 ? 1 : 0) + (d.nlong > 0 ? 1 : 0) + (nc ? 1 : 0);
#define CKN(call)                                                       \
  do {                                                                  \
    const int e_ = (call);                                              \
    if (e_ != 0) {                                                      \
      h->err = std::string(#call) + ": " + nc->GetErrorString(e_);      \
      return -100 + SVS_ERR_CUDA;                                       \
    }                                                                   \
  } while (0)
  constexpr int kEv = 6;   // events per trial: start | built | summed | solved | updated | decided
  for (;;) {
    // Enqueue one Levenberg trial per remaining iteration without waiting for the device: every
    // trial is the same launch sequence, and the device-side control block decides whether a trial
    // is the next iteration or the retry of a rejected step.  Trials enqueued past the end (or after
    // Terminate) return at once (LmCtl::max_iters).  Only rejected steps cost another round trip.
    const int ntr = num_iters - it;
    while ((int)h->tev.size() < kEv * ntr) { cudaEvent_t e; cudaEventCreate(&e); h->tev.push_back(e); }
    for (int k = 0; k < ntr; ++k) {
      CKO(cudaEventRecord(h->tev[kEv * k + 0], h->stream));
      launch_build(d, h->Kmax_gen, robust, huber_delta, h->stream);
      CKO(cudaEventRecord(h->tev[kEv * k + 1], h->stream));
      // every rank holds the partial reduced system of its landmarks: ONE all-reduce of S | bp | bc
      if (nc) CKN(nc->AllReduce(d.S, d.S, h->sys_count, kNcclFloat64, kNcclSum, h->comm, h->stream));
      CKO(cudaEventRecord(h->tev[kEv * k + 2], h->stream));
      launch_solve(d, h->max_col_branch, std::max(h->max_col_blocks, h->max_row_blocks - 2), h->nsep_blk, h->stream);
      CKO(cudaEventRecord(h->tev[kEv * k + 3], h->stream));
      launch_update(d, robust, huber_delta, nc ? 1 : 0, h->stream);
      CKO(cudaEventRecord(h->tev[kEv * k + 4], h->stream));
      if (nc) {   // chi2 (accepted, trial) and the gain-ratio denominator of this rank's landmarks -> the same decision everywhere
        CKN(nc->AllReduce(d.totals, d.totals, 3, kNcclFloat64, kNcclSum, h->comm, h->stream));
        launch_decide_deferred(d, h->stream);
      }
      CKO(cudaEventRecord(h->tev[kEv * k + 5], h->stream));
    }
    CKO(cudaMemcpyAsync(h->h_ctl, d.ctl, sizeof(LmCtl), cudaMemcpyDeviceToHost, h->stream));
    if (h->export_next) {   // one-call API: the accepted state rides back with the control block, in the caller's order
      const size_t n = 7 * (size_t)d.P + 3 * (size_t)d.L;
      launch_export(d, h->d_out, h->stream);
      CKO(cudaMemcpyAsync(h->h_out, h->d_out, n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    }
    CKO(cudaStreamSynchronize(h->stream));
    CKO(cudaGetLastError());
    const int done_trials = h->h_ctl->trials_total - trials_seen;
    trials_seen = h->h_ctl->trials_total;
    launches += per_trial * done_trials;
    for (int k = 0; k < done_trials && k < ntr; ++k) {
      static const int slot[kEv - 1] = {0, 3, 1, 2, 3};   // build | collective | solve | update | collective + decision
      for (int q = 0; q < kEv - 1; ++q) {
        float t = 0;
        cudaEventElapsedTime(&t, h->tev[kEv * k + q], h->tev[kEv * k + q + 1]);
        ms[slot[q]] += t;
      }
    }
    it = h->h_ctl->iter;
    if (it >= num_iters || (h->h_ctl->stop && !h->h_ctl->again)) break;
  }
  CKO(cudaEventRecord(h->ev[6], h->stream));
  CKO(cudaEventSynchronize(h->ev[6]));
  h->cur_known = h->h_ctl->cur;   // read back after the last trial of this call
  if (st) {
    const LmCtl& c = *h->h_ctl;
    st->iterations = c.iter;
    st->trials_total = c.trials_total;
    st->chi2_init = c.chi_init;
    st->chi2_final = c.chi_cur;
    st->lambda_final = c.lambda;
    for (int i = 0; i < c.iter && i < SVS_BA_MAX_ITERS; ++i) {
      st->chi2_iter[i] = c.chi_iter[i];
      st->lambda_iter[i] = c.lambda_iter[i];
      st->trials_iter[i] = c.trials_iter[i];
    }
    st->num_frames = d.P; st->num_points = d.L; st->num_point_edges = d.E_user; st->num_frame_edges = d.C;
    st->nnzb_S = h->nnzb_S; st->nnzb_L = d.nblk; st->max_track = h->Kmax;
    cudaEventElapsedTime(&st->ms_total, h->ev[0], h->ev[6]);
    st->ms_build = ms[0]; st->ms_solve = ms[1]; st->ms_update = ms[2]; st->ms_control = ms[3];
    st->launches = launches;
  }
  if (getenv("SVS_BUILD_TIMING")) {
    long long dbg[64];
    cudaMemcpy(dbg, d.dbg, sizeof dbg, cudaMemcpyDeviceToHost);
    fprintf(stderr, "k_build_wave warp-cycles summed over warps and launches: setup %lld linearise %lld landmark-sums %lld inverse+Y+spill %lld "
            "schur+direct %lld gradients %lld flush %lld\n", dbg[48], dbg[49], dbg[50], dbg[51], dbg[52], dbg[53], dbg[54]);
    cudaMemset(d.dbg + 48, 0, 8 * sizeof(long long));
  }
  if (getenv("SVS_SOLVE_TIMING")) {
    const bool roles = atoi(getenv("SVS_SOLVE_TIMING")) > 1;
    if (roles) {
      long long tr[160];
      cudaMemcpy(tr, d.dbg, sizeof tr, cudaMemcpyDeviceToHost);
      const long long* t0 = tr + 12 + 52;
      fprintf(stderr, "trace (CTA 0, columns 10..25 of its branch; cycles relative to the chain's publish of column 10):\n");
      const char* nm[5] = {"chain published  ", "chain has U(j-1)  ", "urgent past Pub   ", "urgent arrives U  ", "unit 0 past Pub   "};
      for (int k = 0; k < 5; ++k) {
        fprintf(stderr, "  %s", nm[k]);
        for (int c = 0; c < 16; ++c) fprintf(stderr, " %6lld", t0[k * 16 + c] - t0[0]);
        fprintf(stderr, "\n");
      }
    }
    long long dbg[64];
    cudaMemcpy(dbg, d.dbg, sizeof dbg, cudaMemcpyDeviceToHost);
    fprintf(stderr, "k_solve cycles since setup (branch factored, cluster sync, separators factored, separators solved + sync, "
            "branch solved, end):\n");
    for (int g = 0; g < 2; ++g) {
      fprintf(stderr, "  CTA %d:", g);
      for (int i = 0; i < 6; ++i) fprintf(stderr, " %lld", dbg[g * 6 + i]);
      const long long* q = dbg + 12 + 16 * g;
      if (!roles) { fprintf(stderr, "\n"); continue; }
      fprintf(stderr, "\n     chain: hand-over %lld chol %lld wait-urgent+load %lld publish %lld | unit thread 8: loop-top+factor %lld wait-rows %lld "
              "units %lld | row thread 0: wait-factor %lld rows %lld wait-rows %lld N+rhs %lld | urgent: wait-factor %lld rows %lld units %lld\n",
              q[0], q[1], q[2], q[3], q[4], q[5], q[6], q[8], q[9], q[10], q[11], q[12], q[13], q[14]);
    }
  }
  return h->h_ctl->iter;
#undef CKN
#undef CKO
}

static int current_buffer(svs_ba* h, int* cur) {
  CK(cudaMemcpyAsync(h->h_ctl, h->d.ctl, sizeof(LmCtl), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  *cur = h->h_ctl->cur;
  return SVS_OK;
}

int svs_ba_get_poses(svs_ba* h, double* T_qt) {
  if (!h || !h->has_problem) return h ? fail(h, SVS_ERR_STATE, "no problem set") : SVS_ERR_INVALID;
  cudaSetDevice(h->device);
  int cur, rc;
  if ((rc = current_buffer(h, &cur))) return rc;
  if (h->d.P)
    CK(cudaMemcpyAsync(T_qt, h->d.pose[cur], 7 * (size_t)h->d.P * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return SVS_OK;
}

int svs_ba_get_points(svs_ba* h, double* psi) {
  if (!h || !h->has_problem) return h ? fail(h, SVS_ERR_STATE, "no problem set") : SVS_ERR_INVALID;
  cudaSetDevice(h->device);
  int cur, rc;
  if ((rc = current_buffer(h, &cur))) return rc;
  const int L = h->d.L;
  std::vector<double> tmp(3 * (size_t)L);
  if (L) CK(cudaMemcpyAsync(tmp.data(), h->d.psi[cur], 3 * (size_t)L * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  // a sharded window (svs_ba_set_problem_sharded) addresses the caller's full-size array: only this rank's entries are written
  const size_t mul = h->L_full ? (size_t)h->comm_size : 1, add = h->L_full ? (size_t)h->comm_rank : 0;
  for (int li = 0; li < L; ++li)
    for (int q = 0; q < 3; ++q) psi[3 * ((size_t)h->lm_to_user[li] * mul + add) + q] = tmp[3 * (size_t)li + q];
  return SVS_OK;
}

int svs_optimiseInnerAndOuterWindow(svs_ba* h, int P, double* T_qt, const unsigned char* fixed, int L, double* psi,
                                    int E, const int* e_point, const int* e_pose, const int* e_anchor,
                                    const double* e_obs, const double* e_info, int C, const int* c_i, const int* c_j,
                                    const double* c_T, const double* c_Lambda, const svs_cam* cam, int num_iters,
                                    int robust, double huber_delta, svs_ba_stats* stats) {
  int rc = svs_ba_set_problem(h, P, T_qt, fixed, L, psi, E, e_point, e_pose, e_anchor, e_obs, e_info, C, c_i, c_j,
                              c_T, c_Lambda, cam);
  if (rc) return -100 + rc;
  // the optimised state comes back in ONE copy behind the last trial (no separate read-out round trips)
  const size_t n = 7 * (size_t)P + 3 * (size_t)L;
  if (n > h->out_cap) {
    if (h->d_out) cudaFree(h->d_out);
    if (h->h_out) cudaFreeHost(h->h_out);
    h->d_out = h->h_out = nullptr; h->out_cap = 0;
    if (cudaMalloc((void**)&h->d_out, (n + n / 4) * sizeof(double)) != cudaSuccess ||
        cudaMallocHost((void**)&h->h_out, (n + n / 4) * sizeof(double)) != cudaSuccess)
      return -100 + fail(h, SVS_ERR_CUDA, "out of memory for the read-out buffer");
    h->out_cap = n + n / 4;
  }
  h->export_next = n > 0 && h->L_full == 0;
  // lambda0 = 50, 5 trials: slam_graph.cpp:338, :1073
  const int it = svs_ba_optimize(h, num_iters, robust, huber_delta, 50., 5, stats);
  const bool exported = h->export_next && it >= 0;
  h->export_next = false;
  if (it <= -100) return it;
  if (exported) {
    memcpy(T_qt, h->h_out, 7 * (size_t)P * sizeof(double));
    memcpy(psi, h->h_out + 7 * (size_t)P, 3 * (size_t)L * sizeof(double));
    return it;
  }
  if ((rc = svs_ba_get_poses(h, T_qt))) return -100 + rc;
  if ((rc = svs_ba_get_points(h, psi))) return -100 + rc;
  return it;
}

int svs_ba_chi2(svs_ba* h, int robust, double huber_delta, double* chi2) {
  if (!h || !h->has_problem) return h ? fail(h, SVS_ERR_STATE, "no problem set") : SVS_ERR_INVALID;
  cudaSetDevice(h->device);
  BaDev& d = h->d;
  launch_chi2(d, robust, huber_delta, h->stream);
  std::vector<double> a(d.L), c(d.C);
  if (d.L) CK(cudaMemcpyAsync(a.data(), d.chi_l, d.L * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  if (d.C) CK(cudaMemcpyAsync(c.data(), d.chi_c, d.C * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  CK(cudaGetLastError());
  double s = 0;
  for (double v : a) s += v;
  for (double v : c) s += v;
  *chi2 = s;
  return SVS_OK;
}

static int set_lambda(svs_ba* h, double lambda) {
  CK(cudaMemcpyAsync(h->h_ctl, h->d.ctl, sizeof(LmCtl), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  h->h_ctl->lambda = lambda;
  h->h_ctl->max_iters = 0;   // inspection hooks run the kernels unconditionally
  CK(cudaMemcpyAsync(h->d.ctl, h->h_ctl, sizeof(LmCtl), cudaMemcpyHostToDevice, h->stream));
  return SVS_OK;
}

int svs_ba_reduced_system(svs_ba* h, int robust, double huber_delta, double lambda, double* Sd, double* bs,
                          double* chi2) {
  if (!h || !h->has_problem) return h ? fail(h, SVS_ERR_STATE, "no problem set") : SVS_ERR_INVALID;
  cudaSetDevice(h->device);
  BaDev& d = h->d;
  int rc;
  if ((rc = set_lambda(h, lambda))) return rc;
  if ((rc = clear_system(h))) return rc;
  launch_build(d, h->Kmax_gen, robust, huber_delta, h->stream);
  const int P = d.P, n = 6 * P;
  std::vector<double> S(36 * (size_t)d.nblk), bp(n), bc(n), chl(d.L), chc(d.C);
  std::vector<int> colp(P + 1), rowi(d.nblk), perm(P);
  std::vector<unsigned char> fx(P);
  CK(cudaMemcpyAsync(S.data(), d.S, S.size() * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  if (P) {
    CK(cudaMemcpyAsync(bp.data(), d.bp, n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(bc.data(), d.bc, n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(perm.data(), d.perm, P * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(fx.data(), d.fixed, P, cudaMemcpyDeviceToHost, h->stream));
  }
  CK(cudaMemcpyAsync(colp.data(), d.col_ptr, (P + 1) * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaMemcpyAsync(rowi.data(), d.row_idx, d.nblk * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  if (d.L) CK(cudaMemcpyAsync(chl.data(), d.chi_l, d.L * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  if (d.C) CK(cudaMemcpyAsync(chc.data(), d.chi_c, d.C * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  CK(cudaGetLastError());
  if ((rc = clear_system(h))) return rc;
  std::fill(Sd, Sd + (size_t)n * n, 0.);
  for (int j = 0; j < P; ++j)
    for (int b = colp[j]; b < colp[j + 1]; ++b) {
      const int pi = perm[rowi[b]], pj = perm[j];
      for (int r = 0; r < 6; ++r)
        for (int c = 0; c < 6; ++c) {
          double v = S[36 * (size_t)b + r * 6 + c];
          if (pi == pj && r == c) v += lambda + (fx[pi] ? 1. : 0.);
          Sd[(size_t)(6 * pi + r) * n + 6 * pj + c] = v;
          Sd[(size_t)(6 * pj + c) * n + 6 * pi + r] = v;
        }
    }
  for (int i = 0; i < n; ++i) bs[i] = bp[i] - bc[i];
  if (chi2) {
    double s = 0;
    for (double v : chl) s += v;
    for (double v : chc) s += v;
    *chi2 = s;
  }
  return SVS_OK;
}

int svs_ba_solve_reduced(svs_ba* h, int robust, double huber_delta, double lambda, double* x) {
  if (!h || !h->has_problem) return h ? fail(h, SVS_ERR_STATE, "no problem set") : SVS_ERR_INVALID;
  cudaSetDevice(h->device);
  BaDev& d = h->d;
  int rc;
  if ((rc = set_lambda(h, lambda))) return rc;
  if ((rc = clear_system(h))) return rc;
  launch_build(d, h->Kmax_gen, robust, huber_delta, h->stream);
  launch_solve(d, h->max_col_branch, std::max(h->max_col_blocks, h->max_row_blocks - 2), h->nsep_blk, h->stream);
  if (d.P) CK(cudaMemcpyAsync(x, d.x, 6 * (size_t)d.P * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaMemcpyAsync(h->h_ctl, d.ctl, sizeof(LmCtl), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  CK(cudaGetLastError());
  const int failed = h->h_ctl->chol_fail;
  if ((rc = clear_system(h))) return rc;
  return failed ? 1 : 0;
}

// ---- one window sharded by landmarks across GPUs, driven inside the library (SURVEY.md 8e, BASELINE config C5)

int svs_comm_unique_id(char id[128]) {
  const NcclApi* nc = nccl_api();
  if (!nc || !id) return SVS_ERR_STATE;
  NcclUniqueId u;
  if (nc->GetUniqueId(&u) != 0) return SVS_ERR_CUDA;
  memcpy(id, u.internal, 128);
  return SVS_OK;
}

int svs_ba_comm_init(svs_ba* h, int nranks, int rank, const char id[128]) {
  if (!h || !id || nranks < 1 || rank < 0 || rank >= nranks) return SVS_ERR_INVALID;
  const NcclApi* nc = nccl_api();
  if (!nc) return fail(h, SVS_ERR_STATE, "NCCL library not loadable");
  cudaSetDevice(h->device);
  if (h->comm) { nc->CommDestroy(h->comm); h->comm = nullptr; }
  NcclUniqueId u;
  memcpy(u.internal, id, 128);
  const int e = nc->CommInitRank(&h->comm, nranks, u, rank);
  if (e != 0) { h->comm = nullptr; return fail(h, SVS_ERR_CUDA, std::string("ncclCommInitRank: ") + nc->GetErrorString(e)); }
  h->comm_rank = rank; h->comm_size = nranks;
  return SVS_OK;
}

// The whole window goes in on every rank; this rank keeps landmarks l with l % nranks == rank and their
// edges (poses replicated, pose-pose constraints on rank 0) and the block pattern of the WHOLE window, so
// that every rank's reduced system has the same layout and one all-reduce per trial sums them.
int svs_ba_set_problem_sharded(svs_ba* h, int P, const double* T_qt, const unsigned char* fixed, int L, const double* psi,
                               int E, const int* e_point, const int* e_pose, const int* e_anchor, const double* e_obs,
                               const double* e_info, int C, const int* c_i, const int* c_j, const double* c_T,
                               const double* c_Lambda, const svs_cam* cam) {
  svs::NvtxRange nvtx_("copyDataToG2o");
  if (!h) return SVS_ERR_INVALID;
  if (P < 0 || L < 0 || E < 0 || C < 0) return fail(h, SVS_ERR_INVALID, "negative size");
  if (E && (!e_point || !e_pose || !e_anchor || !e_obs || !e_info)) return fail(h, SVS_ERR_INVALID, "null array");
  const int W = h->comm_size, R = h->comm_rank;
  for (int e = 0; e < E; ++e)
    if (e_point[e] < 0 || e_point[e] >= L || e_pose[e] < 0 || e_pose[e] >= P || e_anchor[e] < 0 || e_anchor[e] >= P)
      return fail(h, SVS_ERR_INVALID, "observation edge index out of range");
  // block pattern of the whole window: pose pairs coupled by any landmark track (anchor included)
  {
    std::vector<int> ptr(L + 1, 0), ord(E);
    for (int e = 0; e < E; ++e) ptr[e_point[e] + 1]++;
    for (int l = 0; l < L; ++l) ptr[l + 1] += ptr[l];
    std::vector<int> fill(ptr.begin(), ptr.end() - 1);
    for (int e = 0; e < E; ++e) ord[fill[e_point[e]]++] = e;
    std::vector<unsigned char> A((size_t)P * P, 0);
    std::vector<int> ps;
    h->extra_pairs.clear();
    for (int l = 0; l < L; ++l) {
      if (ptr[l] == ptr[l + 1]) continue;
      ps.clear();
      const int anchor = e_anchor[ord[ptr[l]]];
      ps.push_back(anchor);
      int nself = 0, lo = P, hi = -1;
      for (int k = ptr[l]; k < ptr[l + 1]; ++k) {
        const int f = e_pose[ord[k]];
        ps.push_back(f);
        if (f == anchor) ++nself;
        else { lo = std::min(lo, f); hi = std::max(hi, f); }
      }
      // the frames the owning rank's set_problem pads this track with (zero-weight edges) are part of the pattern too
      if (!getenv("SVS_BUILD_NO_PAD") && nself <= 1 && track_padding(ptr[l + 1] - ptr[l] - nself, lo, hi, anchor) > 0)
        for (int f = lo; f <= hi; ++f)
          if (f != anchor) ps.push_back(f);
      for (size_t x = 0; x < ps.size(); ++x)
        for (size_t y = x + 1; y < ps.size(); ++y) {
          const int a = std::min(ps[x], ps[y]), b = std::max(ps[x], ps[y]);
          if (a != b && !A[(size_t)a * P + b]) { A[(size_t)a * P + b] = 1; h->extra_pairs.push_back(a); h->extra_pairs.push_back(b); }
        }
    }
    for (int c = 0; c < C; ++c) {
      const int a = std::min(c_i[c], c_j[c]), b = std::max(c_i[c], c_j[c]);
      if (a < 0 || b >= P) return fail(h, SVS_ERR_INVALID, "pose-pose edge index out of range");
      if (a != b && !A[(size_t)a * P + b]) { A[(size_t)a * P + b] = 1; h->extra_pairs.push_back(a); h->extra_pairs.push_back(b); }
    }
  }
  // this rank's share
  const int Ll = L > R ? (L - R + W - 1) / W : 0;
  std::vector<double> lpsi(3 * (size_t)Ll);
  for (int l = R, q = 0; l < L; l += W, ++q)
    for (int k = 0; k < 3; ++k) lpsi[3 * (size_t)q + k] = psi[3 * (size_t)l + k];
  std::vector<int> lp, lf, la;
  std::vector<double> lo, li;
  lp.reserve(E / W + 16); lf.reserve(E / W + 16); la.reserve(E / W + 16); lo.reserve(3 * (size_t)(E / W + 16)); li.reserve(3 * (size_t)(E / W + 16));
  for (int e = 0; e < E; ++e) {
    if (e_point[e] % W != R) continue;
    lp.push_back(e_point[e] / W); lf.push_back(e_pose[e]); la.push_back(e_anchor[e]);
    for (int k = 0; k < 3; ++k) { lo.push_back(e_obs[3 * (size_t)e + k]); li.push_back(e_info[3 * (size_t)e + k]); }
  }
  const int Cl = R == 0 ? C : 0;
  const int rc = set_problem_impl(h, P, T_qt, fixed, Ll, lpsi.data(), (int)lp.size(), lp.data(), lf.data(), la.data(), lo.data(),
                                  li.data(), Cl, c_i, c_j, c_T, c_Lambda, cam, nullptr);
  h->extra_pairs.clear();
  h->L_full = rc == SVS_OK ? L : 0;
  h->sharded = rc == SVS_OK;
  return rc;
}

// restoreDataFromG2o on every rank: all landmarks of the sharded window (each rank contributes its own,
// summed over the communicator)
int svs_ba_get_points_all(svs_ba* h, double* psi) {
  if (!h || !h->has_problem || !psi) return h ? fail(h, SVS_ERR_STATE, "no problem set") : SVS_ERR_INVALID;
  if (!h->L_full) return svs_ba_get_points(h, psi);
  const size_t n = 3 * (size_t)h->L_full;
  std::fill(psi, psi + n, 0.);
  int rc;
  if ((rc = svs_ba_get_points(h, psi))) return rc;
  if (!h->comm || h->comm_size == 1) return SVS_OK;
  const NcclApi* nc = nccl_api();
  if (!nc) return fail(h, SVS_ERR_STATE, "NCCL library not loadable");
  if (n > h->psi_all_cap) {
    if (h->d_psi_all) cudaFree(h->d_psi_all);
    h->d_psi_all = nullptr; h->psi_all_cap = 0;
    CK(cudaMalloc((void**)&h->d_psi_all, n * sizeof(double)));
    h->psi_all_cap = n;
  }
  CK(cudaMemcpyAsync(h->d_psi_all, psi, n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  if (nc->AllReduce(h->d_psi_all, h->d_psi_all, n, kNcclFloat64, kNcclSum, h->comm, h->stream) != 0)
    return fail(h, SVS_ERR_CUDA, "ncclAllReduce failed");
  CK(cudaMemcpyAsync(psi, h->d_psi_all, n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return SVS_OK;
}

// ---- stepwise Levenberg trial for a window whose landmarks are split across ranks
// (SURVEY.md 8e): build -> [caller all-reduces S, bp, bc] -> solve -> [caller all-reduces totals] -> decide

int svs_ba_set_structure(svs_ba* h, int npairs, const int* pose_i, const int* pose_j) {
  if (!h || npairs < 0 || (npairs && (!pose_i || !pose_j))) return SVS_ERR_INVALID;
  h->extra_pairs.clear();
  for (int q = 0; q < npairs; ++q) { h->extra_pairs.push_back(pose_i[q]); h->extra_pairs.push_back(pose_j[q]); }
  // A caller that prescribes the block pattern (several handles summing their reduced systems element by element)
  // has derived it from its own edge lists: this handle must not add pose pairs of its own, so its tracks are not padded
  h->extra_pairs_from_caller = npairs > 0;
  return SVS_OK;
}

int svs_ba_lm_begin(svs_ba* h, double lambda_init, int max_trials) {
  if (!h || !h->has_problem) return h ? fail(h, SVS_ERR_STATE, "no problem set") : SVS_ERR_INVALID;
  cudaSetDevice(h->device);
  CK(cudaMemcpyAsync(h->h_ctl, h->d.ctl, sizeof(LmCtl), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  const int cur = h->h_ctl->cur;
  LmCtl z{};
  z.cur = cur; z.lambda = lambda_init; z.ni = 2; z.max_trials = max_trials;
  *h->h_ctl = z;
  CK(cudaMemcpyAsync(h->d.ctl, h->h_ctl, sizeof(LmCtl), cudaMemcpyHostToDevice, h->stream));
  return clear_system(h);
}

int svs_ba_trial_build(svs_ba* h, int robust, double huber_delta) {
  if (!h || !h->has_problem) return h ? fail(h, SVS_ERR_STATE, "no problem set") : SVS_ERR_INVALID;
  cudaSetDevice(h->device);
  launch_build(h->d, h->Kmax_gen, robust, huber_delta, h->stream);
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(h->stream));   // the caller's collective runs on its own stream
  return SVS_OK;
}

int svs_ba_system_buffers(svs_ba* h, double** S, long long* nS, double** bp, double** bc, long long* nb,
                          double** totals) {
  if (!h || !h->has_problem) return h ? fail(h, SVS_ERR_STATE, "no problem set") : SVS_ERR_INVALID;
  if (S) *S = h->d.S;
  if (nS) *nS = 36ll * h->d.nblk;
  if (bp) *bp = h->d.bp;
  if (bc) *bc = h->d.bc;
  if (nb) *nb = 6ll * h->d.P;
  if (totals) *totals = h->d.totals;
  return SVS_OK;
}

int svs_ba_trial_solve(svs_ba* h, int robust, double huber_delta) {
  if (!h || !h->has_problem) return h ? fail(h, SVS_ERR_STATE, "no problem set") : SVS_ERR_INVALID;
  cudaSetDevice(h->device);
  launch_solve(h->d, h->max_col_branch, std::max(h->max_col_blocks, h->max_row_blocks - 2), h->nsep_blk, h->stream);
  launch_update(h->d, robust, huber_delta, 1, h->stream);
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(h->stream));
  return SVS_OK;
}

int svs_ba_trial_decide(svs_ba* h, int* again, int* stop, int* iter) {
  if (!h || !h->has_problem) return h ? fail(h, SVS_ERR_STATE, "no problem set") : SVS_ERR_INVALID;
  cudaSetDevice(h->device);
  launch_decide_deferred(h->d, h->stream);
  CK(cudaMemcpyAsync(h->h_ctl, h->d.ctl, sizeof(LmCtl), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  h->cur_known = h->h_ctl->cur;
  CK(cudaGetLastError());
  if (again) *again = h->h_ctl->again;
  if (stop) *stop = h->h_ctl->stop;
  if (iter) *iter = h->h_ctl->iter;
  return SVS_OK;
}

int svs_ba_lm_stats(svs_ba* h, svs_ba_stats* st) {
  if (!h || !h->has_problem || !st) return SVS_ERR_INVALID;
  memset(st, 0, sizeof *st);
  const LmCtl& c = *h->h_ctl;
  st->iterations = c.iter; st->trials_total = c.trials_total; st->chi2_init = c.chi_init; st->chi2_final = c.chi_cur;
  st->lambda_final = c.lambda;
  for (int i = 0; i < c.iter && i < SVS_BA_MAX_ITERS; ++i) {
    st->chi2_iter[i] = c.chi_iter[i]; st->lambda_iter[i] = c.lambda_iter[i]; st->trials_iter[i] = c.trials_iter[i];
  }
  st->num_frames = h->d.P; st->num_points = h->d.L; st->num_point_edges = h->d.E_user; st->num_frame_edges = h->d.C;
  st->nnzb_S = h->nnzb_S; st->nnzb_L = h->d.nblk; st->max_track = h->Kmax;
  return SVS_OK;
}

}  // extern "C"

// ---- hooks for the other modules of the library (internal.cuh)
namespace svs {
int ba_set_problem_device_obs(svs_ba* h, int P, const double* T_qt, const unsigned char* fixed, int L, const double* psi, int E,
                              const int* e_point, const int* e_pose, const int* e_anchor, const double* d_obs_info, int C,
                              const int* c_i, const int* c_j, const double* c_T, const double* c_Lambda, const svs_cam* cam) {
  if (h) { h->L_full = 0; h->sharded = false; }
  const int rc = set_problem_impl(h, P, T_qt, fixed, L, psi, E, e_point, e_pose, e_anchor, nullptr, nullptr, C, c_i, c_j, c_T,
                                  c_Lambda, cam, d_obs_info);
  if (rc == SVS_OK && cudaStreamSynchronize(h->stream) != cudaSuccess) return SVS_ERR_CUDA;   // d_obs_info may be reused now
  return rc;
}
int ba_device(const svs_ba* h) { return h->device; }
int ba_state_on_device(svs_ba* h, const double* const** pose, const double* const** psi, const int** lm_user, const int** cur,
                       cudaStream_t* stream, int* P, int* L) {
  if (!h || !h->has_problem) return SVS_ERR_STATE;
  *pose = h->d.pose; *psi = h->d.psi; *lm_user = h->d.lm_user; *cur = &h->d.ctl->cur; *stream = h->stream; *P = h->d.P; *L = h->d.L;
  return SVS_OK;
}
}  // namespace svs

