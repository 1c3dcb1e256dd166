// engine.cu -- the B200-native ADMM iteration engine behind include/cosmo_b200.h.
//
// Host-side driver of the hot loop of COSMO.optimize! (reference
// src/solver.jl:125-167, restated in SURVEY.md Appendix A) plus the C ABI.
// All arithmetic runs in the hand-written sm_100a kernels of spmv.cuh,
// vector_kernels.cuh and psd.cuh; the host only sequences launches, reads
// back a handful of scalars at the reference's own decision points
// (termination / infeasibility / rho-adaptation checks, CG convergence) and
// never touches vector data.  There is no CPU fallback: without a CUDA device
// every entry point fails with COSMO_B200_ERR_CUDA.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <functional>
#include <thread>
#include <chrono>
#include <string>
#include <vector>

#include "../../include/cosmo_b200.h"
#include "common.cuh"
#include "psd.cuh"
#include "cone3.cuh"
#include "aa.cuh"
#include "spmv.cuh"
#include "vector_kernels.cuh"
#include "ruiz.cuh"
#include "cg_persistent.cuh"
#include "direct.cuh"
#include "ldl_symbolic.h"

namespace cosmo {

static thread_local std::string g_create_error;

struct EngineError {
  int code;
  std::string msg;
};

#define CUDA_TRY(expr)                                                                              \
  do {                                                                                              \
    cudaError_t _e = (expr);                                                                        \
    if (_e != cudaSuccess) {                                                                        \
      char _b[512];                                                                                 \
      snprintf(_b, sizeof(_b), "CUDA error %s at %s:%d: %s", cudaGetErrorName(_e), __FILE__,        \
               __LINE__, cudaGetErrorString(_e));                                                   \
      throw EngineError{COSMO_B200_ERR_CUDA, _b};                                                   \
    }                                                                                               \
  } while (0)

static inline double now_s() {
  return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// ---- NCCL through dlopen (the single-GPU path has no NCCL dependency) --------
struct NcclUniqueId { char internal[128]; };
typedef void* NcclComm;
struct NcclApi {
  void* lib = nullptr;
  int (*GetUniqueId)(NcclUniqueId*) = nullptr;
  int (*CommInitRank)(NcclComm*, int, NcclUniqueId, int) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, NcclComm, cudaStream_t) = nullptr;
  int (*CommDestroy)(NcclComm) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  bool load(std::string& err) {
    if (lib) return true;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* nm : names) {
      lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
      if (lib) break;
    }
    if (!lib) { err = std::string("cannot dlopen libnccl: ") + dlerror(); return false; }
    GetUniqueId = (int (*)(NcclUniqueId*))dlsym(lib, "ncclGetUniqueId");
    CommInitRank = (int (*)(NcclComm*, int, NcclUniqueId, int))dlsym(lib, "ncclCommInitRank");
    AllReduce = (int (*)(const void*, void*, size_t, int, int, NcclComm, cudaStream_t))dlsym(lib, "ncclAllReduce");
    CommDestroy = (int (*)(NcclComm))dlsym(lib, "ncclCommDestroy");
    GetErrorString = (const char* (*)(int))dlsym(lib, "ncclGetErrorString");
    if (!GetUniqueId || !CommInitRank || !AllReduce || !CommDestroy) { err = "libnccl lacks required symbols"; return false; }
    return true;
  }
};
static NcclApi g_nccl;
constexpr int kNcclFloat32 = 7, kNcclFloat64 = 8, kNcclSum = 0, kNcclMax = 2;

// ---- phase timers (ResultTimes.proj_time / kkt_time, types.jl:26-41) ------------
// CUDA events on the engine stream around a phase; elapsed times are harvested in batches so that the loop never
// waits for a timer (one event synchronisation per kCap phases).
struct PhaseTimer {
  static constexpr int kCap = 64;
  cudaEvent_t a[kCap], b[kCap];
  int n = 0;
  bool created = false, on = false;
  double total_ms = 0.0;
  ~PhaseTimer() {
    if (created) for (int i = 0; i < kCap; ++i) { cudaEventDestroy(a[i]); cudaEventDestroy(b[i]); }
  }
  void enable(bool e) {
    on = e;
    if (on && !created) {
      for (int i = 0; i < kCap; ++i) { cudaEventCreate(&a[i]); cudaEventCreate(&b[i]); }
      created = true;
    }
    n = 0; total_ms = 0.0;
  }
  void begin(cudaStream_t st) { if (on) cudaEventRecord(a[n], st); }
  void end(cudaStream_t st) {
    if (!on) return;
    cudaEventRecord(b[n], st);
    if (++n == kCap) harvest();
  }
  void harvest() {
    if (!on || n == 0) return;
    cudaEventSynchronize(b[n - 1]);
    for (int i = 0; i < n; ++i) { float ms = 0.f; cudaEventElapsedTime(&ms, a[i], b[i]); total_ms += ms; }
    n = 0;
  }
};

// ---- device buffer -----------------------------------------------------------
template <typename U>
struct DevBuf {
  U* p = nullptr;
  size_t n = 0;
  DevBuf() {}
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { if (p) cudaFree(p); }
  void alloc(size_t count, bool zero = true) {
    if (p) { cudaFree(p); p = nullptr; }
    n = count;
    size_t bytes = (count + 8) * sizeof(U);   // +8: bulk (TMA) copies round the tail up to 16 bytes
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) throw EngineError{COSMO_B200_ERR_ALLOC, std::string("cudaMalloc failed: ") + cudaGetErrorString(e)};
    if (zero) {
      // cudaMemset runs on the legacy default stream, which does NOT order against the engine's
      // non-blocking stream: wait for it here or a later kernel may race with the pending fill.
      CUDA_TRY(cudaMemset(p, 0, bytes));
      CUDA_TRY(cudaDeviceSynchronize());
    }
  }
  void upload(const U* host, size_t count, cudaStream_t st) {
    if (count) CUDA_TRY(cudaMemcpyAsync(p, host, count * sizeof(U), cudaMemcpyHostToDevice, st));
  }
  void upload(const std::vector<U>& h, cudaStream_t st) {
    if (n < h.size()) alloc(h.size(), false);
    upload(h.data(), h.size(), st);
  }
};

template <typename T>
struct DevCsr {
  int nrows = 0, ncols = 0;
  long long nnz = 0;
  DevBuf<int> rowptr, col;
  DevBuf<T> val;
  int lanes = 32;
  // column-windowed copy (spmv_win_kernel); absent when the rows are too short to pay off
  bool windowed = false;
  int nwin = 0, W = 0, nctas = 0;
  DevBuf<int> w_rowptr, w_cta_rows;
  DevBuf<unsigned short> w_col;
  DevBuf<T> w_val;
  long long w_elems = 0;
  WcsrView<T> wview() const { return WcsrView<T>{w_rowptr.p, w_col.p, w_val.p, w_cta_rows.p, nwin, W, nrows, ncols}; }
  CsrView<T> view() const { return CsrView<T>{rowptr.p, col.p, val.p}; }
  double spmv_bytes() const {  // SURVEY.md 8d: 12 nnz + 4 (rows+1) + 8 cols + 8 rows   (fp64)
    return (double)nnz * (sizeof(T) + 4) + 4.0 * (nrows + 1) + (double)sizeof(T) * ncols + (double)sizeof(T) * nrows;
  }
};

static int pick_lanes(double mean_row) {
  if (mean_row > 24.0) return 32;
  if (mean_row > 3.0) return 8;
  return 2;
}

struct HostCsr {
  int nrows = 0, ncols = 0;
  std::vector<int> rowptr, col;
  std::vector<double> val;  // staged in double, narrowed on upload when T=float
};

class EngineBase {
 public:
  virtual ~EngineBase() {}
  std::string err;
  virtual void update_settings(const cosmo_b200_settings& st) = 0;
  virtual void warm_start(const void* x, const void* s, const void* mu) = 0;
  virtual void update_qb(const void* q, const void* b) = 0;
  virtual void update_rho(const void* rho_vec, double rho) = 0;
  virtual void reset() = 0;
  virtual void solve(cosmo_b200_result* out) = 0;
  virtual void project(const void* ws, void* s_out) = 0;
  virtual void kkt_solve(const void* rhs, void* sol, int64_t* inner) = 0;
  virtual void residuals(const void* x, const void* s, const void* mu, int ignore_scaling, double* out) = 0;
  virtual void spmv(int which, const void* x, void* y) = 0;
  virtual void spmv_bench(int which, int reps, double* ms, double* bytes) = 0;
  virtual void get_rho_vec(void* out) = 0;
  virtual void get_w(void* out) = 0;
  virtual void psd_stats(int64_t* out8) = 0;
  virtual void kkt_factor_stats(int64_t* factorizations, double* seconds2) = 0;
  virtual void get_scaling(void* D, void* E, double* c) = 0;
  virtual void comm_init(int nranks, int rank, const void* id128) = 0;
  virtual void p2p_export(void* blob128) = 0;
  virtual void p2p_attach(const void* blobs, int nranks) = 0;
};

template <typename T>
class Engine : public EngineBase {
 public:
  Engine(const cosmo_b200_problem& p, const cosmo_b200_settings& st);
  ~Engine() override;
  void update_settings(const cosmo_b200_settings& st) override {
    if (st.kkt_solver == COSMO_B200_KKT_DIRECT && !d_L_.p)
      throw EngineError{COSMO_B200_ERR_UNSUPPORTED, "kkt_solver DIRECT is chosen when the engine is created (its factor is set up there)"};
    if (st.sigma != st_.sigma) {
      destroy_cg_graphs();   // sigma is baked into the captured kernel arguments
      d_stale_ = true;       // and into the diagonal of the reduced matrix
    }
    st_ = st;
  }
  void warm_start(const void* x, const void* s, const void* mu) override;
  void update_qb(const void* q, const void* b) override;
  void update_rho(const void* rho_vec, double rho) override;
  void reset() override;
  void solve(cosmo_b200_result* out) override;
  void project(const void* ws, void* s_out) override;
  void kkt_solve(const void* rhs, void* sol, int64_t* inner) override;
  void residuals(const void* x, const void* s, const void* mu, int ignore_scaling, double* out) override;
  void spmv(int which, const void* x, void* y) override;
  void spmv_bench(int which, int reps, double* ms, double* bytes) override;
  void get_rho_vec(void* out) override;
  void get_w(void* out) override;
  void psd_stats(int64_t* out8) override;
  void kkt_factor_stats(int64_t* factorizations, double* seconds2) override {
    *factorizations = d_factorizations_;
    seconds2[0] = d_init_s_;
    seconds2[1] = d_update_s_;
  }
  void get_scaling(void* D, void* E, double* c) override;
  void equilibrate();
  void comm_init(int nranks, int rank, const void* id128) override;
  void p2p_export(void* blob128) override;
  void p2p_attach(const void* blobs, int nranks) override;

 private:
  // ---- problem ----
  int n_ = 0, m_ = 0, device_ = 0;
  double create_time_ = 0.0;      // engine construction (the device part of setup!)
  bool device_scaled_ = false;    // D, E, c were computed here (equilibrate), not handed over by the host
  int auto_rho_interval_ = 0;     // adaptive_rho_interval chosen by the automatic rule (kept across solves like settings)
  cosmo_b200_settings st_;
  bool scaled_ = false;
  double c_ = 1.0;
  DevCsr<T> A_, At_, P_;
  DevBuf<T> q_, b_, D_, Dinv_, E_, Einv_;
  std::vector<double> hb_;                       // host copy of b (row classification)
  std::vector<double> hl_, hu_;                  // host box bounds (m-length, +-inf elsewhere)
  std::vector<cosmo_b200_set> sets_;             // type + dim only
  std::vector<int> set_off_;
  // cones
  DevBuf<unsigned char> row_class_, rho_class_;
  DevBuf<int> row_cone_;
  DevBuf<T> box_l_, box_u_;
  int n_soc_ = 0, n_soc_chunks_ = 0;
  DevBuf<int> soc_off_, soc_dim_, soc_chunk_start_, soc_chunk_len_, soc_cone_chunk_ptr_;
  DevBuf<T> soc_norm_, soc_chunk_sum_, soc_norm2_;
  PsdBatch<T> psd_;
  PhaseTimer t_proj_, t_kkt_;
  DevBuf<T> proj_w_, proj_s_;     // scratch of the plugin-level project() entry point
  int n_c3_ = 0;             // exponential / power cones and their duals (cone3.cuh)
  DevBuf<int> c3_off_, c3_maxit_;
  DevBuf<unsigned char> c3_kind_;
  DevBuf<T> c3_alpha_, c3_tol_;
  Cone3Table<T> c3_table() const {
    return Cone3Table<T>{n_c3_, c3_off_.p, c3_kind_.p, c3_alpha_.p, c3_maxit_.p, c3_tol_.p};
  }
  // ---- accelerator (aa.cuh) ----
  DevBuf<T> aaG_, aaQ_, aaR_, aa_eta_, aa_glast_, aa_f_, aa_flast_, aa_sc_;
  T* h_aa_ = nullptr;          // pinned mirror of aa_sc_
  int aa_mem_ = 0;             // allocated history length (min(mem, dim)), 0 = not allocated
  int aa_iter_ = 0;            // columns filled since the last restart
  bool aa_init_ = true, aa_success_ = false, aa_active_ = false;
  long long aa_accelerated_ = 0, aa_declined_ = 0;
  void aa_prepare();
  void aa_restart() { aa_iter_ = 0; aa_init_ = true; }
  void aa_update(const T* g, const T* x);
  bool aa_accelerate(T* g);
  // ---- state ----
  DevBuf<T> W_[2];           // operator variable, ping-pong (w / w_prev)
  int cur_ = 0, prev_ = 1;
  DevBuf<T> xs_, s_, mu_;    // warm-start / exit copies of x; s; mu
  DevBuf<T> rho_vec_;
  double rho_ = 0.1;
  std::vector<double> rho_updates_;
  bool is_optimized_ = false;
  // KKT (reduced CG)
  DevBuf<T> ls_, t0_, tm_, xsol_, rhsb_, cb_, r_, u_, nu_;
  DevBuf<T> mr_[6], mr_x_, mr_c_, mr_b_;   // MINRES Lanczos / direction vectors, solution, operator output, rhs
  int cur_maxit_ = -1;
  // CUDA graphs of 1, 2, 4, 8 CG iterations (the inner loop is launch-bound for small problems)
  cudaGraphExec_t cg_graph_[4] = {nullptr, nullptr, nullptr, nullptr};
  bool use_graphs_ = true;
  bool graph_multi_ = true;
  // persistent cooperative CG kernel for launch-latency-bound (small / medium, non-windowed) problems
  bool use_persistent_ = true;
  int persist_grid_ = 0, persist_lanes_ = 0, persist_ctas_per_sm_ = 2;
  DevBuf<T> persist_part_;
  long long persist_solves_ = 0;
  bool persistent_cg_ok();
  void launch_persistent_cg(double tol_num);
  void cg_iteration_launches(const int* done);
  void build_cg_graphs(const int* done);
  void destroy_cg_graphs();
  // direct solve of the reduced system (direct.cuh): dense fp64 tile Cholesky factor of M = P + sigma I + A'RA
  int d_NT_ = 0, d_nd_ = 0, d_G_ = 0;
  int d_ctas_cap_ = 0;                            // COSMO_B200_DIRECT_CTAS: upper bound of the sweep grid (0: none)
  long long d_ldg_ = 0;
  size_t d_smem_ = 0;
  std::vector<int> d_rows_host_;                  // the dense rows of A (assembled through the panel product)
  DevBuf<double> d_L_, d_Gt_, d_y_, d_x_, d_dinv_;
  DevBuf<int> d_rows_, d_fail_;
  DevBuf<unsigned char> d_dense_;
  DevBuf<unsigned> d_ready_;
  unsigned d_epoch_ = 0;
  bool d_stale_ = true;                           // rho or sigma changed since the last factorisation
  long long d_factorizations_ = 0;
  double d_init_s_ = 0.0, d_update_s_ = 0.0;      // init_factor_time / factor_update_time (types.jl:31-32)
  void direct_plan(const HostCsr& a, const HostCsr& p);
  void direct_alloc();
  void direct_factor();
  void direct_solve();
  void ensure_factor() { if (st_.kkt_solver == COSMO_B200_KKT_DIRECT && d_stale_) direct_factor(); }
  long long kkt_counter_ = 1;   // S.iteration_counter
  int last_cg_iters_ = 1;
  long long total_inner_ = 0, total_mults_ = 0;
  // scratch
  DevBuf<T> vec_m_, vec_n_, vec_n2_, dy_, dx_, ypart_;
  DevBuf<unsigned> chunk_ticket_;
  int num_sms_ = 148;
  bool use_windows_ = true;
  int win_group_ = 16;
  DevBuf<T> sc_;       // device scalars
  DevBuf<int> isc_;
  DevBuf<T> partials_;
  DevBuf<unsigned> ticket_;
  T* h_sc_ = nullptr;  // pinned mirrors
  int* h_isc_ = nullptr;
  cudaStream_t stream_ = nullptr;
  cudaEvent_t ev0_ = nullptr, ev1_ = nullptr;
  long long launches_ = 0;
  // multi-GPU
  int nranks_ = 1, rank_ = 0;
  NcclComm comm_ = nullptr;
  // peer-memory exchange of the reduced-KKT operator partials (replaces the per-application allreduce)
  bool p2p_ = false;
  P2pView<T> xv_;
  DevBuf<T> xchg_data_;
  DevBuf<unsigned> xchg_flags_, xchg_seq_, xchg_arrive_;
  std::vector<void*> ipc_opened_;

  // ---- helpers ----
  RedBuf<T> red(int out_slot) { return RedBuf<T>{partials_.p, sc_.p + out_slot, ticket_.p}; }
  RedBuf<T> red_ptr(T* out) { return RedBuf<T>{partials_.p, out, ticket_.p}; }
  // K5 + K7 pass: 128-bit kernel for fp64 when every (n+m)-vector's m-part is 16-byte aligned (n even; ws_rhs too)
  void launch_proj_rhs(const ProjRhsArgs<T>& a) {
    if constexpr (std::is_same<T, double>::value) {
      if ((a.n & 1) == 0 && ((reinterpret_cast<uintptr_t>(a.ws_rhs) & 15) == 0) && ((reinterpret_cast<uintptr_t>(a.w) & 15) == 0)) {
        const long long pairs = (a.n >> 1) + ((a.m + 1) >> 1);
        proj_rhs_vec2_kernel<<<vgrid(pairs), kBlock, 0, stream_>>>(a);
        check_launch("proj_rhs_vec2");
        return;
      }
    }
    proj_rhs_kernel<T><<<vgrid((long long)a.n + a.m), kBlock, 0, stream_>>>(a);
    check_launch("proj_rhs");
  }
  static int vgrid(long long n) { return (int)std::min<long long>(std::max<long long>((n + kBlock - 1) / kBlock, 1), kMaxGrid); }
  static int sgrid(long long rows, int lanes) {
    long long per = kBlock / lanes;
    return (int)std::min<long long>(std::max<long long>((rows + per - 1) / per, 1), kMaxGrid);
  }
  void check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) throw EngineError{COSMO_B200_ERR_CUDA, std::string("launch of ") + what + " failed: " + cudaGetErrorString(e)};
    ++launches_;
  }
  void sync() { CUDA_TRY(cudaStreamSynchronize(stream_)); }
  void upload_vec(DevBuf<T>& dst, const void* host, size_t count);
  void download_vec(void* host, const T* src, size_t count);
  void build_csr(DevCsr<T>& dst, const HostCsr& h);
  void build_windows(DevCsr<T>& dst, const HostCsr& h);
  void classify_and_set_rho(bool reset_rho, bool rebuild_vec = true);
  void allreduce_sum(T* buf, size_t count);
  void allreduce_max(T* buf, size_t count);

  template <typename Epi>
  void launch_spmv(const DevCsr<T>& M1, const T* x1, const DevCsr<T>* M2, const T* x2, int nrows, const Epi& epi,
                   RedBuf<T> rb, const char* name);
  void project_device(const T* w, bool with_rhs, const T* ws_rhs);
  void soc_norms(const T* ws, T* norm_out);
  void kkt_core(bool fused_tail, const T* w_src, T* w_dst);
  void kkt_op_stage2(const int* done, const T* u, const T* t_in, T* c_out, bool exchange = false);
  void kkt_cg(const int* done);
  void kkt_minres(bool full);
  void set_maxit(int v);
  void compute_residuals(const T* x, const T* s, const T* mu, bool ignore_scaling, double out[5]);
  bool adapt_rho(const T* x);
  bool primal_infeasible();
  bool dual_infeasible();
  void recover_mu(const T* w_prev) {
    recover_mu_kernel<T><<<vgrid(m_), kBlock, 0, stream_>>>(m_, rho_vec_.p, w_prev + n_, s_.p, mu_.p);
    check_launch("recover_mu");
  }
  void read_scalars(int first, int count) {
    CUDA_TRY(cudaMemcpyAsync(h_sc_ + first, sc_.p + first, count * sizeof(T), cudaMemcpyDeviceToHost, stream_));
    sync();
  }
};

// ---------------------------------------------------------------------------
template <typename T>
void Engine<T>::upload_vec(DevBuf<T>& dst, const void* host, size_t count) {
  if (count == 0) return;
  CUDA_TRY(cudaMemcpyAsync(dst.p, host, count * sizeof(T), cudaMemcpyHostToDevice, stream_));
}
template <typename T>
void Engine<T>::download_vec(void* host, const T* src, size_t count) {
  if (count == 0) return;
  CUDA_TRY(cudaMemcpyAsync(host, src, count * sizeof(T), cudaMemcpyDeviceToHost, stream_));
}

template <typename T>
void Engine<T>::build_csr(DevCsr<T>& dst, const HostCsr& h) {
  dst.nrows = h.nrows;
  dst.ncols = h.ncols;
  dst.nnz = (long long)h.col.size();
  dst.lanes = pick_lanes(h.nrows ? (double)dst.nnz / h.nrows : 0.0);
  dst.rowptr.alloc(h.nrows + 1, false);
  dst.col.alloc(dst.nnz + 4, true);   // +4: the vector path never reads past nnz, padding keeps ASAN-style tools quiet
  dst.val.alloc(dst.nnz + 4, true);
  CUDA_TRY(cudaMemcpyAsync(dst.rowptr.p, h.rowptr.data(), (h.nrows + 1) * sizeof(int), cudaMemcpyHostToDevice, stream_));
  if (dst.nnz) {
    CUDA_TRY(cudaMemcpyAsync(dst.col.p, h.col.data(), dst.nnz * sizeof(int), cudaMemcpyHostToDevice, stream_));
    if (sizeof(T) == sizeof(double)) {
      CUDA_TRY(cudaMemcpyAsync(dst.val.p, h.val.data(), dst.nnz * sizeof(double), cudaMemcpyHostToDevice, stream_));
      sync();
    } else {
      std::vector<float> tmp(h.val.begin(), h.val.end());
      CUDA_TRY(cudaMemcpyAsync(dst.val.p, tmp.data(), dst.nnz * sizeof(float), cudaMemcpyHostToDevice, stream_));
      sync();
    }
  }
  sync();
}

// Column-windowed storage for spmv_win_kernel (see spmv.cuh).
//
// Inside one 256-entry step of a row segment, lane l / slot i reads entry l*8+i, and the
// shared-memory gather of slot i is issued per half-warp: the 16 lanes of a half-warp hit
// distinct 8-byte banks iff their window-local columns differ mod 16.  The order of the
// nonzeros inside a row is ours to choose (a dot product does not care), so the builder
// deals the entries of every residue class (col mod 16) over the (step, half-warp, slot)
// groups such that a group holds at most one entry per class whenever that is possible:
// the gathers become (nearly) bank-conflict free.
namespace {
struct WinGroupScratch {
  std::vector<int> cap, load, order;
  std::vector<unsigned short> used;
  std::vector<std::vector<int>> members;
  std::vector<int> bucket[16];
};
}  // namespace

template <typename T>
static void win_fill_segment(const int* cols, const double* vals, const int* idx, int k, int wbase, long long start,
                             unsigned short* wc, T* wv, WinGroupScratch& S, int GL) {
  // GL = lanes that share one shared-memory wavefront (16: half-warp, 8: quarter-warp)
  const int kpad = (k + 7) & ~7;
  if (kpad == 0) return;
  const int lanes_total = kpad / 8;
  const int steps = (lanes_total + 31) / 32;
  const int SUB = 32 / GL;              // lane groups per step
  const int GPS = SUB * 8;              // (lane group, slot) groups per step
  const int G = steps * GPS;
  S.cap.assign(G, 0); S.load.assign(G, 0); S.used.assign(G, 0);
  if ((int)S.members.size() < G) S.members.resize(G);
  for (int g = 0; g < G; ++g) S.members[g].clear();
  for (int st = 0; st < steps; ++st) {
    const int ls = std::min(32, lanes_total - 32 * st);
    for (int h = 0; h < SUB; ++h) {
      const int cap = std::max(0, std::min(GL, ls - GL * h));
      for (int i = 0; i < 8; ++i) S.cap[st * GPS + h * 8 + i] = cap;
    }
  }
  for (int r = 0; r < 16; ++r) S.bucket[r].clear();
  for (int e = 0; e < k; ++e) S.bucket[(cols[idx[e]] - wbase) & 15].push_back(idx[e]);
  int cls[16];
  for (int r = 0; r < 16; ++r) cls[r] = r;
  std::sort(cls, cls + 16, [&](int a, int b) { return S.bucket[a].size() > S.bucket[b].size(); });
  int cursor = 0;   // rotating start keeps the scan short and the loads balanced
  for (int ci = 0; ci < 16; ++ci) {
    const int r = cls[ci];
    for (int e : S.bucket[r]) {
      int best = -1, best_free = 0, fallback = -1, fb_free = 0;
      // bounded scan from the rotating cursor (long rows have hundreds of groups: an unbounded scan made the build
      // quadratic in the row length -- 15 s for the 10 000-entry rows of config C3); a second, unbounded pass only if
      // the window found no free slot at all
      const int scan = std::min(G, 96);
      for (int pass = 0; pass < 2 && best < 0 && fallback < 0; ++pass) {
        const int lim = pass == 0 ? scan : G;
        for (int t = 0; t < lim; ++t) {
          const int g = (cursor + t) % G;
          const int free_slots = S.cap[g] - S.load[g];
          if (free_slots <= 0) continue;
          if (!((S.used[g] >> r) & 1)) { if (free_slots > best_free) { best = g; best_free = free_slots; if (free_slots == GL) break; } }
          else if (free_slots > fb_free) { fallback = g; fb_free = free_slots; }
        }
      }
      const int g = best >= 0 ? best : fallback;
      S.members[g].push_back(e);
      S.used[g] |= (unsigned short)(1u << r);
      S.load[g]++;
      cursor = (g + 1) % G;
    }
  }
  for (int g = 0; g < G; ++g) {
    const int st = g / GPS, h = (g % GPS) / 8, i = g % 8;
    const int nl = S.cap[g];
    for (int t = 0; t < nl; ++t) {
      // column index: lane-contiguous (one 16-byte load per lane); value: instruction-coalesced
      // (load k of lane l at k * EPL * L + l * EPL, see load8_coalesced)
      const int lane = GL * h + t;
      const int ls = std::min(32, lanes_total - 32 * st);
      constexpr int EPL = 16 / (int)sizeof(T);
      const long long pos_c = start + (long long)st * 256 + (long long)lane * 8 + i;
      const long long pos_v = start + (long long)st * 256 + (long long)(i / EPL) * (EPL * ls) + (long long)lane * EPL + (i % EPL);
      if (t < S.load[g]) {
        const int e = S.members[g][t];
        wc[pos_c] = (unsigned short)(cols[e] - wbase);
        wv[pos_v] = (T)vals[e];
      } else {   // padding: zero value on a bank this group does not use yet
        int r0 = 0;
        while (r0 < 15 && ((S.used[g] >> r0) & 1)) ++r0;
        S.used[g] |= (unsigned short)(1u << r0);
        wc[pos_c] = (unsigned short)r0;
        wv[pos_v] = T(0);
      }
    }
  }
}

template <typename T>
void Engine<T>::build_windows(DevCsr<T>& dst, const HostCsr& h) {
  dst.windowed = false;
  if (!use_windows_ || h.nrows == 0 || h.ncols == 0) return;
  const long long nnz = (long long)h.col.size();
  const int Wmax = (int)(204800 / sizeof(T));
  const int nwin = (h.ncols + Wmax - 1) / Wmax;
  if (nwin > 16) return;
  const double per_seg = (double)nnz / ((double)h.nrows * nwin);
  if (per_seg < 24.0) return;                     // short rows: padding + per-row overhead would dominate
  int W = (h.ncols + nwin - 1) / nwin;
  W = (W + 31) & ~31;
  if (W > 65536) return;                          // 16-bit window-local indices
  const int nr = h.nrows;
  std::vector<int> rp((size_t)nwin * (nr + 1), 0);
  std::vector<long long> row_cost(nr, 0);
  const int nthreads = (int)std::max(1u, std::min(32u, std::thread::hardware_concurrency()));
  auto parallel_rows = [&](const std::function<void(int, int)>& fn) {
    std::vector<std::thread> th;
    const int chunk = (nr + nthreads - 1) / nthreads;
    for (int t = 0; t < nthreads; ++t) {
      const int a = t * chunk, b = std::min(nr, a + chunk);
      if (a < b) th.emplace_back(fn, a, b);
    }
    for (auto& x : th) x.join();
  };
  // pass 1: padded segment lengths
  parallel_rows([&](int a, int b) {
    std::vector<int> cnt(nwin);
    for (int r = a; r < b; ++r) {
      std::fill(cnt.begin(), cnt.end(), 0);
      for (int k = h.rowptr[r]; k < h.rowptr[r + 1]; ++k) cnt[h.col[k] / W]++;
      for (int w = 0; w < nwin; ++w) {
        const int padded = (cnt[w] + 7) & ~7;
        rp[(size_t)w * (nr + 1) + r + 1] = padded;
        row_cost[r] += padded + 48;   // per-row latency overhead measured at ~40 streamed entries (C3: 40k one-entry rows)
      }
    }
  });
  // window-major layout: all rows of window 0, then window 1, ...
  long long run = 0;
  for (int w = 0; w < nwin; ++w) {
    int* p = rp.data() + (size_t)w * (nr + 1);
    long long prev = run;
    for (int r = 0; r < nr; ++r) { const int len = p[r + 1]; p[r] = (int)prev; prev += len; if (prev >= (1LL << 31) - 16) return; }
    p[nr] = (int)prev;
    run = prev;
  }
  const long long total = run;
  std::vector<unsigned short> wc((size_t)total + 8, 0);
  std::vector<T> wv((size_t)total + 8, T(0));
  // pass 2: bank-aware placement of every row segment
  parallel_rows([&](int a, int b) {
    WinGroupScratch S;
    std::vector<std::vector<int>> seg(nwin);
    for (int r = a; r < b; ++r) {
      for (int w = 0; w < nwin; ++w) seg[w].clear();
      for (int k = h.rowptr[r]; k < h.rowptr[r + 1]; ++k) seg[h.col[k] / W].push_back(k);
      for (int w = 0; w < nwin; ++w)
        win_fill_segment<T>(h.col.data(), h.val.data(), seg[w].data(), (int)seg[w].size(), w * W,
                            rp[(size_t)w * (nr + 1) + r], wc.data(), wv.data(), S, win_group_);
    }
  });
  // contiguous row chunks per CTA, balanced by padded nnz (+ per-row overhead)
  // one CTA per (row chunk, window): chunks are contiguous row ranges balanced by padded nnz
  const int nchunks = std::max(1, num_sms_ / nwin);
  const int nctas = nchunks * nwin;
  std::vector<int> cta_rows(nchunks + 1, nr);
  long long all_cost = 0;
  for (int r = 0; r < nr; ++r) all_cost += row_cost[r];
  cta_rows[0] = 0;
  long long acc = 0;
  int g = 1;
  for (int r = 0; r < nr && g < nchunks; ++r) {
    acc += row_cost[r];
    while (g < nchunks && acc * nchunks >= all_cost * g) { cta_rows[g] = r + 1; ++g; }
  }
  for (; g < nchunks; ++g) cta_rows[g] = nr;
  cta_rows[nchunks] = nr;
  dst.nwin = nwin; dst.W = W; dst.nctas = nctas; dst.w_elems = total;
  dst.w_rowptr.upload(rp, stream_);
  dst.w_cta_rows.upload(cta_rows, stream_);
  dst.w_col.upload(wc, stream_);
  dst.w_val.upload(wv, stream_);
  sync();
  dst.windowed = true;
}

// Julia CSC -> (a) CSR of the transpose (zero conversion: same arrays, rebased)
//              (b) CSR of the matrix itself (stable counting-sort transposition)
template <typename T>
static void csc_to_host_csrs(const cosmo_b200_csc& M, int base, HostCsr& csr, HostCsr& csr_t) {
  const long long nr = M.nrows, nc = M.ncols;
  if (nr < 0 || nc < 0 || nr >= (1LL << 31) - 8 || nc >= (1LL << 31) - 8)
    throw EngineError{COSMO_B200_ERR_INVALID, "matrix dimensions out of int32 range"};
  const long long nnz = nc ? (M.colptr[nc] - base) : 0;
  if (nnz < 0 || nnz >= (1LL << 31) - 8) throw EngineError{COSMO_B200_ERR_INVALID, "nnz out of int32 range"};
  const T* vals = static_cast<const T*>(M.nzval);
  csr_t.nrows = (int)nc; csr_t.ncols = (int)nr;
  csr_t.rowptr.resize(nc + 1);
  csr_t.col.resize(nnz);
  csr_t.val.resize(nnz);
  for (long long j = 0; j <= nc; ++j) {
    long long v = nc ? M.colptr[j] - base : 0;
    if (v < 0 || v > nnz || (j > 0 && v < csr_t.rowptr[j - 1])) throw EngineError{COSMO_B200_ERR_INVALID, "colptr not monotone"};
    csr_t.rowptr[j] = (int)v;
  }
  csr.nrows = (int)nr; csr.ncols = (int)nc;
  csr.rowptr.assign(nr + 1, 0);
  csr.col.resize(nnz);
  csr.val.resize(nnz);
  // Stable counting-sort transposition, parallel over column blocks: thread t counts the rows of its columns, a prefix
  // over (row, thread) gives every thread its own slots in every row, so the scatter needs no synchronisation and the
  // entries of a row stay ordered by column whatever the thread count (deterministic).
  const int nt = (int)std::max<long long>(1, std::min<long long>(std::min<long long>(32, (long long)std::thread::hardware_concurrency()),
                                                                  std::min<long long>(nnz / 200000 + 1, nc ? nc : 1)));
  std::vector<long long> cb(nt + 1, 0);                    // column block boundaries, balanced by nnz
  for (int t = 1; t < nt; ++t) {
    const long long target = nnz * t / nt;
    cb[t] = std::lower_bound(csr_t.rowptr.begin(), csr_t.rowptr.end(), (int)target) - csr_t.rowptr.begin();
    if (cb[t] > nc) cb[t] = nc;
    if (cb[t] < cb[t - 1]) cb[t] = cb[t - 1];
  }
  cb[nt] = nc;
  std::vector<std::vector<int>> cnt(nt);
  std::vector<int> bad(nt, 0);
  auto run = [&](const std::function<void(int)>& fn) {
    if (nt == 1) { fn(0); return; }
    std::vector<std::thread> th;
    for (int t = 0; t < nt; ++t) th.emplace_back(fn, t);
    for (auto& x : th) x.join();
  };
  run([&](int t) {
    cnt[t].assign(nr, 0);
    for (long long k = csr_t.rowptr[cb[t]]; k < csr_t.rowptr[cb[t + 1]]; ++k) {
      const long long r = M.rowval[k] - base;
      if (r < 0 || r >= nr) { bad[t] = 1; return; }
      csr_t.col[k] = (int)r;
      csr_t.val[k] = (double)vals[k];
      cnt[t][r]++;
    }
  });
  for (int t = 0; t < nt; ++t) if (bad[t]) throw EngineError{COSMO_B200_ERR_INVALID, "rowval out of range"};
  for (long long r = 0; r < nr; ++r) {
    int run_sum = csr.rowptr[r];
    for (int t = 0; t < nt; ++t) { const int c = cnt[t][r]; cnt[t][r] = run_sum; run_sum += c; }   // cnt -> first slot of (t, r)
    csr.rowptr[r + 1] = run_sum;
  }
  run([&](int t) {
    std::vector<int>& next = cnt[t];
    for (long long j = cb[t]; j < cb[t + 1]; ++j)
      for (int k = csr_t.rowptr[j]; k < csr_t.rowptr[j + 1]; ++k) {
        const int dstk = next[csr_t.col[k]]++;
        csr.col[dstk] = (int)j;
        csr.val[dstk] = csr_t.val[k];
      }
  });
}

template <typename T>
Engine<T>::Engine(const cosmo_b200_problem& p, const cosmo_b200_settings& st) : st_(st) {
  if (p.m < 0 || p.n < 0 || p.m >= (1LL << 31) - 8 || p.n >= (1LL << 31) - 8)
    throw EngineError{COSMO_B200_ERR_INVALID, "model size out of range"};
  n_ = (int)p.n; m_ = (int)p.m; device_ = p.device;
  if (p.A.nrows != p.m || p.A.ncols != p.n) throw EngineError{COSMO_B200_ERR_INVALID, "A must be m x n"};
  if (p.P.nrows != p.n || p.P.ncols != p.n) throw EngineError{COSMO_B200_ERR_INVALID, "P must be n x n"};
  if (st.adaptive_rho && st.adaptive_rho_interval < 0) throw EngineError{COSMO_B200_ERR_INVALID, "adaptive_rho_interval < 0"};
  const double t_ctor0 = now_s();
  int ndev = 0;
  cudaError_t de = cudaGetDeviceCount(&ndev);
  if (de != cudaSuccess || ndev == 0)
    throw EngineError{COSMO_B200_ERR_CUDA, "no CUDA device available: the COSMO B200 engine has no CPU fallback"};
  if (device_ < 0 || device_ >= ndev) throw EngineError{COSMO_B200_ERR_INVALID, "bad device ordinal"};
  CUDA_TRY(cudaSetDevice(device_));
  CUDA_TRY(cudaDeviceGetAttribute(&num_sms_, cudaDevAttrMultiProcessorCount, device_));
  if (num_sms_ < 1 || num_sms_ > kMaxGrid) num_sms_ = 148;
  {
    const char* e = getenv("COSMO_B200_NO_WINDOWS");
    use_windows_ = !(e && e[0] == '1');
    const char* ng = getenv("COSMO_B200_NO_GRAPH");
    use_graphs_ = !(ng && ng[0] == '1');
    const char* np_ = getenv("COSMO_B200_NO_PERSISTENT");
    use_persistent_ = !(np_ && np_[0] == '1');
    const char* pc = getenv("COSMO_B200_PERSIST_CTAS");
    if (pc && atoi(pc) > 0) persist_ctas_per_sm_ = atoi(pc);
    const char* dc = getenv("COSMO_B200_DIRECT_CTAS");
    if (dc && atoi(dc) > 0) d_ctas_cap_ = atoi(dc);
    const char* gm = getenv("COSMO_B200_GRAPH_MULTI");
    graph_multi_ = !(gm && gm[0] == '0');
    const char* g = getenv("COSMO_B200_WIN_GROUP");
    if (g && atoi(g) == 8) win_group_ = 8;
  }
  CUDA_TRY(cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking));
  CUDA_TRY(cudaEventCreate(&ev0_));
  CUDA_TRY(cudaEventCreate(&ev1_));
  CUDA_TRY(cudaMallocHost(&h_sc_, SC_COUNT * sizeof(T)));
  CUDA_TRY(cudaMallocHost(&h_isc_, ISC_COUNT * sizeof(int)));

  // ---- sets -> row tables -------------------------------------------------
  long long off = 0;
  std::vector<unsigned char> row_class(m_);
  std::vector<int> row_cone(m_, 0);
  hl_.assign(m_, -INFINITY);
  hu_.assign(m_, INFINITY);
  std::vector<int> soc_off, soc_dim;
  std::vector<PsdConeDesc> psd_descs;
  std::vector<int> c3_off, c3_maxit;
  std::vector<unsigned char> c3_kind;
  std::vector<T> c3_alpha, c3_tol;
  for (long long k = 0; k < p.n_sets; ++k) {
    const cosmo_b200_set& sdesc = p.sets[k];
    if (sdesc.dim < 0 || off + sdesc.dim > m_) throw EngineError{COSMO_B200_ERR_INVALID, "set dimensions exceed m"};
    cosmo_b200_set keep = sdesc; keep.l = keep.u = nullptr;
    sets_.push_back(keep);
    set_off_.push_back((int)off);
    unsigned char cls;
    switch (sdesc.type) {
      case COSMO_B200_ZERO: cls = ROW_ZERO; break;
      case COSMO_B200_NONNEG: cls = ROW_NONNEG; break;
      case COSMO_B200_BOX: {
        cls = ROW_BOX;
        if (!sdesc.l || !sdesc.u) throw EngineError{COSMO_B200_ERR_INVALID, "Box set without bounds"};
        const T* l = static_cast<const T*>(sdesc.l);
        const T* u = static_cast<const T*>(sdesc.u);
        for (long long i = 0; i < sdesc.dim; ++i) {
          if (l[i] > u[i]) throw EngineError{COSMO_B200_ERR_INVALID, "Box set: inconsistent lower/upper bounds"};
          hl_[off + i] = l[i]; hu_[off + i] = u[i];
        }
        break;
      }
      case COSMO_B200_SOC:
        cls = ROW_SOC;
        for (long long i = 0; i < sdesc.dim; ++i) row_cone[off + i] = (int)soc_off.size();
        if (sdesc.dim > 0) { soc_off.push_back((int)off); soc_dim.push_back((int)sdesc.dim); }
        break;
      case COSMO_B200_PSD_SQUARE:
      case COSMO_B200_PSD_TRIANGLE: {
        cls = ROW_PSD;
        long long N;
        if (sdesc.type == COSMO_B200_PSD_SQUARE) {
          N = (long long)llround(sqrt((double)sdesc.dim));
          if (N * N != sdesc.dim) throw EngineError{COSMO_B200_ERR_INVALID, "PsdCone: dimension must be a square"};
        } else {
          N = ((long long)floor(sqrt(1.0 + 8.0 * (double)sdesc.dim)) - 1) / 2;
          while (N * (N + 1) / 2 < sdesc.dim) ++N;
          if (N * (N + 1) / 2 != sdesc.dim) throw EngineError{COSMO_B200_ERR_INVALID, "PsdConeTriangle: dimension must be N(N+1)/2"};
        }
        for (long long i = 0; i < sdesc.dim; ++i) row_cone[off + i] = (int)psd_descs.size();
        if (sdesc.dim > 0) psd_descs.push_back(PsdConeDesc{(int)off, (int)N, sdesc.type == COSMO_B200_PSD_TRIANGLE ? 1 : 0});
        break;
      }
      case COSMO_B200_PSD_TRIANGLE_COMPLEX: {
        cls = ROW_PSD;
        const long long Nc = (long long)llround(sqrt((double)sdesc.dim));
        if (Nc * Nc != sdesc.dim) throw EngineError{COSMO_B200_ERR_INVALID, "complex PsdConeTriangle: dimension must be a square"};
        if (2 * Nc >= (1LL << 15)) throw EngineError{COSMO_B200_ERR_INVALID, "complex PsdConeTriangle: N too large"};
        for (long long i = 0; i < sdesc.dim; ++i) row_cone[off + i] = (int)psd_descs.size();
        // N = 1: project! is max(x, 0) (convexset.jl:404-405), the real 1 x 1 case
        if (sdesc.dim == 1) psd_descs.push_back(PsdConeDesc{(int)off, 1, 1});
        else if (sdesc.dim > 0) psd_descs.push_back(PsdConeDesc{(int)off, (int)(2 * Nc), 2});
        break;
      }
      case COSMO_B200_EXP:
      case COSMO_B200_DUAL_EXP:
      case COSMO_B200_POW:
      case COSMO_B200_DUAL_POW: {
        cls = ROW_CONE3;
        if (sdesc.dim != 3) throw EngineError{COSMO_B200_ERR_INVALID, "exponential / power cones have dimension 3"};
        const bool is_pow = (sdesc.type == COSMO_B200_POW || sdesc.type == COSMO_B200_DUAL_POW);
        if (is_pow && !(sdesc.alpha > 0.0 && sdesc.alpha < 1.0))
          throw EngineError{COSMO_B200_ERR_INVALID, "The exponent alpha of the power cone has to be in (0, 1)."};
        for (int i = 0; i < 3; ++i) row_cone[off + i] = (int)c3_off.size();
        c3_off.push_back((int)off);
        c3_kind.push_back((unsigned char)(sdesc.type - COSMO_B200_EXP));
        c3_alpha.push_back(is_pow ? (T)sdesc.alpha : T(0.5));
        c3_maxit.push_back(sdesc.max_iter > 0 ? sdesc.max_iter : (is_pow ? 20 : 100));   // convexset.jl:503, 631
        c3_tol.push_back(sdesc.tol > 0.0 ? (T)sdesc.tol : (T)1e-8);
        break;
      }
      default:
        throw EngineError{COSMO_B200_ERR_UNSUPPORTED, "unsupported cone type (complex PSD): fall back to the host loop"};
    }
    for (long long i = 0; i < sdesc.dim; ++i) row_class[off + i] = cls;
    off += sdesc.dim;
  }
  if (off != m_) throw EngineError{COSMO_B200_ERR_INVALID, "sum of set dimensions != m"};

  // ---- matrices -----------------------------------------------------------
  {
    const bool dbg = getenv("COSMO_B200_SETUP_DEBUG") != nullptr;
    double tp = now_s();
    auto lap = [&](const char* what) {
      if (dbg) { const double t = now_s(); fprintf(stderr, "[setup] %-22s %.3f s\n", what, t - tp); tp = t; }
    };
    lap("cone tables");
    HostCsr a, at, pp, ppt;
    csc_to_host_csrs<T>(p.A, p.index_base, a, at);
    lap("csc -> csr (A, A')");
    if (st_.kkt_solver == COSMO_B200_KKT_DIRECT) {   // memory gate before anything of the problem is allocated
      csc_to_host_csrs<T>(p.P, p.index_base, pp, ppt);
      direct_plan(a, pp);
    }
    build_csr(A_, a);
    lap("upload csr A");
    build_windows(A_, a);
    lap("windows A");
    build_csr(At_, at);
    lap("upload csr A'");
    build_windows(At_, at);
    lap("windows A'");
    csc_to_host_csrs<T>(p.P, p.index_base, pp, ppt);
    build_csr(P_, pp);
    lap("P");
    // A' and P rows are traversed by the same lane group in the fused operator kernel
    double mean = n_ ? (double)(At_.nnz + P_.nnz) / n_ : 0.0;
    At_.lanes = pick_lanes(mean);
  }
  // ---- vectors ------------------------------------------------------------
  auto up = [&](DevBuf<T>& d, const void* h, size_t cnt) { d.alloc(cnt); if (h) upload_vec(d, h, cnt); };
  up(q_, p.q, n_);
  up(b_, p.b, m_);
  hb_.resize(m_);
  for (int i = 0; i < m_; ++i) hb_[i] = (double)static_cast<const T*>(p.b)[i];
  scaled_ = (p.D && p.Dinv && p.E && p.Einv);
  c_ = p.c;
  if (scaled_) { up(D_, p.D, n_); up(Dinv_, p.Dinv, n_); up(E_, p.E, m_); up(Einv_, p.Einv, m_); }
  row_class_.alloc(m_); row_cone_.alloc(m_); rho_class_.alloc(m_);
  if (m_) {
    CUDA_TRY(cudaMemcpyAsync(row_class_.p, row_class.data(), m_, cudaMemcpyHostToDevice, stream_));
    CUDA_TRY(cudaMemcpyAsync(row_cone_.p, row_cone.data(), m_ * sizeof(int), cudaMemcpyHostToDevice, stream_));
  }
  box_l_.alloc(m_); box_u_.alloc(m_);
  {
    std::vector<T> l(hl_.begin(), hl_.end()), u(hu_.begin(), hu_.end());
    upload_vec(box_l_, l.data(), m_);
    upload_vec(box_u_, u.data(), m_);
    sync();
  }
  // SOC tables (chunks of <= 8192 tail rows)
  n_soc_ = (int)soc_off.size();
  if (n_soc_) {
    const int CH = 8192;
    std::vector<int> cs, cl, ptr(1, 0);
    for (int k = 0; k < n_soc_; ++k) {
      int start = soc_off[k] + 1, len = soc_dim[k] - 1;
      for (int o = 0; o < len; o += CH) { cs.push_back(start + o); cl.push_back(std::min(CH, len - o)); }
      ptr.push_back((int)cs.size());
    }
    n_soc_chunks_ = (int)cs.size();
    soc_off_.upload(soc_off, stream_); soc_dim_.upload(soc_dim, stream_);
    soc_chunk_start_.upload(cs, stream_); soc_chunk_len_.upload(cl, stream_); soc_cone_chunk_ptr_.upload(ptr, stream_);
    soc_norm_.alloc(n_soc_); soc_norm2_.alloc(n_soc_); soc_chunk_sum_.alloc(std::max(n_soc_chunks_, 1));
    sync();
  }
  psd_.init(psd_descs, stream_);
  n_c3_ = (int)c3_off.size();
  if (n_c3_) {
    c3_off_.upload(c3_off, stream_); c3_kind_.upload(c3_kind, stream_); c3_alpha_.upload(c3_alpha, stream_);
    c3_maxit_.upload(c3_maxit, stream_); c3_tol_.upload(c3_tol, stream_);
    sync();
  }

  // ---- state / scratch ------------------------------------------------------
  W_[0].alloc(n_ + m_); W_[1].alloc(n_ + m_);
  xs_.alloc(n_); s_.alloc(m_); mu_.alloc(m_); rho_vec_.alloc(m_);
  ls_.alloc(n_ + m_); t0_.alloc(m_); tm_.alloc(m_); xsol_.alloc(n_);
  rhsb_.alloc(n_ + 8); cb_.alloc(n_ + 8); r_.alloc(n_); u_.alloc(n_); nu_.alloc(m_);
  vec_m_.alloc(m_); vec_n_.alloc(n_ + 8); vec_n2_.alloc(n_); dy_.alloc(m_); dx_.alloc(n_);
  ypart_.alloc((size_t)std::max(n_, m_) * 16);   // nwin <= 16 per-window partial sums
  chunk_ticket_.alloc(kMaxGrid);
  sc_.alloc(SC_COUNT); isc_.alloc(ISC_COUNT);
  partials_.alloc((size_t)kMaxGrid * kMaxRed); ticket_.alloc(1);
  {
    int h[ISC_COUNT] = {0};
    h[ISC_MAXIT] = n_;   // IterativeSolvers default maxiter = size(A, 2)
    CUDA_TRY(cudaMemcpyAsync(isc_.p, h, sizeof(h), cudaMemcpyHostToDevice, stream_));
    sync();
  }
  memset(&xv_, 0, sizeof(xv_));
  rho_ = st_.rho;
  // scaling requested but no scaling matrices handed over: the data are unscaled, equilibrate them here
  // (setup.jl:27-33 -> scale_ruiz!); the host reads D, E, c back with cosmo_b200_get_scaling
  if ((p.flags & COSMO_B200_PROBLEM_EQUILIBRATE) && st_.scaling != 0) {
    if (scaled_) throw EngineError{COSMO_B200_ERR_INVALID, "COSMO_B200_PROBLEM_EQUILIBRATE expects D = Dinv = E = Einv = NULL"};
    equilibrate();
  }
  classify_and_set_rho(true);
  sync();
  if (st_.kkt_solver == COSMO_B200_KKT_DIRECT) {   // the initial factorisation of setup! (setup.jl:56)
    direct_alloc();
    direct_factor();
  }
  create_time_ = now_s() - t_ctor0;
  auto_rho_interval_ = 0;
}

template <typename T>
void Engine<T>::destroy_cg_graphs() {
  for (auto& g : cg_graph_) {
    if (g) cudaGraphExecDestroy(g);
    g = nullptr;
  }
}

template <typename T>
Engine<T>::~Engine() {
  destroy_cg_graphs();
  for (void* p : ipc_opened_) cudaIpcCloseMemHandle(p);
  if (comm_ && g_nccl.CommDestroy) g_nccl.CommDestroy(comm_);
  if (h_sc_) cudaFreeHost(h_sc_);
  if (h_isc_) cudaFreeHost(h_isc_);
  if (h_aa_) cudaFreeHost(h_aa_);
  if (ev0_) cudaEventDestroy(ev0_);
  if (ev1_) cudaEventDestroy(ev1_);
  if (stream_) cudaStreamDestroy(stream_);
}

// classify_constraints! (setup.jl:75-85; convexset.jl:62-69, 831-842) and
// set_rho_vec! / update_rho_vec! (parameters.jl:3-13, 75-81)
template <typename T>
void Engine<T>::classify_and_set_rho(bool reset_rho, bool rebuild_vec) {
  std::vector<unsigned char> cls(m_, 0);
  const double big = st_.COSMO_INFTY * st_.MIN_SCALING;
  for (size_t k = 0; k < sets_.size(); ++k) {
    const int off = set_off_[k];
    const long long dim = sets_[k].dim;
    if (sets_[k].type == COSMO_B200_ZERO) {
      for (long long i = 0; i < dim; ++i) cls[off + i] = 1;
    } else if (sets_[k].type == COSMO_B200_NONNEG) {
      for (long long i = 0; i < dim; ++i) if (hb_[off + i] > big) cls[off + i] = 2;
    } else if (sets_[k].type == COSMO_B200_BOX) {
      for (long long i = 0; i < dim; ++i) {
        const double l = hl_[off + i], u = hu_[off + i];
        if (l < -big && u > big) cls[off + i] = 2;
        else if ((u - l) < st_.RHO_TOL) cls[off + i] = 1;
      }
    }
  }
  if (m_) CUDA_TRY(cudaMemcpyAsync(rho_class_.p, cls.data(), m_, cudaMemcpyHostToDevice, stream_));
  sync();
  if (reset_rho) {
    rho_ = st_.rho;
    rho_updates_.clear();
    rho_updates_.push_back(rho_);
  }
  rho_vec_kernel<T><<<vgrid(m_), kBlock, 0, stream_>>>(m_, rho_class_.p, (T)rho_, (T)st_.RHO_EQ_OVER_RHO_INEQ, (T)st_.RHO_MIN, rho_vec_.p);
  check_launch("rho_vec");
  d_stale_ = true;
}

// scale_ruiz! (scaling.jl:21-116) on the resident data; see ruiz.cuh
template <typename T>
void Engine<T>::equilibrate() {
  const int n = n_, m = m_;
  const T lo = (T)st_.MIN_SCALING, hi = (T)(st_.MAX_SCALING > 0.0 ? st_.MAX_SCALING : 1e4);
  D_.alloc(n, false); Dinv_.alloc(n, false); E_.alloc(m, false); Einv_.alloc(m, false);
  DevBuf<T> cdev;
  cdev.alloc(1, false);
  ruiz_fill_kernel<T><<<vgrid(n), kBlock, 0, stream_>>>(n, D_.p, T(1));
  ruiz_fill_kernel<T><<<vgrid(m), kBlock, 0, stream_>>>(m, E_.p, T(1));
  ruiz_fill_kernel<T><<<1, 32, 0, stream_>>>(1, cdev.p, T(1));
  T* Dw = Dinv_.p;   // the inverse scalings double as work vectors, like in the reference (scaling.jl:37-41)
  T* Ew = Einv_.p;
  auto wgrid = [&](long long rows) { return (int)std::min<long long>((rows * 32 + kBlock - 1) / kBlock + 1, kMaxGrid); };
  for (int it = 0; it < st_.scaling; ++it) {
    // kkt_col_norms! (scaling.jl:3-8)
    ruiz_row_inf_kernel<T><<<wgrid(n), kBlock, 0, stream_>>>(n, P_.view(), D_.p, D_.p, cdev.p, Dw, 0);
    ruiz_row_inf_kernel<T><<<wgrid(n), kBlock, 0, stream_>>>(n, At_.view(), D_.p, E_.p, (const T*)nullptr, Dw, 1);
    ruiz_row_inf_kernel<T><<<wgrid(m), kBlock, 0, stream_>>>(m, A_.view(), E_.p, D_.p, (const T*)nullptr, Ew, 0);
    ruiz_update_kernel<T><<<vgrid(n), kBlock, 0, stream_>>>(n, Dw, D_.p, lo, hi);
    ruiz_update_kernel<T><<<vgrid(m), kBlock, 0, stream_>>>(m, Ew, E_.p, lo, hi);
    // cost scaling (scaling.jl:73-90): column norms of the newly scaled P, |q|_inf
    ruiz_row_inf_kernel<T><<<wgrid(n), kBlock, 0, stream_>>>(n, P_.view(), D_.p, D_.p, cdev.p, Dw, 0);
    ruiz_cost_kernel<T><<<1, 1024, 0, stream_>>>(n, Dw, q_.p, D_.p, cdev.p, lo, hi);
    launches_ += 7;
  }
  // rectify_set_scalings! (scaling.jl:129-142): one scalar per SOC / PSD / exponential / power cone
  {
    std::vector<int> off, dim;
    for (size_t k = 0; k < sets_.size(); ++k) {
      const int t = sets_[k].type;
      if (t != COSMO_B200_ZERO && t != COSMO_B200_NONNEG && t != COSMO_B200_BOX && sets_[k].dim > 0) {
        off.push_back(set_off_[k]);
        dim.push_back((int)sets_[k].dim);
      }
    }
    if (!off.empty()) {
      DevBuf<int> off_d, dim_d;
      off_d.upload(off, stream_); dim_d.upload(dim, stream_);
      ruiz_rectify_kernel<T><<<(int)off.size(), kBlock, 0, stream_>>>(off_d.p, dim_d.p, E_.p);
      sync();
    }
  }
  // apply D, E, c to every copy of the data
  ruiz_apply_csr_kernel<T><<<wgrid(m), kBlock, 0, stream_>>>(m, A_.rowptr.p, A_.col.p, A_.val.p, E_.p, D_.p, (const T*)nullptr);
  ruiz_apply_csr_kernel<T><<<wgrid(n), kBlock, 0, stream_>>>(n, At_.rowptr.p, At_.col.p, At_.val.p, D_.p, E_.p, (const T*)nullptr);
  ruiz_apply_csr_kernel<T><<<wgrid(n), kBlock, 0, stream_>>>(n, P_.rowptr.p, P_.col.p, P_.val.p, D_.p, D_.p, cdev.p);
  if (A_.windowed)
    ruiz_apply_win_kernel<T><<<wgrid((long long)A_.nwin * m), kBlock, 0, stream_>>>(A_.nwin, A_.W, m, n, A_.w_rowptr.p, A_.w_col.p, A_.w_val.p, E_.p, D_.p);
  if (At_.windowed)
    ruiz_apply_win_kernel<T><<<wgrid((long long)At_.nwin * n), kBlock, 0, stream_>>>(At_.nwin, At_.W, n, m, At_.w_rowptr.p, At_.w_col.p, At_.w_val.p, D_.p, E_.p);
  ruiz_finish_n_kernel<T><<<vgrid(n), kBlock, 0, stream_>>>(n, q_.p, D_.p, Dinv_.p, cdev.p);
  ruiz_finish_m_kernel<T><<<vgrid(m), kBlock, 0, stream_>>>(m, b_.p, E_.p, Einv_.p, row_class_.p, box_l_.p, box_u_.p);
  check_launch("ruiz");
  // the rho classification (setup.jl:75-85) looks at the SCALED b and Box bounds: refresh the host mirrors
  {
    std::vector<T> hb(m), hl(m), hu(m);
    T ch = T(1);
    if (m) {
      CUDA_TRY(cudaMemcpyAsync(hb.data(), b_.p, (size_t)m * sizeof(T), cudaMemcpyDeviceToHost, stream_));
      CUDA_TRY(cudaMemcpyAsync(hl.data(), box_l_.p, (size_t)m * sizeof(T), cudaMemcpyDeviceToHost, stream_));
      CUDA_TRY(cudaMemcpyAsync(hu.data(), box_u_.p, (size_t)m * sizeof(T), cudaMemcpyDeviceToHost, stream_));
    }
    CUDA_TRY(cudaMemcpyAsync(&ch, cdev.p, sizeof(T), cudaMemcpyDeviceToHost, stream_));
    sync();
    for (int i = 0; i < m; ++i) { hb_[i] = (double)hb[i]; hl_[i] = (double)hl[i]; hu_[i] = (double)hu[i]; }
    c_ = (double)ch;
  }
  scaled_ = true;
  device_scaled_ = true;
}

template <typename T>
void Engine<T>::get_scaling(void* D, void* E, double* c) {
  if (!scaled_) {
    std::vector<T> one_n(n_, T(1)), one_m(m_, T(1));
    if (D) memcpy(D, one_n.data(), (size_t)n_ * sizeof(T));
    if (E) memcpy(E, one_m.data(), (size_t)m_ * sizeof(T));
    if (c) *c = 1.0;
    return;
  }
  if (D) download_vec(D, D_.p, n_);
  if (E) download_vec(E, E_.p, m_);
  sync();
  if (c) *c = c_;
}

template <typename T>
void Engine<T>::warm_start(const void* x, const void* s, const void* mu) {
  if (x) upload_vec(xs_, x, n_);
  if (s) upload_vec(s_, s, m_);
  if (mu) upload_vec(mu_, mu, m_);
  sync();
}

template <typename T>
void Engine<T>::update_qb(const void* q, const void* b) {
  if (q) upload_vec(q_, q, n_);
  if (b) {
    upload_vec(b_, b, m_);
    for (int i = 0; i < m_; ++i) hb_[i] = (double)static_cast<const T*>(b)[i];
  }
  sync();
  if (b) classify_and_set_rho(false, !is_optimized_);
  sync();
}

template <typename T>
void Engine<T>::update_rho(const void* rho_vec, double rho) {
  if (rho_vec) upload_vec(rho_vec_, rho_vec, m_);
  rho_ = rho;
  d_stale_ = true;
  sync();
}

template <typename T>
void Engine<T>::reset() {
  CUDA_TRY(cudaMemsetAsync(xs_.p, 0, std::max(n_, 1) * sizeof(T), stream_));
  CUDA_TRY(cudaMemsetAsync(s_.p, 0, std::max(m_, 1) * sizeof(T), stream_));
  CUDA_TRY(cudaMemsetAsync(mu_.p, 0, std::max(m_, 1) * sizeof(T), stream_));
  CUDA_TRY(cudaMemsetAsync(xsol_.p, 0, std::max(n_, 1) * sizeof(T), stream_));
  CUDA_TRY(cudaMemsetAsync(W_[0].p, 0, std::max(n_ + m_, 1) * sizeof(T), stream_));
  CUDA_TRY(cudaMemsetAsync(W_[1].p, 0, std::max(n_ + m_, 1) * sizeof(T), stream_));
  if (mr_x_.p) CUDA_TRY(cudaMemsetAsync(mr_x_.p, 0, mr_x_.n * sizeof(T), stream_));
  kkt_counter_ = 1;
  last_cg_iters_ = 1;
  is_optimized_ = false;
  psd_.reset_warm_start();
  classify_and_set_rho(true);
  sync();
}

template <typename T>
void Engine<T>::allreduce_sum(T* buf, size_t count) {
  if (nranks_ <= 1) return;
  int rc = g_nccl.AllReduce(buf, buf, count, sizeof(T) == 8 ? kNcclFloat64 : kNcclFloat32, kNcclSum, comm_, stream_);
  if (rc != 0) throw EngineError{COSMO_B200_ERR_NCCL, "ncclAllReduce(sum) failed"};
}
template <typename T>
void Engine<T>::allreduce_max(T* buf, size_t count) {
  if (nranks_ <= 1) return;
  int rc = g_nccl.AllReduce(buf, buf, count, sizeof(T) == 8 ? kNcclFloat64 : kNcclFloat32, kNcclMax, comm_, stream_);
  if (rc != 0) throw EngineError{COSMO_B200_ERR_NCCL, "ncclAllReduce(max) failed"};
}

template <typename T>
void Engine<T>::comm_init(int nranks, int rank, const void* id128) {
  if (nranks < 1 || rank < 0 || rank >= nranks) throw EngineError{COSMO_B200_ERR_INVALID, "bad rank / nranks"};
  if (nranks > 1 && st_.kkt_solver == COSMO_B200_KKT_DIRECT)
    throw EngineError{COSMO_B200_ERR_UNSUPPORTED, "the direct KKT solver is single-GPU (use CG or MINRES when sharded)"};
  nranks_ = nranks; rank_ = rank;
  if (nranks == 1) return;
  std::string e;
  if (!g_nccl.load(e)) throw EngineError{COSMO_B200_ERR_NCCL, e};
  NcclUniqueId id;
  memcpy(&id, id128, sizeof(id));
  CUDA_TRY(cudaSetDevice(device_));
  int rc = g_nccl.CommInitRank(&comm_, nranks, id, rank);
  if (rc != 0) throw EngineError{COSMO_B200_ERR_NCCL, std::string("ncclCommInitRank failed: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?")};
}

// Peer-memory exchange set-up: every rank exports its exchange buffer + flag array as two CUDA IPC
// handles (64 B each); the host plumbing all-gathers the blobs; attach() maps the peers' buffers.
template <typename T>
void Engine<T>::p2p_export(void* blob128) {
  CUDA_TRY(cudaSetDevice(device_));
  const size_t stride = ((size_t)n_ + 8 + 15) & ~(size_t)15;
  xchg_data_.alloc(2 * (size_t)kMaxRanks * stride);   // [slot][source rank][stride]
  xchg_flags_.alloc(2 * kMaxRanks);
  xchg_seq_.alloc(1);
  xchg_arrive_.alloc(kMaxRanks);
  xv_.stride = stride;
  cudaIpcMemHandle_t hd, hf;
  CUDA_TRY(cudaIpcGetMemHandle(&hd, xchg_data_.p));
  CUDA_TRY(cudaIpcGetMemHandle(&hf, xchg_flags_.p));
  memcpy(blob128, &hd, 64);
  memcpy(static_cast<char*>(blob128) + 64, &hf, 64);
}

template <typename T>
void Engine<T>::p2p_attach(const void* blobs, int nranks) {
  if (nranks != nranks_ || nranks > kMaxRanks) throw EngineError{COSMO_B200_ERR_INVALID, "p2p_attach: rank count mismatch (max 8)"};
  if (!xchg_data_.p) throw EngineError{COSMO_B200_ERR_INVALID, "p2p_attach before p2p_export"};
  CUDA_TRY(cudaSetDevice(device_));
  for (int r = 0; r < nranks; ++r) {
    if (r == rank_) {
      xv_.peer_data[r] = xchg_data_.p;
      xv_.peer_flags[r] = xchg_flags_.p;
      continue;
    }
    cudaIpcMemHandle_t hd, hf;
    memcpy(&hd, static_cast<const char*>(blobs) + (size_t)r * 128, 64);
    memcpy(&hf, static_cast<const char*>(blobs) + (size_t)r * 128 + 64, 64);
    void *pd = nullptr, *pf = nullptr;
    CUDA_TRY(cudaIpcOpenMemHandle(&pd, hd, cudaIpcMemLazyEnablePeerAccess));
    CUDA_TRY(cudaIpcOpenMemHandle(&pf, hf, cudaIpcMemLazyEnablePeerAccess));
    ipc_opened_.push_back(pd);
    ipc_opened_.push_back(pf);
    xv_.peer_data[r] = static_cast<T*>(pd);
    xv_.peer_flags[r] = static_cast<unsigned*>(pf);
  }
  for (int r = nranks; r < kMaxRanks; ++r) { xv_.peer_data[r] = nullptr; xv_.peer_flags[r] = nullptr; }
  xv_.local_flags = xchg_flags_.p;
  xv_.seq = xchg_seq_.p;
  xv_.nranks = nranks;
  xv_.rank = rank_;
  destroy_cg_graphs();
  p2p_ = true;
}

// ---------------------------------------------------------------------------
template <typename T>
template <typename Epi>
void Engine<T>::launch_spmv(const DevCsr<T>& M1, const T* x1, const DevCsr<T>* M2, const T* x2, int nrows,
                            const Epi& epi, RedBuf<T> rb, const char* name) {
  const CsrView<T> v2 = M2 ? M2->view() : CsrView<T>{nullptr, nullptr, nullptr};
  if (M1.windowed) {
    const size_t smem = (size_t)M1.W * sizeof(T);
    // function attributes are per device: one flag per (T, Epi) instantiation AND device ordinal
    static bool configured[64] = {false};
    const int dev_slot = device_ & 63;
    if (!configured[dev_slot] || device_ >= 64) {
      CUDA_TRY(cudaFuncSetAttribute(spmv_win_kernel<T, Epi>, cudaFuncAttributeMaxDynamicSharedMemorySize, 204800));
      configured[dev_slot] = true;
    }
    spmv_win_kernel<T, Epi><<<M1.nctas, kWinThreads, smem, stream_>>>(M1.wview(), x1, v2, x2, epi, rb, ypart_.p,
                                                                      chunk_ticket_.p);
    check_launch(name);
    return;
  }
  const int lanes = M1.lanes;
  const int grid = sgrid(nrows, lanes);
  if (lanes == 32) spmv_kernel<T, 32, Epi><<<grid, kBlock, 0, stream_>>>(M1.view(), x1, v2, x2, nrows, epi, rb);
  else if (lanes == 8) spmv_kernel<T, 8, Epi><<<grid, kBlock, 0, stream_>>>(M1.view(), x1, v2, x2, nrows, epi, rb);
  else spmv_kernel<T, 2, Epi><<<grid, kBlock, 0, stream_>>>(M1.view(), x1, v2, x2, nrows, epi, rb);
  check_launch(name);
}

template <typename T>
void Engine<T>::soc_norms(const T* ws, T* norm_out) {
  if (!n_soc_) return;
  if (n_soc_chunks_) {
    soc_chunk_kernel<T><<<n_soc_chunks_, kBlock, 0, stream_>>>(ws, soc_chunk_start_.p, soc_chunk_len_.p, soc_chunk_sum_.p);
    check_launch("soc_chunk");
  }
  soc_final_kernel<T><<<(n_soc_ + 127) / 128, 128, 0, stream_>>>(soc_chunk_sum_.p, soc_cone_chunk_ptr_.p, n_soc_, norm_out);
  check_launch("soc_final");
}

// admm_z! (solver.jl:7-21) [+ rhs of admm_x!, solver.jl:50-51]
template <typename T>
void Engine<T>::project_device(const T* w, bool with_rhs, const T* ws_rhs) {
  soc_norms(w + n_, soc_norm_.p);
  psd_.project(w + n_, s_.p, stream_, st_.psd_max_sweeps, launches_);
  if (n_c3_) {
    cone3_project_kernel<T><<<(n_c3_ + 127) / 128, 128, 0, stream_>>>(c3_table(), w + n_, s_.p);
    check_launch("cone3_project");
  }
  ProjRhsArgs<T> a;
  a.n = n_; a.m = m_; a.w = w; a.ws_rhs = ws_rhs ? ws_rhs : w + n_;
  a.q = q_.p; a.b = b_.p; a.rho = rho_vec_.p; a.box_l = box_l_.p; a.box_u = box_u_.p;
  a.row_class = row_class_.p; a.row_cone = row_cone_.p;
  a.soc = SocTable<T>{soc_off_.p, soc_norm_.p};
  a.s = s_.p; a.ls = ls_.p; a.t0 = t0_.p; a.sigma = (T)st_.sigma;
  a.do_proj = 1; a.do_rhs = with_rhs ? 1 : 0;
  launch_proj_rhs(a);
}

// c = A' tm + P u + sigma u ; cb[n] = u'c   (second half of reduced_mul!, kktsolver_indirect.jl:61-65)
// Rank 0 alone adds the replicated P / sigma terms of a row-sharded run.
template <typename T>
void Engine<T>::kkt_op_stage2(const int* done, const T* u, const T* t_in, T* c_out, bool exchange) {
  const bool lead = (rank_ == 0);
  const bool px = exchange && p2p_;
  const T sig = lead ? (T)st_.sigma : (T)0;
  const DevCsr<T>* M2 = nullptr;
  const T* pu = nullptr;
  if (At_.windowed) {
    // the slab kernel cannot walk P's rows without unbalancing its window-0 CTAs: P u goes first
    if (lead && P_.nnz > 0) {
      launch_spmv(P_, u, (const DevCsr<T>*)nullptr, (const T*)nullptr, n_, EpiStore<T>{done, vec_n2_.p}, red(SC_TMP0), "spmv_P");
      pu = vec_n2_.p;
    }
  } else if (lead) {
    M2 = &P_;
  }
  launch_spmv(At_, t_in, M2, u, n_, EpiKktOp<T>{done, c_out, u, sig, pu}, red_ptr(cb_.p + n_), "spmv_kkt_op");
  if (px) {
    // one-shot allreduce over NVLink: push [c; u'c] into every peer's exchange buffer (coalesced 16-byte remote
    // stores), the consumers (cg_init / cg_update_xr) wait for the flags and sum their local segments in rank order
    if (c_out != cb_.p) throw EngineError{COSMO_B200_ERR_INVALID, "peer exchange expects the operator output in cb_"};
    const int len = n_ + 1;
    const int gx = std::max(1, std::min(16, (len * (int)sizeof(T) + 32767) / 32768));
    p2p_push_kernel<T><<<dim3(gx, nranks_), kBlock, 0, stream_>>>(xv_, cb_.p, len, done, xchg_arrive_.p);
    check_launch("p2p_push");
  }
}

template <typename T>
void Engine<T>::set_maxit(int v) {
  if (cur_maxit_ == v) return;
  h_isc_[ISC_MAXIT] = v;
  CUDA_TRY(cudaMemcpyAsync(isc_.p + ISC_MAXIT, h_isc_ + ISC_MAXIT, sizeof(int), cudaMemcpyHostToDevice, stream_));
  sync();
  cur_maxit_ = v;
}

// solve!(S::IndirectReducedKKTSolver, y, x) with CG (kktsolver_indirect.jl:36-88).
// Inputs: ls_ = [x1; x2], t0_ = rho .* x2.  Output: xsol_ = y1; then either
//   fused_tail: w_dst = admm_w!(...) computed in the epilogue of the last SpMV, or
//   plain:      nu_ = y2 = rho .* (A y1 - x2).
template <typename T>
void Engine<T>::kkt_core(bool fused_tail, const T* w_src, T* w_dst) {
  const bool lead = (rank_ == 0);
  const bool full = (st_.kkt_solver == COSMO_B200_KKT_MINRES);
  const bool direct = (st_.kkt_solver == COSMO_B200_KKT_DIRECT);
  if (st_.kkt_solver != COSMO_B200_KKT_CG && st_.kkt_solver != COSMO_B200_KKT_MINRES_REDUCED && !full && !direct)
    throw EngineError{COSMO_B200_ERR_UNSUPPORTED, "unknown kkt_solver"};
  if (direct && nranks_ > 1)
    throw EngineError{COSMO_B200_ERR_UNSUPPORTED, "the direct KKT solver is single-GPU (use CG or MINRES when sharded)"};
  if (full && nranks_ > 1)
    throw EngineError{COSMO_B200_ERR_UNSUPPORTED, "full-KKT MINRES is single-GPU in this build (use CG or reduced MINRES when sharded)"};
  if (full) {
    kkt_minres(true);   // xsol_ = y1, nu_ = y2
    if (fused_tail) {
      admm_tail_kernel<T><<<vgrid(m_), kBlock, 0, stream_>>>(m_, nu_.p, rho_vec_.p, s_.p, w_src + n_, w_dst + n_, (T)st_.alpha);
      check_launch("admm_tail");
    }
    return;
  }
  // reduced system: rhs = x1 + A' (rho .* x2)   (kktsolver_indirect.jl:50-54)
  launch_spmv(At_, t0_.p, (const DevCsr<T>*)nullptr, (const T*)nullptr, n_,
              EpiAddVec<T>{nullptr, rhsb_.p, lead ? ls_.p : nullptr}, red(SC_TMP0), "spmv_rhs");
  allreduce_sum(rhsb_.p, n_);
  if (st_.kkt_solver == COSMO_B200_KKT_CG) kkt_cg(isc_.p + ISC_DONE);
  else if (direct) direct_solve();
  else kkt_minres(false);
  kkt_counter_ += 1;
  if (fused_tail) {
    launch_spmv(A_, xsol_.p, (const DevCsr<T>*)nullptr, (const T*)nullptr, m_,
                EpiAdmmTail<T>{nullptr, ls_.p + n_, rho_vec_.p, s_.p, w_src + n_, w_dst + n_, (T)st_.alpha}, red(SC_TMP0),
                "spmv_admm_tail");
  } else {
    launch_spmv(A_, xsol_.p, (const DevCsr<T>*)nullptr, (const T*)nullptr, m_,
                EpiY2<T>{nullptr, nu_.p, ls_.p + n_, rho_vec_.p}, red(SC_TMP0), "spmv_y2");
  }
}

// cg!(previous_solution, L, y1; abstol = tol_k/|y1|, reltol = 0) (kktsolver_indirect.jl:70)
template <typename T>
void Engine<T>::kkt_cg(const int* done) {
  set_maxit(n_);   // IterativeSolvers default maxiter = size(A, 2)
  if (persistent_cg_ok()) {
    launch_persistent_cg(st_.tol_constant / pow((double)kkt_counter_, st_.tol_exponent));
    return;
  }
  // c = L x0 (warm start => one product for the initial residual)
  launch_spmv(A_, xsol_.p, (const DevCsr<T>*)nullptr, (const T*)nullptr, m_, EpiScale<T>{nullptr, tm_.p, rho_vec_.p},
              red(SC_TMP0), "spmv_A_scale");
  kkt_op_stage2(nullptr, xsol_.p, tm_.p, cb_.p, true);
  if (!p2p_) allreduce_sum(cb_.p, n_ + 1);
  const double tol_num = st_.tol_constant / pow((double)kkt_counter_, st_.tol_exponent);
  cg_init_kernel<T><<<vgrid(n_), kBlock, 0, stream_>>>(n_, rhsb_.p, cb_.p, r_.p, u_.p, red(SC_RES2),
                                                      CgInitFin<T>{sc_.p, isc_.p, (T)tol_num, p2p_ ? xchg_seq_.p : nullptr}, p2p_, xv_);
  check_launch("cg_init");
  // NCCL collectives are capturable too; COSMO_B200_GRAPH_MULTI=0 restores eager launches when sharded
  const bool graphs = use_graphs_ && (nranks_ == 1 || graph_multi_);
  if (graphs && !cg_graph_[0]) build_cg_graphs(done);
  int chunk = std::max(last_cg_iters_, 0);
  for (;;) {
    if (graphs) {
      int left = chunk;
      for (int b = 3; b >= 0; --b)
        while (left >= (1 << b)) {
          CUDA_TRY(cudaGraphLaunch(cg_graph_[b], stream_));
          launches_ += (long long)(1 << b) * (At_.windowed && P_.nnz > 0 ? 5 : 4);
          left -= (1 << b);
        }
    } else {
      for (int i = 0; i < chunk; ++i) cg_iteration_launches(done);
    }
    CUDA_TRY(cudaMemcpyAsync(h_isc_, isc_.p, 2 * sizeof(int), cudaMemcpyDeviceToHost, stream_));
    sync();
    if (h_isc_[ISC_DONE]) break;
    chunk = 1;
  }
  const int iters = h_isc_[ISC_IT];
  last_cg_iters_ = iters;
  total_inner_ += iters;
  total_mults_ += 1 + iters;
}

template <typename T>
bool Engine<T>::persistent_cg_ok() {
  if (!use_persistent_ || nranks_ != 1 || A_.windowed || At_.windowed) return false;
  const long long work = A_.nnz + At_.nnz + P_.nnz + 4LL * ((long long)n_ + m_);
  if (work > 6000000LL) return false;           // bigger problems are bandwidth-bound: separate kernels win
  if (persist_grid_ == 0) {
    int coop = 0;
    CUDA_TRY(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, device_));
    if (!coop) { persist_grid_ = -1; return false; }
    const int la = std::max(A_.lanes, At_.lanes);
    persist_lanes_ = la;
    int nb = 0;
    if (la == 32) CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, cg_persistent_kernel<T, 32>, kBlock, 0));
    else if (la == 8) CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, cg_persistent_kernel<T, 8>, kBlock, 0));
    else CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, cg_persistent_kernel<T, 2>, kBlock, 0));
    const long long per = kBlock / la;
    const long long need = std::max<long long>(1, (std::max(n_, m_) + per - 1) / per);
    // a grid barrier costs more the more CTAs take part: at most two CTAs per SM
    persist_grid_ = (int)std::max<long long>(1, std::min<long long>(std::min<long long>((long long)nb, persist_ctas_per_sm_) * num_sms_, need));
    if (nb <= 0) { persist_grid_ = -1; return false; }
    persist_part_.alloc((size_t)persist_grid_ * 4);
  }
  return persist_grid_ > 0;
}

template <typename T>
void Engine<T>::launch_persistent_cg(double tol_num) {
  CgPersistArgs<T> a;
  a.A = A_.view(); a.At = At_.view(); a.P = P_.view();
  a.n = n_; a.m = m_;
  a.rhs = rhsb_.p; a.rho = rho_vec_.p; a.x = xsol_.p; a.r = r_.p; a.u = u_.p; a.tm = tm_.p; a.c = cb_.p;
  a.partA = persist_part_.p; a.partB = persist_part_.p + (size_t)persist_grid_ * 2;
  a.sc = sc_.p; a.isc = isc_.p; a.sigma = (T)st_.sigma; a.tol_num = (T)tol_num;
  void* args[] = {&a};
  const void* fn = persist_lanes_ == 32 ? (const void*)cg_persistent_kernel<T, 32>
                 : persist_lanes_ == 8 ? (const void*)cg_persistent_kernel<T, 8> : (const void*)cg_persistent_kernel<T, 2>;
  CUDA_TRY(cudaLaunchCooperativeKernel(fn, dim3(persist_grid_), dim3(kBlock), args, 0, stream_));
  check_launch("cg_persistent");
  ++persist_solves_;
}

// one CG iteration: u = r + beta u ; c = L u ; alpha = res^2/u'c ; x += alpha u ; r -= alpha c
template <typename T>
void Engine<T>::cg_iteration_launches(const int* done) {
  cg_update_u_kernel<T><<<vgrid(n_), kBlock, 0, stream_>>>(n_, r_.p, u_.p, sc_.p, isc_.p);
  check_launch("cg_update_u");
  launch_spmv(A_, u_.p, (const DevCsr<T>*)nullptr, (const T*)nullptr, m_, EpiScale<T>{done, tm_.p, rho_vec_.p}, red(SC_TMP0),
              "spmv_A_scale");
  kkt_op_stage2(done, u_.p, tm_.p, cb_.p, true);
  if (!p2p_) allreduce_sum(cb_.p, n_ + 1);
  cg_update_xr_kernel<T><<<vgrid(n_), kBlock, 0, stream_>>>(n_, u_.p, cb_.p, cb_.p + n_, xsol_.p, r_.p, sc_.p, isc_.p, red(SC_RES2),
                                                         CgStepFin<T>{sc_.p, isc_.p, p2p_ ? xchg_seq_.p : nullptr}, p2p_, xv_);
  check_launch("cg_update_xr");
}

// Stream-capture 1, 2, 4 and 8 CG iterations into executable graphs.  All kernel arguments are
// fixed device pointers (the scalars alpha, beta, tolerance, done flag live on the device), so the
// graphs stay valid for the lifetime of the handle.
template <typename T>
void Engine<T>::build_cg_graphs(const int* done) {
  // make sure one-time function attributes are set outside of the capture
  cg_iteration_launches(done);
  sync();
  const long long saved = launches_;
  for (int b = 0; b < 4; ++b) {
    cudaGraph_t graph = nullptr;
    CUDA_TRY(cudaStreamBeginCapture(stream_, cudaStreamCaptureModeThreadLocal));
    for (int i = 0; i < (1 << b); ++i) cg_iteration_launches(done);
    CUDA_TRY(cudaStreamEndCapture(stream_, &graph));
    CUDA_TRY(cudaGraphInstantiate(&cg_graph_[b], graph, 0));
    CUDA_TRY(cudaGraphDestroy(graph));
  }
  launches_ = saved;
}

// minres!(previous_solution, L, b; abstol = tol_k/|L x0 - b|, reltol = 0) on the reduced system
// (kktsolver_indirect.jl:72-73) or on the full KKT operator (:123-162).
template <typename T>
void Engine<T>::kkt_minres(bool full) {
  const int npad = (n_ + 3) & ~3;                 // x2 starts 16-byte aligned (TMA bulk copies of v + npad)
  const int L = full ? npad + m_ : n_;
  if (mr_c_.n < (size_t)L) {
    for (auto& b : mr_) b.alloc(L);
    mr_c_.alloc(L);
    if (full) { mr_x_.alloc(L); mr_b_.alloc(L); }
  }
  const int* done = isc_.p + ISC_DONE;
  T* x = full ? mr_x_.p : xsol_.p;
  const T* b = full ? mr_b_.p : rhsb_.p;
  set_maxit(full ? n_ + m_ : n_);
  if (full) {
    CUDA_TRY(cudaMemcpyAsync(mr_b_.p, ls_.p, n_ * sizeof(T), cudaMemcpyDeviceToDevice, stream_));
    CUDA_TRY(cudaMemcpyAsync(mr_b_.p + npad, ls_.p + n_, m_ * sizeof(T), cudaMemcpyDeviceToDevice, stream_));
  }
  // y = L v : reduced (P + sigma I + A' rho A) v  or  full [P + sigma I, A'; A, -1/rho] v
  auto apply = [&](const int* dn, const T* v, T* y) {
    if (full) {
      kkt_op_stage2(dn, v, v + npad, y);                                                        // y1 = A'x2 + P x1 + sigma x1
      launch_spmv(A_, v, (const DevCsr<T>*)nullptr, (const T*)nullptr, m_,
                  EpiKktFullLower<T>{dn, y + npad, v + npad, rho_vec_.p}, red(SC_TMP0), "spmv_kkt_lower");  // y2 = A x1 - x2/rho
    } else {
      launch_spmv(A_, v, (const DevCsr<T>*)nullptr, (const T*)nullptr, m_, EpiScale<T>{dn, tm_.p, rho_vec_.p}, red(SC_TMP0),
                  "spmv_A_scale");
      kkt_op_stage2(dn, v, tm_.p, y);
      allreduce_sum(y, n_);
    }
  };
  T* v_prev = mr_[0].p; T* v_curr = mr_[1].p; T* v_next = mr_[2].p;
  T* w_prev = mr_[3].p; T* w_curr = mr_[4].p; T* w_next = mr_[5].p;
  apply(nullptr, x, mr_c_.p);
  const double tol_num = st_.tol_constant / pow((double)kkt_counter_, st_.tol_exponent);
  minres_init_kernel<T><<<vgrid(L), kBlock, 0, stream_>>>(L, b, mr_c_.p, v_curr, red(SC_RES2), MinresInitFin<T>{sc_.p, isc_.p, (T)tol_num});
  check_launch("minres_init");
  minres_start_kernel<T><<<vgrid(L), kBlock, 0, stream_>>>(L, v_curr, v_prev, w_prev, w_curr, sc_.p);
  check_launch("minres_start");
  int it_host = 0;
  int chunk = std::max(last_cg_iters_, 0);
  for (;;) {
    for (int i = 0; i < chunk; ++i) {
      ++it_host;
      apply(done, v_curr, mr_c_.p);
      minres_lanczos1_kernel<T><<<vgrid(L), kBlock, 0, stream_>>>(L, mr_c_.p, v_prev, v_curr, v_next, sc_.p, isc_.p, red(SC_H3));
      check_launch("minres_lanczos1");
      minres_lanczos2_kernel<T><<<vgrid(L), kBlock, 0, stream_>>>(L, v_curr, v_next, sc_.p, isc_.p, red(SC_RES2), MinresStepFin<T>{sc_.p, isc_.p});
      check_launch("minres_lanczos2");
      minres_update_kernel<T><<<vgrid(L), kBlock, 0, stream_>>>(L, it_host, v_curr, v_next, w_prev, w_curr, w_next, x, sc_.p, isc_.p);
      check_launch("minres_update");
      T* t = v_prev; v_prev = v_curr; v_curr = v_next; v_next = t;
      t = w_prev; w_prev = w_curr; w_curr = w_next; w_next = t;
    }
    CUDA_TRY(cudaMemcpyAsync(h_isc_, isc_.p, 2 * sizeof(int), cudaMemcpyDeviceToHost, stream_));
    sync();
    if (h_isc_[ISC_DONE]) break;
    chunk = 1;
  }
  const int iters = h_isc_[ISC_IT];
  last_cg_iters_ = iters;
  total_inner_ += iters;
  total_mults_ += 2 + iters;   // + init residual + the reference's explicit L*x0 - b (kktsolver_indirect.jl:72,151)
  if (full) {
    CUDA_TRY(cudaMemcpyAsync(xsol_.p, mr_x_.p, n_ * sizeof(T), cudaMemcpyDeviceToDevice, stream_));
    CUDA_TRY(cudaMemcpyAsync(nu_.p, mr_x_.p + npad, m_ * sizeof(T), cudaMemcpyDeviceToDevice, stream_));
    kkt_counter_ += 1;
  }
}

// ---- direct solve of the reduced system (direct.cuh) ------------------------------------------------------------
// Sizes the factor and its workspace from the host copies of A and P, before anything is allocated: refuses when they
// need more than half of the free device memory (the GPU may be shared; the caller falls back to an indirect solver).
template <typename T>
void Engine<T>::direct_plan(const HostCsr& a, const HostCsr& p) {
  // one warp adds a row's entries in parallel: duplicate entries inside a row would race
  for (const HostCsr* h : {&a, &p})
    for (int r = 0; r < h->nrows; ++r)
      for (int k = h->rowptr[r] + 1; k < h->rowptr[r + 1]; ++k)
        if (h->col[k] == h->col[k - 1])
          throw EngineError{COSMO_B200_ERR_INVALID, "the direct KKT solver needs A and P without duplicate entries"};
  d_NT_ = std::max(1, (n_ + direct::NB - 1) / direct::NB);
  d_rows_host_.clear();
  for (int i = 0; i < a.nrows; ++i)
    if (direct::dense_row(a.rowptr[i + 1] - a.rowptr[i], n_)) d_rows_host_.push_back(i);
  d_nd_ = (int)d_rows_host_.size();
  d_ldg_ = (long long)(d_nd_ + direct::NB - 1) / direct::NB * direct::NB;
  const double npad = (double)d_NT_ * direct::NB;
  const double need = 8.0 * (double)direct::tile_off(d_NT_, 0) + 8.0 * npad * (double)d_ldg_ + 16.0 * npad +
                      8.0 * d_NT_ + (double)m_ + 4.0 * d_nd_;
  size_t free_b = 0, total_b = 0;
  CUDA_TRY(cudaMemGetInfo(&free_b, &total_b));
  if (need > 0.5 * (double)free_b) {
    char b[320];
    snprintf(b, sizeof(b), "the direct KKT solver needs %.0f bytes for its dense factor (n = %d) and workspace, more than half of "
             "the %zu bytes of free device memory: use an indirect kkt_solver", need, n_, free_b);
    throw EngineError{COSMO_B200_ERR_UNSUPPORTED, b};
  }
}

template <typename T>
void Engine<T>::direct_alloc() {
  const int NT = d_NT_;
  d_L_.alloc(direct::tile_off(NT, 0), false);
  if (d_nd_) {
    d_Gt_.alloc((size_t)NT * direct::NB * d_ldg_, false);
    d_rows_.upload(d_rows_host_, stream_);
  }
  std::vector<unsigned char> dense(std::max(m_, 1), 0);
  for (int i : d_rows_host_) dense[i] = 1;
  d_dense_.upload(dense, stream_);
  d_y_.alloc((size_t)NT * direct::NB);
  d_x_.alloc((size_t)NT * direct::NB);
  d_dinv_.alloc((size_t)NT * direct::NB);
  d_ready_.alloc(2 * (size_t)NT);
  d_fail_.alloc(1);
  d_epoch_ = 0;
  CUDA_TRY(cudaFuncSetAttribute(direct::trsm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)direct::kPanelSmem));
  // persistent sweep grid: at most two CTAs per SM and at most COSMO_B200_DIRECT_CTAS, all co-resident (cooperative launch)
  int coop = 0;
  CUDA_TRY(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, device_));
  if (!coop) throw EngineError{COSMO_B200_ERR_UNSUPPORTED, "the direct KKT solver needs cooperative launches"};
  d_G_ = 0;
  for (int per_sm = 2; per_sm >= 1 && d_G_ == 0; --per_sm) {
    int G = std::min(NT, per_sm * num_sms_);
    if (d_ctas_cap_ > 0) G = std::min(G, d_ctas_cap_);
    const int R = (NT + G - 1) / G;
    const size_t smem = direct::trsv_smem_bytes(R);
    CUDA_TRY(cudaFuncSetAttribute(direct::trsv_persistent_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int nb = 0;
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, direct::trsv_persistent_kernel<T>, direct::kThreads, smem));
    if (nb >= per_sm || (G <= num_sms_ && nb >= 1)) { d_G_ = G; d_smem_ = smem; }
  }
  if (d_G_ == 0) throw EngineError{COSMO_B200_ERR_UNSUPPORTED, "the direct KKT solver's sweep kernel does not fit on an SM"};
  sync();
}

// assemble M = P + sigma I + A' R A and factor it (right-looking tile Cholesky); one host synchronisation for the
// pivot check, at the reference's own decision points (setup!, update_rho!)
template <typename T>
void Engine<T>::direct_factor() {
  const int NT = d_NT_, Npad = NT * direct::NB;
  cudaEvent_t ev[3];
  for (auto& e : ev) CUDA_TRY(cudaEventCreate(&e));
  CUDA_TRY(cudaEventRecord(ev[0], stream_));
  CUDA_TRY(cudaMemsetAsync(d_L_.p, 0, direct::tile_off(NT, 0) * sizeof(double), stream_));
  CUDA_TRY(cudaMemsetAsync(d_fail_.p, 0, sizeof(int), stream_));
  direct::assemble_sparse_kernel<T><<<(int)(((long long)Npad * 32 + direct::kThreads - 1) / direct::kThreads), direct::kThreads, 0,
                                      stream_>>>(n_, Npad, d_L_.p, P_.view(), At_.view(), A_.view(), rho_vec_.p, d_dense_.p, st_.sigma);
  check_launch("direct_assemble_sparse");
  if (d_nd_) {
    CUDA_TRY(cudaMemsetAsync(d_Gt_.p, 0, (size_t)Npad * d_ldg_ * sizeof(double), stream_));
    direct::gather_dense_kernel<T><<<d_nd_, direct::kThreads, 0, stream_>>>(d_rows_.p, d_ldg_, A_.view(), rho_vec_.p, d_Gt_.p);
    check_launch("direct_gather_dense");
    direct::tile_update_kernel<true><<<(unsigned)((long long)NT * (NT + 1) / 2), direct::kThreads, 0, stream_>>>(
        d_L_.p, NT, 0, 0, d_Gt_.p, d_ldg_, 1.0);
    check_launch("direct_assemble_dense");
  }
  CUDA_TRY(cudaEventRecord(ev[1], stream_));
  for (int K = 0; K < NT; ++K) {
    direct::potrf_kernel<<<1, direct::kThreads, direct::kPanelSmem / 2, stream_>>>(d_L_.p, d_dinv_.p, K, d_fail_.p);
    check_launch("direct_potrf");
    const long long c = NT - K - 1;
    if (c > 0) {
      direct::trsm_kernel<<<(unsigned)c, direct::kThreads, direct::kPanelSmem, stream_>>>(d_L_.p, K);
      check_launch("direct_trsm");
      direct::tile_update_kernel<false><<<(unsigned)(c * (c + 1) / 2), direct::kThreads, 0, stream_>>>(d_L_.p, NT, K + 1, K, nullptr, 0, -1.0);
      check_launch("direct_update");
    }
  }
  CUDA_TRY(cudaEventRecord(ev[2], stream_));
  int fail = 0;
  CUDA_TRY(cudaMemcpyAsync(&fail, d_fail_.p, sizeof(int), cudaMemcpyDeviceToHost, stream_));
  sync();
  float ms_asm = 0.f, ms_fac = 0.f;
  CUDA_TRY(cudaEventElapsedTime(&ms_asm, ev[0], ev[1]));
  CUDA_TRY(cudaEventElapsedTime(&ms_fac, ev[1], ev[2]));
  for (auto& e : ev) cudaEventDestroy(e);
  if (getenv("COSMO_B200_SETUP_DEBUG"))
    fprintf(stderr, "[direct] n %d NT %d dense rows %d assembly %.3f ms factorisation %.3f ms pivot failure in tile column %d\n",
            n_, NT, d_nd_, ms_asm, ms_fac, fail - 1);
  // positive_inertia(ldlfact) == n || error(...) (kktsolver.jl:304): inertia (n, m, 0) <=> M positive definite
  if (fail) throw EngineError{COSMO_B200_ERR_INVALID, "Objective function is not convex."};
  const double sec = 1e-3 * ((double)ms_asm + (double)ms_fac);
  if (d_factorizations_ == 0) d_init_s_ = sec; else d_update_s_ += sec;
  ++d_factorizations_;
  d_stale_ = false;
}

// xsol_ = M^-1 rhsb_ : both triangular sweeps in one cooperative launch
template <typename T>
void Engine<T>::direct_solve() {
  if (++d_epoch_ == 0) {   // the ready flags carry the epoch: clear them once per 2^32 solves
    CUDA_TRY(cudaMemsetAsync(d_ready_.p, 0, 2 * (size_t)d_NT_ * sizeof(unsigned), stream_));
    d_epoch_ = 1;
  }
  direct::TrsvArgs<T> a;
  a.L = d_L_.p; a.dinv = d_dinv_.p; a.n = n_; a.NT = d_NT_; a.G = d_G_;
  a.rhs = rhsb_.p; a.out = xsol_.p; a.y = d_y_.p; a.x = d_x_.p;
  a.ready_f = d_ready_.p; a.ready_b = d_ready_.p + d_NT_; a.epoch = d_epoch_;
  void* args[] = {&a};
  CUDA_TRY(cudaLaunchCooperativeKernel((const void*)direct::trsv_persistent_kernel<T>, dim3(d_G_), dim3(direct::kThreads), args,
                                       d_smem_, stream_));
  check_launch("direct_trsv");
}

// calculate_residuals! + max_res_component_norm + calculate_cost! (residuals.jl:30-96, 143-147)
template <typename T>
void Engine<T>::compute_residuals(const T* x, const T* s, const T* mu, bool ignore_scaling, double out[5]) {
  const bool unscale = (st_.scaling != 0) && scaled_ && !ignore_scaling;
  launch_spmv(A_, x, (const DevCsr<T>*)nullptr, (const T*)nullptr, m_,
              EpiPrimalRes<T>{nullptr, s, b_.p, unscale ? Einv_.p : nullptr, nullptr}, red(SC_TMP0), "spmv_primal_res");
  allreduce_max(sc_.p + SC_TMP0, 4);
  launch_spmv(At_, mu, (const DevCsr<T>*)nullptr, (const T*)nullptr, n_, EpiStore<T>{nullptr, vec_n_.p}, red(SC_TMP4),
              "spmv_At_mu");
  allreduce_sum(vec_n_.p, n_);
  // slots: [SC_TMP0..3] primal maxes are read first, the dual pass then reuses TMP0.. via a second read
  read_scalars(SC_TMP0, 4);
  const double rp = (double)h_sc_[SC_TMP0], m1 = (double)h_sc_[SC_TMP0 + 1], m2 = (double)h_sc_[SC_TMP0 + 2], m3 = (double)h_sc_[SC_TMP0 + 3];
  // P lanes may differ from A' lanes: P_ has its own
  launch_spmv(P_, x, (const DevCsr<T>*)nullptr, (const T*)nullptr, n_,
              EpiDualRes<T>{nullptr, x, q_.p, vec_n_.p, unscale ? Dinv_.p : nullptr, unscale ? (T)(1.0 / c_) : (T)1},
              red(SC_TMP0), "spmv_dual_res");
  read_scalars(SC_TMP0, 6);
  const double xPx = (double)h_sc_[SC_TMP0], qx = (double)h_sc_[SC_TMP0 + 1];
  const double rd = (double)h_sc_[SC_TMP0 + 2], d1 = (double)h_sc_[SC_TMP0 + 3], d2 = (double)h_sc_[SC_TMP0 + 4], d3 = (double)h_sc_[SC_TMP0 + 5];
  auto nmax = [](double a, double b) { return (a > b || a != a) ? a : b; };
  out[0] = rp;
  out[1] = rd;
  out[2] = nmax(nmax(m1, m2), m3);
  out[3] = nmax(nmax(d1, d2), d3);
  out[4] = (1.0 / c_) * (0.5 * xPx + qx);
}

// adapt_rho_vec! / update_rho_vec! (parameters.jl:53-92)
template <typename T>
bool Engine<T>::adapt_rho(const T* x) {
  double r[5];
  compute_residuals(x, s_.p, mu_.p, true, r);
  double rp = r[0] / (r[2] + 1e-10);
  double rd = r[1] / (r[3] + 1e-10);
  double new_rho = rho_ * sqrt(rp / (rd + 1e-10));
  new_rho = std::min(std::max(new_rho, st_.RHO_MIN), st_.RHO_MAX);
  if (new_rho > st_.adaptive_rho_tolerance * rho_ || new_rho < (1.0 / st_.adaptive_rho_tolerance) * rho_) {
    rho_ = new_rho;
    rho_vec_kernel<T><<<vgrid(m_), kBlock, 0, stream_>>>(m_, rho_class_.p, (T)rho_, (T)st_.RHO_EQ_OVER_RHO_INEQ, (T)st_.RHO_MIN, rho_vec_.p);
    check_launch("rho_vec");
    d_stale_ = true;   // update_rho! refactors (parameters.jl:86), lazily before the next solve
    rho_updates_.push_back(new_rho);
    return true;
  }
  return false;
}

// is_primal_infeasible! (infeasibility.jl:1-29); dy_ holds delta_y
template <typename T>
bool Engine<T>::primal_infeasible() {
  const T eps = (T)st_.eps_prim_inf;
  scaled_norminf_kernel<T><<<vgrid(m_), kBlock, 0, stream_>>>(m_, scaled_ ? E_.p : nullptr, dy_.p, red(SC_TMP0));
  check_launch("norminf_dy");
  allreduce_max(sc_.p + SC_TMP0, 1);
  read_scalars(SC_TMP0, 1);
  const double norm_dy = (double)h_sc_[SC_TMP0];
  if (!(norm_dy > st_.eps_prim_inf)) return false;
  launch_spmv(At_, dy_.p, (const DevCsr<T>*)nullptr, (const T*)nullptr, n_, EpiStore<T>{nullptr, vec_n_.p}, red(SC_TMP0), "spmv_At_dy");
  allreduce_sum(vec_n_.p, n_);
  scaled_norminf_kernel<T><<<vgrid(n_), kBlock, 0, stream_>>>(n_, scaled_ ? Dinv_.p : nullptr, vec_n_.p, red(SC_TMP0));
  check_launch("norminf_Atdy");
  read_scalars(SC_TMP0, 1);
  if (!((double)h_sc_[SC_TMP0] <= st_.eps_prim_inf * norm_dy)) return false;
  scal_kernel<T><<<vgrid(m_), kBlock, 0, stream_>>>(m_, (T)(-1.0 / norm_dy), dy_.p);
  check_launch("scal_dy");
  dot_kernel<T><<<vgrid(m_), kBlock, 0, stream_>>>(m_, dy_.p, b_.p, red(SC_TMP0));
  check_launch("dot_dy_b");
  cone_rows_certificate_kernel<T><<<vgrid(m_), kBlock, 0, stream_>>>(m_, 0, dy_.p, row_class_.p, box_l_.p, box_u_.p, eps, red(SC_TMP1));
  check_launch("cone_cert_primal");
  // SOC: -v in K*  <=>  |v[2:]| <= tol - v[1]  ;  PSD: -V + tol I positive definite
  T flag = 0;
  if (n_soc_) {
    soc_norms(dy_.p, soc_norm2_.p);
    soc_cert_kernel<T><<<1, kBlock, 0, stream_>>>(n_soc_, soc_off_.p, soc_norm2_.p, dy_.p, eps, sc_.p + SC_TMP3);
    check_launch("soc_cert");
  } else {
    CUDA_TRY(cudaMemsetAsync(sc_.p + SC_TMP3, 0, sizeof(T), stream_));
  }
  if (n_c3_) {
    cone3_cert_kernel<T><<<1, kBlock, 0, stream_>>>(c3_table(), dy_.p, eps, sc_.p + SC_TMP5);
    check_launch("cone3_cert");
  } else {
    CUDA_TRY(cudaMemsetAsync(sc_.p + SC_TMP5, 0, sizeof(T), stream_));
  }
  const bool psd_ok = psd_.certificate(dy_.p, /*negate=*/true, (double)eps, stream_, st_.psd_max_sweeps, launches_);
  (void)flag;
  // the PSD verdict is a host bool of THIS rank: put it next to the device flags so that the
  // max-allreduce makes every rank take the same decision
  h_sc_[SC_TMP4] = psd_ok ? T(0) : T(1);
  CUDA_TRY(cudaMemcpyAsync(sc_.p + SC_TMP4, h_sc_ + SC_TMP4, sizeof(T), cudaMemcpyHostToDevice, stream_));
  if (nranks_ > 1) {
    allreduce_sum(sc_.p + SC_TMP0, 2);   // dy'b, box support sum
    allreduce_max(sc_.p + SC_TMP2, 4);   // flags: rows, SOC, PSD, Exp/Pow
  }
  read_scalars(SC_TMP0, 6);
  const double dyt_b = (double)h_sc_[SC_TMP0];
  const double box_sum = (double)h_sc_[SC_TMP1];
  const bool cone_bad = (h_sc_[SC_TMP2] != 0) || (h_sc_[SC_TMP3] != 0) || (h_sc_[SC_TMP4] != 0) || (h_sc_[SC_TMP5] != 0);
  const double sF = (cone_bad ? INFINITY : 0.0) + box_sum - dyt_b;
  return sF <= st_.eps_prim_inf;
}

// is_dual_infeasible! (infeasibility.jl:32-68); dx_ holds delta_x
template <typename T>
bool Engine<T>::dual_infeasible() {
  const T eps = (T)st_.eps_dual_inf;
  scaled_norminf_kernel<T><<<vgrid(n_), kBlock, 0, stream_>>>(n_, scaled_ ? D_.p : nullptr, dx_.p, red(SC_TMP0));
  check_launch("norminf_dx");
  dot_kernel<T><<<vgrid(n_), kBlock, 0, stream_>>>(n_, q_.p, dx_.p, red(SC_TMP1));
  check_launch("dot_q_dx");
  read_scalars(SC_TMP0, 2);
  const double norm_dx = (double)h_sc_[SC_TMP0];
  if (!(norm_dx > st_.eps_dual_inf)) return false;
  if (!((double)h_sc_[SC_TMP1] / (norm_dx * c_) < -st_.eps_dual_inf)) return false;
  launch_spmv(P_, dx_.p, (const DevCsr<T>*)nullptr, (const T*)nullptr, n_,
              EpiStoreScaledMax<T>{nullptr, nullptr, scaled_ ? Dinv_.p : nullptr}, red(SC_TMP0), "spmv_P_dx");
  read_scalars(SC_TMP0, 1);
  if (!((double)h_sc_[SC_TMP0] / (norm_dx * c_) <= st_.eps_dual_inf)) return false;
  launch_spmv(A_, dx_.p, (const DevCsr<T>*)nullptr, (const T*)nullptr, m_, EpiStore<T>{nullptr, vec_m_.p}, red(SC_TMP0), "spmv_A_dx");
  if (scaled_) {
    scale_kernel<T><<<vgrid(m_), kBlock, 0, stream_>>>(m_, Einv_.p, vec_m_.p, vec_m_.p);
    check_launch("scale_Adx");
  }
  scal_kernel<T><<<vgrid(m_), kBlock, 0, stream_>>>(m_, (T)(1.0 / norm_dx), vec_m_.p);
  check_launch("scal_Adx");
  cone_rows_certificate_kernel<T><<<vgrid(m_), kBlock, 0, stream_>>>(m_, 1, vec_m_.p, row_class_.p, box_l_.p, box_u_.p, eps, red(SC_TMP1));
  check_launch("cone_cert_dual");
  if (n_soc_) {
    soc_norms(vec_m_.p, soc_norm2_.p);
    soc_cert_kernel<T><<<1, kBlock, 0, stream_>>>(n_soc_, soc_off_.p, soc_norm2_.p, vec_m_.p, eps, sc_.p + SC_TMP3);
    check_launch("soc_cert");
  } else {
    CUDA_TRY(cudaMemsetAsync(sc_.p + SC_TMP3, 0, sizeof(T), stream_));
  }
  if (n_c3_) {
    cone3_cert_kernel<T><<<1, kBlock, 0, stream_>>>(c3_table(), vec_m_.p, eps, sc_.p + SC_TMP5);
    check_launch("cone3_cert");
  } else {
    CUDA_TRY(cudaMemsetAsync(sc_.p + SC_TMP5, 0, sizeof(T), stream_));
  }
  const bool psd_ok = psd_.certificate(vec_m_.p, /*negate=*/true, (double)eps, stream_, st_.psd_max_sweeps, launches_);
  h_sc_[SC_TMP4] = psd_ok ? T(0) : T(1);
  CUDA_TRY(cudaMemcpyAsync(sc_.p + SC_TMP4, h_sc_ + SC_TMP4, sizeof(T), cudaMemcpyHostToDevice, stream_));
  if (nranks_ > 1) allreduce_max(sc_.p + SC_TMP2, 4);
  read_scalars(SC_TMP2, 4);
  return (h_sc_[SC_TMP2] == 0) && (h_sc_[SC_TMP3] == 0) && (h_sc_[SC_TMP4] == 0) && (h_sc_[SC_TMP5] == 0);
}

// ---------------------------------------------------------------------------
// Accelerator: AndersonAccelerator{T, Type2{QRDecomp}, RestartedMemory, NoRegularizer} (aa.cuh)
// ---------------------------------------------------------------------------
template <typename T>
void Engine<T>::aa_prepare() {   // _make_accelerator!, setup.jl:10-14 (built once per dimension / memory)
  const long long dim = (long long)n_ + m_;
  if (st_.accelerator_mem <= 2) throw EngineError{COSMO_B200_ERR_INVALID, "accelerator: Memory has to be bigger than two."};
  if (st_.accelerator_mem > 32 && dim > 32)
    throw EngineError{COSMO_B200_ERR_UNSUPPORTED, "accelerator_mem > 32 is not supported by the device accelerator"};
  int mem = (int)std::min<long long>(st_.accelerator_mem, std::max<long long>(dim, 1));   // mem = min(mem, dim)
  if (aa_mem_ != mem) {
    aaG_.alloc((size_t)dim * mem, false); aaQ_.alloc((size_t)dim * mem, false);
    aaR_.alloc((size_t)mem * mem); aa_eta_.alloc(32);
    aa_glast_.alloc(dim); aa_f_.alloc(dim); aa_flast_.alloc(dim); aa_sc_.alloc(AA_SC_COUNT);
    if (!h_aa_) CUDA_TRY(cudaMallocHost(&h_aa_, AA_SC_COUNT * sizeof(T)));
    aa_mem_ = mem;
  }
  aa_restart();               // setup.jl:47-49
  aa_active_ = false; aa_success_ = false;
  aa_accelerated_ = aa_declined_ = 0;
}

// CA.update!(aa, g = w, x = w_prev): history columns + QR update by modified Gram-Schmidt
template <typename T>
void Engine<T>::aa_update(const T* g, const T* x) {
  const int dim = n_ + m_, lo = (rank_ == 0) ? 0 : n_;
  const int grid = vgrid(dim);
  if (aa_init_) {
    aa_update_kernel<T><<<grid, kBlock, 0, stream_>>>(dim, lo, g, x, aa_f_.p, aa_flast_.p, aa_glast_.p, (T*)nullptr, (T*)nullptr, 1,
                                                      red_ptr(aa_sc_.p + AA_F2));
    check_launch("aa_update");
    allreduce_sum(aa_sc_.p + AA_F2, 1);
    aa_init_ = false;
    return;
  }
  int j = aa_iter_ % aa_mem_;
  if (j == 0 && aa_iter_ != 0) aa_iter_ = 0;   // RestartedMemory: the history is full, start again
  T* Gj = aaG_.p + (size_t)j * dim;
  T* q = aaQ_.p + (size_t)j * dim;
  aa_update_kernel<T><<<grid, kBlock, 0, stream_>>>(dim, lo, g, x, aa_f_.p, aa_flast_.p, aa_glast_.p, Gj, q, 0,
                                                    red_ptr(aa_sc_.p + AA_F2));
  check_launch("aa_update");
  allreduce_sum(aa_sc_.p + AA_F2, 1);
  T* Rj = aaR_.p + (size_t)j * aa_mem_;        // column j of R
  for (int i = 0; i <= j; ++i) {
    const T* Qp = i > 0 ? aaQ_.p + (size_t)(i - 1) * dim : nullptr;
    const T* Qi = i < j ? aaQ_.p + (size_t)i * dim : nullptr;
    T* out = i < j ? Rj + i : aa_sc_.p + AA_NRM2;
    aa_mgs_kernel<T><<<grid, kBlock, 0, stream_>>>(dim, lo, q, Qp, i > 0 ? Rj + (i - 1) : nullptr, Qi, red_ptr(out));
    check_launch("aa_mgs");
    allreduce_sum(out, 1);
  }
  aa_normalize_kernel<T><<<grid, kBlock, 0, stream_>>>(dim, q, aa_sc_.p + AA_NRM2, Rj + j);
  check_launch("aa_normalize");
  ++aa_iter_;
}

// CA.accelerate!(g = w, ...): w -= G eta with R eta = Q'f; returns was_successful(aa)
template <typename T>
bool Engine<T>::aa_accelerate(T* g) {
  const int l = std::min(aa_iter_, aa_mem_);
  if (l < std::max(st_.accelerator_min_mem, 1)) return false;
  const int dim = n_ + m_, lo = (rank_ == 0) ? 0 : n_;
  const int grid = vgrid(dim);
  for (int c0 = 0; c0 < l; c0 += 8) {
    aa_qtf_kernel<T><<<grid, kBlock, 0, stream_>>>(dim, lo, aa_f_.p, aaQ_.p, (size_t)dim, c0, std::min(8, l - c0),
                                                   red_ptr(aa_eta_.p + c0));
    check_launch("aa_qtf");
  }
  allreduce_sum(aa_eta_.p, l);
  aa_solve_kernel<T><<<1, 32, 0, stream_>>>(aaR_.p, aa_mem_, l, aa_eta_.p, aa_sc_.p + AA_FLAG);
  check_launch("aa_solve");
  aa_apply_kernel<T><<<grid, kBlock, 0, stream_>>>(dim, g, aaG_.p, (size_t)dim, l, aa_eta_.p, aa_sc_.p + AA_FLAG);
  check_launch("aa_apply");
  CUDA_TRY(cudaMemcpyAsync(h_aa_ + AA_FLAG, aa_sc_.p + AA_FLAG, sizeof(T), cudaMemcpyDeviceToHost, stream_));
  sync();
  return h_aa_[AA_FLAG] != T(0);
}

// ---------------------------------------------------------------------------
// The hot loop: COSMO.optimize!, src/solver.jl:125-167 (SURVEY.md Appendix A)
// ---------------------------------------------------------------------------
template <typename T>
void Engine<T>::solve(cosmo_b200_result* out) {
  const double t_start = now_s();
  CUDA_TRY(cudaSetDevice(device_));
  const int n = n_, m = m_;
  const long long launches0 = launches_;
  total_inner_ = 0; total_mults_ = 0;
  persist_solves_ = 0;
  CUDA_TRY(cudaMemsetAsync(isc_.p + ISC_TOTAL, 0, sizeof(int), stream_));
  int status = COSMO_B200_UNDETERMINED;
  double cost = INFINITY;
  double info[5] = {INFINITY, INFINITY, 0.0, 0.0, INFINITY};
  long long iter = 0;
  bool rho_update_due = false, infeasibility_check_due = false;
  double res_time = 0.0;

  // warm starting the operator variable (solver.jl:128-129): w_x = x, w_s = mu ./ rho + s
  cur_ = 0; prev_ = 1;
  CUDA_TRY(cudaMemcpyAsync(W_[cur_].p, xs_.p, n * sizeof(T), cudaMemcpyDeviceToDevice, stream_));
  ws_from_mu_kernel<T><<<vgrid(m), kBlock, 0, stream_>>>(m, rho_vec_.p, mu_.p, s_.p, W_[cur_].p + n);
  check_launch("ws_from_mu");
  is_optimized_ = true;
  // phase timers: on request (verbose & 2 = settings.verbose_timing) and for every problem that is not latency-bound
  {
    const bool timers = (st_.verbose & 2) != 0 || (long long)n + m >= 20000 || !psd_.large_h.empty();
    t_proj_.enable(timers);
    t_kkt_.enable(timers);
  }
  CUDA_TRY(cudaEventRecord(ev0_, stream_));
  const double iter_start = now_s();
  // setup time as the reference counts it (ws.times.setup_time): the host's figure when it reports one (it then includes
  // the creation of this engine), else the engine's own creation time
  const double setup_time_total = st_.setup_time > 0.0 ? st_.setup_time : create_time_;

  // x-step + w-step reading W[src], writing W[dst]
  auto xw_step = [&](int src, int dst, bool do_proj, const T* ws_override) {
    const T* w = W_[src].p;
    const T* ws_rhs = ws_override ? ws_override : w + n;
    if (do_proj) {
      t_proj_.begin(stream_);
      project_device(w, true, ws_rhs);      // admm_z! fused with the right-hand side of admm_x! (one pass over w)
      t_proj_.end(stream_);
    } else {
      ProjRhsArgs<T> a;
      a.n = n; a.m = m; a.w = w; a.ws_rhs = ws_rhs; a.q = q_.p; a.b = b_.p; a.rho = rho_vec_.p;
      a.box_l = box_l_.p; a.box_u = box_u_.p; a.row_class = row_class_.p; a.row_cone = row_cone_.p;
      a.soc = SocTable<T>{soc_off_.p, soc_norm_.p};
      a.s = s_.p; a.ls = ls_.p; a.t0 = t0_.p; a.sigma = (T)st_.sigma; a.do_proj = 0; a.do_rhs = 1;
      launch_proj_rhs(a);
    }
    // the tail reads w_s from ws_rhs's buffer and writes W[dst] (elementwise, may alias)
    T* wd = W_[dst].p;
    ensure_factor();
    t_kkt_.begin(stream_);
    kkt_core(true, ws_override ? (ws_override - n) : w, wd);
    t_kkt_.end(stream_);
    wx_update_kernel<T><<<vgrid(n), kBlock, 0, stream_>>>(n, w, xsol_.p, (T)st_.alpha, wd);
    check_launch("wx_update");
  };

  // one initialisation step (solver.jl:137-138)
  xw_step(cur_, 1 - cur_, false, nullptr);
  cur_ = 1 - cur_; prev_ = 1 - cur_;

  const bool use_aa = (st_.accelerator == COSMO_B200_ACC_ANDERSON);
  long long safeguarding_iter = 0;
  if (use_aa) aa_prepare();
  // update_suggested (solver.jl:284-292): with an Anderson accelerator, rho updates and the infeasibility
  // snapshot wait for the next iteration whose candidate was not accelerated
  auto suggested = [&](bool due) { return due && !(use_aa && aa_success_); };

  while (iter + safeguarding_iter < st_.max_iter) {
    ++iter;
    // acceleration_pre! (accelerator_interface.jl:58-75), ImmediateActivation (:24-28)
    if (use_aa) {
      if (!aa_active_ && iter >= 2) aa_active_ = true;
      if (aa_active_) {
        aa_update(W_[cur_].p, W_[prev_].p);
        aa_success_ = aa_accelerate(W_[cur_].p);   // overwrites w with the candidate
        if (aa_success_) ++aa_accelerated_;
      }
    }
    if (suggested(infeasibility_check_due)) {  // solver.jl:145-148
      recover_mu(W_[prev_].p);
      CUDA_TRY(cudaMemcpyAsync(dy_.p, mu_.p, m * sizeof(T), cudaMemcpyDeviceToDevice, stream_));
    }
    // w_prev = w (solver.jl:151): the current buffer becomes w_prev, the other one receives w_{k+1}
    const int src = cur_, dst = 1 - cur_;
    // rho adaptation rules (solver.jl:242-282)
    // automatic interval (solver.jl:244-256): once the loop has run for adaptive_rho_fraction * setup_time, fix the
    // interval at the current iteration count rounded to a multiple of check_termination (at least one multiple)
    if (st_.adaptive_rho && st_.adaptive_rho_interval == 0 && auto_rho_interval_ == 0 &&
        (now_s() - iter_start) > st_.adaptive_rho_fraction * setup_time_total) {
      const long long N = st_.check_termination > 0 ? st_.check_termination : 25;
      const double xr = (double)iter + 0.5 * (double)N;            // round_multiple, algebra.jl:245-247
      const long long rm = (long long)floor(xr - fmod(xr, (double)N));
      auto_rho_interval_ = (int)std::max<long long>(rm, N);
    }
    const int rho_interval = st_.adaptive_rho_interval > 0 ? st_.adaptive_rho_interval : auto_rho_interval_;
    if (st_.adaptive_rho && rho_interval > 0 && (iter % rho_interval) == 0 &&
        (long long)(rho_updates_.size() - 1) < st_.adaptive_rho_max_adaptions)
      rho_update_due = true;
    if (suggested(rho_update_due)) {
      rho_update_due = false;
      t_proj_.begin(stream_);
      project_device(W_[src].p, false, nullptr);          // admm_z!
      t_proj_.end(stream_);
      recover_mu(W_[src].p);                               // w_prev == w here
      const double t0 = now_s();
      const bool adapted = adapt_rho(W_[src].p);
      res_time += now_s() - t0;
      if (adapted) {
        if (use_aa) aa_restart();   // the operator changed: CA.restart! (solver.jl:272-275)
        // w[n+1:end] = mu ./ rho + s (solver.jl:278), kept apart from w_prev
        ws_from_mu_kernel<T><<<vgrid(m), kBlock, 0, stream_>>>(m, rho_vec_.p, mu_.p, s_.p, W_[dst].p + n);
        check_launch("ws_from_mu");
        xw_step(src, dst, false, W_[dst].p + n);
      } else {
        xw_step(src, dst, false, nullptr);
      }
    } else {
      xw_step(src, dst, true, nullptr);
    }
    prev_ = src; cur_ = dst;
    // acceleration_post! (accelerator_interface.jl:85-114): safeguard the accelerated candidate
    if (use_aa && aa_active_ && aa_success_ && st_.safeguard) {
      const int dim = n + m, lo = (rank_ == 0) ? 0 : n;
      aa_res_kernel<T><<<vgrid(dim), kBlock, 0, stream_>>>(dim, lo, W_[prev_].p, W_[cur_].p, aa_f_.p, red_ptr(aa_sc_.p + AA_FACC2));
      check_launch("aa_res");
      allreduce_sum(aa_sc_.p + AA_FACC2, 1);
      CUDA_TRY(cudaMemcpyAsync(h_aa_, aa_sc_.p, 2 * sizeof(T), cudaMemcpyDeviceToHost, stream_));
      sync();
      const double nrm_f = sqrt((double)h_aa_[AA_F2]), nrm_f_acc = sqrt((double)h_aa_[AA_FACC2]);
      if (nrm_f_acc > nrm_f * st_.safeguard_tol) {
        // decline: w_prev = w = g_last, then one plain ADMM step from there (:100-106)
        CUDA_TRY(cudaMemcpyAsync(W_[prev_].p, aa_glast_.p, (size_t)dim * sizeof(T), cudaMemcpyDeviceToDevice, stream_));
        xw_step(prev_, cur_, true, nullptr);
        ++safeguarding_iter;
        ++aa_declined_;
      }
    }

    // check_termination! (solver.jl:303-356)
    if ((st_.check_termination > 0 && iter % st_.check_termination == 0) || iter == 1) {
      const double t0 = now_s();
      recover_mu(W_[prev_].p);
      compute_residuals(W_[prev_].p, s_.p, mu_.p, false, info);
      res_time += now_s() - t0;
      cost = info[4];
      if (fabs(cost) > 1e20) { status = COSMO_B200_UNSOLVED; break; }
      if (st_.verbose & 1) printf("%lld\t%.4e\t%.4e\t%.4e\t%.4e\n", iter, cost, info[0], info[1], rho_);
      // has_converged (residuals.jl:127-140): a known optimal value, when given, must be met as well
      const bool obj_ok = (st_.obj_true != st_.obj_true) || fabs(st_.obj_true - cost) <= st_.obj_true_tol;
      if (info[0] < st_.eps_abs + st_.eps_rel * info[2] && info[1] < st_.eps_abs + st_.eps_rel * info[3] && obj_ok) {
        status = COSMO_B200_SOLVED;
        break;
      }
    }
    if (st_.check_infeasibility > 0 && iter % st_.check_infeasibility == 0) {
      infeasibility_check_due = true;
    } else if (suggested(infeasibility_check_due)) {
      infeasibility_check_due = false;
      recover_mu(W_[prev_].p);
      sub_kernel<T><<<vgrid(m), kBlock, 0, stream_>>>(m, dy_.p, mu_.p, dy_.p);          // dy -= mu
      check_launch("sub_dy");
      sub_kernel<T><<<vgrid(n), kBlock, 0, stream_>>>(n, W_[cur_].p, W_[prev_].p, dx_.p);  // dx = w_x - w_prev_x
      check_launch("sub_dx");
      if (primal_infeasible()) { status = COSMO_B200_PRIMAL_INFEASIBLE; cost = INFINITY; break; }
      if (dual_infeasible()) { status = COSMO_B200_DUAL_INFEASIBLE; cost = -INFINITY; break; }
    }
    // the reference's clock starts before setup! (time_limit_start, solver.jl:119,349)
    if (st_.time_limit != 0 && (now_s() - iter_start) + setup_time_total > st_.time_limit) {
      recover_mu(W_[prev_].p);
      compute_residuals(W_[prev_].p, s_.p, mu_.p, false, info);
      status = COSMO_B200_TIME_LIMIT_REACHED;
      break;
    }
  }
  recover_mu(W_[prev_].p);  // solver.jl:167
  CUDA_TRY(cudaEventRecord(ev1_, stream_));
  sync();
  const double iter_time = now_s() - iter_start;
  float dev_ms = 0.f;
  CUDA_TRY(cudaEventElapsedTime(&dev_ms, ev0_, ev1_));
  if (iter + safeguarding_iter == st_.max_iter && status == COSMO_B200_UNDETERMINED) {  // solver.jl:173-176
    compute_residuals(W_[prev_].p, s_.p, mu_.p, false, info);
    status = COSMO_B200_MAX_ITER_REACHED;
  }
  if (persist_solves_ > 0) {   // inner-iteration statistics of the persistent CG kernel live on the device
    CUDA_TRY(cudaMemcpyAsync(h_isc_ + ISC_TOTAL, isc_.p + ISC_TOTAL, sizeof(int), cudaMemcpyDeviceToHost, stream_));
    sync();
    total_inner_ += h_isc_[ISC_TOTAL];
    total_mults_ += h_isc_[ISC_TOTAL] + persist_solves_;
  }
  // x = view(w_prev, 1:n): keep it for the next warm start and hand it out
  CUDA_TRY(cudaMemcpyAsync(xs_.p, W_[prev_].p, n * sizeof(T), cudaMemcpyDeviceToDevice, stream_));
  if (out) {
    if (out->x) download_vec(out->x, W_[prev_].p, n);
    if (out->s) download_vec(out->s, s_.p, m);
    if (out->mu) download_vec(out->mu, mu_.p, m);
    sync();
    out->obj_val = cost;
    out->iter = iter + safeguarding_iter;      // total_iter, solver.jl:195
    out->safeguarding_iter = safeguarding_iter;
    out->status = status;
    out->r_prim = info[0]; out->r_dual = info[1]; out->max_norm_prim = info[2]; out->max_norm_dual = info[3];
    out->rho = rho_;
    out->n_rho_updates = (int64_t)rho_updates_.size();
    if (out->rho_updates)
      for (int64_t i = 0; i < std::min<int64_t>(out->rho_updates_cap, out->n_rho_updates); ++i) out->rho_updates[i] = rho_updates_[i];
    out->setup_time = create_time_;   // the device part of setup!; the host adds its own
    out->iter_time = iter_time;
    out->iter_time_device = dev_ms * 1e-3;
    t_proj_.harvest();
    t_kkt_.harvest();
    out->proj_time = t_proj_.total_ms * 1e-3;   // device time of admm_z! (+ the fused rhs pass); 0 when the timers are off
    out->kkt_time = t_kkt_.total_ms * 1e-3;     // device time of the KKT solves incl. the fused ADMM tail
    out->res_time = res_time;
    out->kkt_inner_iterations = total_inner_;
    out->kkt_multiplications = total_mults_;
    out->kernel_launches = launches_ - launches0;
    out->solver_time = now_s() - t_start;
  }
  sync();
}

// ---- plugin-granularity entry points ---------------------------------------------
template <typename T>
void Engine<T>::project(const void* ws, void* s_out) {
  CUDA_TRY(cudaSetDevice(device_));
  // stage w_s in the s-part of a scratch operator variable of its own and put the slack iterate back afterwards: a
  // caller that projects between two solves must not disturb w_prev or s of the finished one
  if (proj_w_.n < (size_t)n_ + m_) { proj_w_.alloc((size_t)n_ + m_); proj_s_.alloc(std::max(m_, 1), false); }
  upload_vec(vec_m_, ws, m_);
  CUDA_TRY(cudaMemcpyAsync(proj_s_.p, s_.p, m_ * sizeof(T), cudaMemcpyDeviceToDevice, stream_));
  CUDA_TRY(cudaMemcpyAsync(proj_w_.p + n_, vec_m_.p, m_ * sizeof(T), cudaMemcpyDeviceToDevice, stream_));
  project_device(proj_w_.p, false, nullptr);
  download_vec(s_out, s_.p, m_);
  CUDA_TRY(cudaMemcpyAsync(s_.p, proj_s_.p, m_ * sizeof(T), cudaMemcpyDeviceToDevice, stream_));
  sync();
}

template <typename T>
void Engine<T>::kkt_solve(const void* rhs, void* sol, int64_t* inner) {
  CUDA_TRY(cudaSetDevice(device_));
  upload_vec(ls_, rhs, (size_t)n_ + m_);
  scale_kernel<T><<<vgrid(m_), kBlock, 0, stream_>>>(m_, rho_vec_.p, ls_.p + n_, t0_.p);
  check_launch("scale_x2");
  ensure_factor();
  kkt_core(false, nullptr, nullptr);
  download_vec(sol, xsol_.p, n_);
  download_vec(static_cast<T*>(sol) + n_, nu_.p, m_);
  sync();
  if (inner) {
    CUDA_TRY(cudaMemcpyAsync(h_isc_, isc_.p, 2 * sizeof(int), cudaMemcpyDeviceToHost, stream_));
    sync();
    *inner = st_.kkt_solver == COSMO_B200_KKT_DIRECT ? 0 : h_isc_[ISC_IT];
  }
}

template <typename T>
void Engine<T>::residuals(const void* x, const void* s, const void* mu, int ignore_scaling, double* out) {
  CUDA_TRY(cudaSetDevice(device_));
  upload_vec(dx_, x, n_);
  upload_vec(vec_m_, s, m_);
  upload_vec(dy_, mu, m_);
  compute_residuals(dx_.p, vec_m_.p, dy_.p, ignore_scaling != 0, out);
}

template <typename T>
void Engine<T>::spmv(int which, const void* x, void* y) {
  CUDA_TRY(cudaSetDevice(device_));
  if (which == 0) {
    upload_vec(dx_, x, n_);
    launch_spmv(A_, dx_.p, (const DevCsr<T>*)nullptr, (const T*)nullptr, m_, EpiStore<T>{nullptr, vec_m_.p}, red(SC_TMP0), "spmv_A");
    download_vec(y, vec_m_.p, m_);
  } else if (which == 1) {
    upload_vec(dy_, x, m_);
    launch_spmv(At_, dy_.p, (const DevCsr<T>*)nullptr, (const T*)nullptr, n_, EpiStore<T>{nullptr, vec_n_.p}, red(SC_TMP0), "spmv_At");
    download_vec(y, vec_n_.p, n_);
  } else if (which == 2) {
    upload_vec(dx_, x, n_);
    launch_spmv(P_, dx_.p, (const DevCsr<T>*)nullptr, (const T*)nullptr, n_, EpiStore<T>{nullptr, vec_n_.p}, red(SC_TMP0), "spmv_P");
    download_vec(y, vec_n_.p, n_);
  } else {
    throw EngineError{COSMO_B200_ERR_INVALID, "spmv: which must be 0 (A), 1 (A') or 2 (P)"};
  }
  sync();
}

template <typename T>
void Engine<T>::spmv_bench(int which, int reps, double* ms, double* bytes) {
  CUDA_TRY(cudaSetDevice(device_));
  if (reps < 1) reps = 1;
  auto one = [&]() {
    if (which == 0)
      launch_spmv(A_, xsol_.p, (const DevCsr<T>*)nullptr, (const T*)nullptr, m_, EpiScale<T>{nullptr, tm_.p, rho_vec_.p}, red(SC_TMP0), "spmv_A_scale");
    else if (which == 1)
      launch_spmv(At_, tm_.p, (const DevCsr<T>*)nullptr, (const T*)nullptr, n_, EpiStore<T>{nullptr, vec_n_.p}, red(SC_TMP0), "spmv_At");
    else if (which == 2)
      launch_spmv(P_, xsol_.p, (const DevCsr<T>*)nullptr, (const T*)nullptr, n_, EpiStore<T>{nullptr, vec_n_.p}, red(SC_TMP0), "spmv_P");
    else  // 3: the reduced-KKT operator stage 2 (A' and P rows + dot)
      kkt_op_stage2(nullptr, xsol_.p, tm_.p, cb_.p);
  };
  for (int i = 0; i < 3; ++i) one();
  CUDA_TRY(cudaEventRecord(ev0_, stream_));
  for (int i = 0; i < reps; ++i) one();
  CUDA_TRY(cudaEventRecord(ev1_, stream_));
  sync();
  float t = 0.f;
  CUDA_TRY(cudaEventElapsedTime(&t, ev0_, ev1_));
  *ms = (double)t / reps;
  if (which == 0) *bytes = A_.spmv_bytes() + sizeof(T) * (double)m_;       // + rho
  else if (which == 1) *bytes = At_.spmv_bytes();
  else if (which == 2) *bytes = P_.spmv_bytes();
  else *bytes = At_.spmv_bytes() + P_.spmv_bytes() - sizeof(T) * (double)n_;
}

template <typename T>
void Engine<T>::get_rho_vec(void* out) { download_vec(out, rho_vec_.p, m_); sync(); }
template <typename T>
void Engine<T>::psd_stats(int64_t* o) {
  o[0] = psd_.tc_projections; o[1] = psd_.tc_fallbacks; o[2] = psd_.tc_.last_steps; o[3] = psd_.tc_.last_checks;
  o[4] = psd_.sign_projections; o[5] = psd_.sign_fallbacks; o[6] = psd_.last_sweeps; o[7] = psd_.tc_.gemm.k;
}
template <typename T>
void Engine<T>::get_w(void* out) { download_vec(out, W_[cur_].p, (size_t)n_ + m_); sync(); }

}  // namespace cosmo

// ============================================================================
// C ABI
// ============================================================================
struct cosmo_b200_handle {
  cosmo::EngineBase* impl = nullptr;
  std::string err;
};

#define ABI_GUARD(h, body)                                                   \
  if (!(h) || !(h)->impl) return COSMO_B200_ERR_INVALID;                     \
  try { body; return COSMO_B200_OK; }                                        \
  catch (const cosmo::EngineError& e) { (h)->err = e.msg; return e.code; }   \
  catch (const cosmo::PsdError& e) { (h)->err = e.msg; return COSMO_B200_ERR_NUMERICAL; } \
  catch (const std::bad_alloc&) { (h)->err = "host allocation failed"; return COSMO_B200_ERR_ALLOC; } \
  catch (...) { (h)->err = "unknown error"; return COSMO_B200_ERR_INVALID; }

extern "C" {

int cosmo_b200_abi_version(void) { return COSMO_B200_ABI_VERSION; }

int cosmo_b200_default_settings(cosmo_b200_settings* s) {
  if (!s) return COSMO_B200_ERR_INVALID;
  memset(s, 0, sizeof(*s));
  s->rho = 0.1; s->sigma = 1e-6; s->alpha = 1.6;
  s->eps_abs = 1e-5; s->eps_rel = 1e-5; s->eps_prim_inf = 1e-4; s->eps_dual_inf = 1e-4;
  s->max_iter = 5000; s->check_termination = 25; s->check_infeasibility = 40;
  s->scaling = 10; s->adaptive_rho = 1; s->adaptive_rho_interval = 40; s->kkt_solver = COSMO_B200_KKT_CG;
  s->adaptive_rho_fraction = 0.4; s->setup_time = 0.0; s->MAX_SCALING = 1e4;
  s->obj_true = NAN; s->obj_true_tol = 1e-3;
  s->adaptive_rho_tolerance = 5.0; s->adaptive_rho_max_adaptions = INT64_MAX;
  s->RHO_MIN = 1e-6; s->RHO_MAX = 1e6; s->RHO_TOL = 1e-4; s->RHO_EQ_OVER_RHO_INEQ = 1e3;
  s->COSMO_INFTY = 1e20; s->MIN_SCALING = 1e-4;
  s->time_limit = 0.0; s->tol_constant = 1.0; s->tol_exponent = 1.5;
  s->verbose = 0; s->psd_max_sweeps = 30;
  s->accelerator = COSMO_B200_ACC_EMPTY; s->accelerator_mem = 15; s->accelerator_min_mem = 3;
  s->safeguard = 1; s->safeguard_tol = 2.0;
  return COSMO_B200_OK;
}

int cosmo_b200_create(cosmo_b200_handle** out, const cosmo_b200_problem* prob, const cosmo_b200_settings* settings) {
  if (!out || !prob || !settings) { cosmo::g_create_error = "null argument"; return COSMO_B200_ERR_INVALID; }
  *out = nullptr;
  try {
    cosmo::EngineBase* impl = nullptr;
    if (prob->dtype == COSMO_B200_F64) impl = new cosmo::Engine<double>(*prob, *settings);
    else if (prob->dtype == COSMO_B200_F32) impl = new cosmo::Engine<float>(*prob, *settings);
    else throw cosmo::EngineError{COSMO_B200_ERR_UNSUPPORTED, "dtype must be Float64 or Float32 (BigFloat models fall back to the host loop)"};
    cosmo_b200_handle* h = new cosmo_b200_handle();
    h->impl = impl;
    *out = h;
    return COSMO_B200_OK;
  } catch (const cosmo::EngineError& e) { cosmo::g_create_error = e.msg; return e.code; }
  catch (const cosmo::PsdError& e) { cosmo::g_create_error = e.msg; return COSMO_B200_ERR_CUDA; }
  catch (const std::bad_alloc&) { cosmo::g_create_error = "host allocation failed"; return COSMO_B200_ERR_ALLOC; }
  catch (...) { cosmo::g_create_error = "unknown error"; return COSMO_B200_ERR_INVALID; }
}

void cosmo_b200_destroy(cosmo_b200_handle* h) {
  if (!h) return;
  delete h->impl;
  delete h;
}

const char* cosmo_b200_last_error(const cosmo_b200_handle* h) {
  return h ? h->err.c_str() : cosmo::g_create_error.c_str();
}

int cosmo_b200_update_settings(cosmo_b200_handle* h, const cosmo_b200_settings* s) {
  if (!s) return COSMO_B200_ERR_INVALID;
  ABI_GUARD(h, h->impl->update_settings(*s));
}
int cosmo_b200_warm_start(cosmo_b200_handle* h, const void* x, const void* s, const void* mu) { ABI_GUARD(h, h->impl->warm_start(x, s, mu)); }
int cosmo_b200_update_qb(cosmo_b200_handle* h, const void* q, const void* b) { ABI_GUARD(h, h->impl->update_qb(q, b)); }
int cosmo_b200_update_rho(cosmo_b200_handle* h, const void* rho_vec, double rho) { ABI_GUARD(h, h->impl->update_rho(rho_vec, rho)); }
int cosmo_b200_reset(cosmo_b200_handle* h) { ABI_GUARD(h, h->impl->reset()); }
int cosmo_b200_solve(cosmo_b200_handle* h, cosmo_b200_result* out) { ABI_GUARD(h, h->impl->solve(out)); }
int cosmo_b200_project(cosmo_b200_handle* h, const void* w_s, void* s_out) {
  if (!w_s || !s_out) return COSMO_B200_ERR_INVALID;
  ABI_GUARD(h, h->impl->project(w_s, s_out));
}
int cosmo_b200_kkt_solve(cosmo_b200_handle* h, const void* rhs, void* sol, int64_t* inner) {
  if (!rhs || !sol) return COSMO_B200_ERR_INVALID;
  ABI_GUARD(h, h->impl->kkt_solve(rhs, sol, inner));
}
int cosmo_b200_residuals(cosmo_b200_handle* h, const void* x, const void* s, const void* mu, int32_t ignore_scaling, double out[5]) {
  if (!x || !s || !mu || !out) return COSMO_B200_ERR_INVALID;
  ABI_GUARD(h, h->impl->residuals(x, s, mu, ignore_scaling, out));
}
int cosmo_b200_spmv(cosmo_b200_handle* h, int32_t which, const void* x, void* y) {
  if (!x || !y) return COSMO_B200_ERR_INVALID;
  ABI_GUARD(h, h->impl->spmv(which, x, y));
}
int cosmo_b200_spmv_bench(cosmo_b200_handle* h, int32_t which, int32_t reps, double* ms, double* bytes) {
  if (!ms || !bytes) return COSMO_B200_ERR_INVALID;
  ABI_GUARD(h, h->impl->spmv_bench(which, reps, ms, bytes));
}
int cosmo_b200_get_rho_vec(cosmo_b200_handle* h, void* out) {
  if (!out) return COSMO_B200_ERR_INVALID;
  ABI_GUARD(h, h->impl->get_rho_vec(out));
}
int cosmo_b200_get_w(cosmo_b200_handle* h, void* out) {
  if (!out) return COSMO_B200_ERR_INVALID;
  ABI_GUARD(h, h->impl->get_w(out));
}
int cosmo_b200_psd_stats(cosmo_b200_handle* h, int64_t out[8]) {
  if (!out) return COSMO_B200_ERR_INVALID;
  ABI_GUARD(h, h->impl->psd_stats(out));
}
int cosmo_b200_get_scaling(cosmo_b200_handle* h, void* D, void* E, double* c) {
  ABI_GUARD(h, h->impl->get_scaling(D, E, c));
}
int cosmo_b200_kkt_factor_stats(cosmo_b200_handle* h, int64_t* factorizations, double seconds[2]) {
  if (!factorizations || !seconds) return COSMO_B200_ERR_INVALID;
  ABI_GUARD(h, h->impl->kkt_factor_stats(factorizations, seconds));
}
int cosmo_b200_comm_unique_id(void* id128) {
  if (!id128) return COSMO_B200_ERR_INVALID;
  std::string e;
  if (!cosmo::g_nccl.load(e)) { cosmo::g_create_error = e; return COSMO_B200_ERR_NCCL; }
  cosmo::NcclUniqueId id;
  if (cosmo::g_nccl.GetUniqueId(&id) != 0) { cosmo::g_create_error = "ncclGetUniqueId failed"; return COSMO_B200_ERR_NCCL; }
  memcpy(id128, &id, sizeof(id));
  return COSMO_B200_OK;
}
int cosmo_b200_comm_init(cosmo_b200_handle* h, int32_t nranks, int32_t rank, const void* id128) {
  if (nranks > 1 && !id128) return COSMO_B200_ERR_INVALID;
  ABI_GUARD(h, h->impl->comm_init(nranks, rank, id128));
}
int cosmo_b200_comm_p2p_export(cosmo_b200_handle* h, void* blob128) {
  if (!blob128) return COSMO_B200_ERR_INVALID;
  ABI_GUARD(h, h->impl->p2p_export(blob128));
}
int cosmo_b200_comm_p2p_attach(cosmo_b200_handle* h, const void* blobs, int32_t nranks) {
  if (!blobs) return COSMO_B200_ERR_INVALID;
  ABI_GUARD(h, h->impl->p2p_attach(blobs, nranks));
}

// ---- diagnostics of the tensor-core PSD path (tc_gemm.cuh, psd_tc.cuh) ----------------------------------------
// C = A B for symmetric commuting N x N fp64 matrices (column-major, ld = N) through the int8-sliced tcgen05 product.
int cosmo_b200_tc_gemm_test(int32_t N, int32_t k, int32_t kstep, int32_t gpb, const double* A, const double* B, double* C,
                            int32_t reps, double* ms_per_product, double* frob2) {
  if (N <= 0 || !A || !B || !C) return COSMO_B200_ERR_INVALID;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cosmo::g_create_error = "no CUDA device"; return COSMO_B200_ERR_CUDA; }
  cudaStream_t st;
  if (cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) != cudaSuccess) return COSMO_B200_ERR_CUDA;
  int rc = COSMO_B200_OK;
  double *A_d = nullptr, *B_d = nullptr, *C_d = nullptr, *coef_d = nullptr, *part_d = nullptr;
  {
    cosmo::tc::OzakiGemm<double> g;
    cosmo::tc::Sliced sa, sb;
    const size_t nn = (size_t)N * N;
    const double coef[3] = {1.0, 0.0, 0.0};
    (void)gpb;
    bool ok = g.configure(k, kstep > 0 ? kstep : (k == 8 ? 10 : (k == 7 ? 7 : k + 2)), st) && g.set_shape(N, st);
    ok = ok && cudaMalloc(&A_d, nn * 8) == cudaSuccess && cudaMalloc(&B_d, nn * 8) == cudaSuccess && cudaMalloc(&C_d, nn * 8) == cudaSuccess &&
         cudaMalloc(&coef_d, 3 * 8) == cudaSuccess && cudaMalloc(&part_d, (size_t)2 * (g.ntiles + 1) * 8) == cudaSuccess;
    ok = ok && sa.ensure(g.Np) && sb.ensure(g.Np) && sa.clear(g.Np, st) && sb.clear(g.Np, st);
    ok = ok && cudaMemcpyAsync(A_d, A, nn * 8, cudaMemcpyHostToDevice, st) == cudaSuccess &&
         cudaMemcpyAsync(B_d, B, nn * 8, cudaMemcpyHostToDevice, st) == cudaSuccess &&
         cudaMemcpyAsync(coef_d, coef, 3 * 8, cudaMemcpyHostToDevice, st) == cudaSuccess &&
         cudaMemsetAsync(C_d, 0, nn * 8, st) == cudaSuccess;
    ok = ok && g.slice(A_d, sa, st) && g.slice(B_d, sb, st);
    ok = ok && g.gemm(sa, sb, C_d, nullptr, nullptr, 1, coef_d, part_d, st);
    ok = ok && cudaStreamSynchronize(st) == cudaSuccess;
    if (ok && reps > 0 && ms_per_product) {
      cudaEvent_t e0, e1;
      cudaEventCreate(&e0); cudaEventCreate(&e1);
      cudaEventRecord(e0, st);
      for (int r = 0; r < reps && ok; ++r) ok = g.gemm(sa, sb, C_d, nullptr, nullptr, 1, coef_d, part_d, st);
      cudaEventRecord(e1, st);
      ok = ok && cudaEventSynchronize(e1) == cudaSuccess;
      float ms = 0.f;
      cudaEventElapsedTime(&ms, e0, e1);
      *ms_per_product = ms / reps;
      cudaEventDestroy(e0); cudaEventDestroy(e1);
    }
    ok = ok && cudaMemcpyAsync(C, C_d, nn * 8, cudaMemcpyDeviceToHost, st) == cudaSuccess;
    if (ok && frob2) {
      std::vector<double> part(2 * g.ntiles);
      ok = cudaMemcpyAsync(part.data(), part_d, part.size() * 8, cudaMemcpyDeviceToHost, st) == cudaSuccess &&
           cudaStreamSynchronize(st) == cudaSuccess;
      frob2[0] = frob2[1] = 0.0;
      for (int i = 0; i < g.ntiles; ++i) { frob2[0] += part[2 * i]; frob2[1] += part[2 * i + 1]; }
    }
    ok = ok && cudaStreamSynchronize(st) == cudaSuccess;
    if (!ok) {
      cudaError_t e = cudaGetLastError();
      cosmo::g_create_error = "tc_gemm_test: " + (g.err.empty() ? std::string(cudaGetErrorString(e)) : g.err);
      rc = COSMO_B200_ERR_CUDA;
    }
  }
  cudaFree(A_d); cudaFree(B_d); cudaFree(C_d); cudaFree(coef_d); cudaFree(part_d);
  cudaStreamDestroy(st);
  return rc;
}

// ---- symbolic analysis of the full KKT matrix (ldl_symbolic.h); host only ---------------------------------------------
static void kkt_pattern(const cosmo_b200_csc& M, int64_t nrows, int64_t ncols, int base, const char* name,
                        std::vector<int64_t>& colptr, std::vector<int64_t>& row) {
  const std::string nm(name);
  if (M.nrows != nrows || M.ncols != ncols) throw cosmo::EngineError{COSMO_B200_ERR_INVALID, nm + " has the wrong shape"};
  colptr.assign(ncols + 1, 0);
  if (ncols > 0 && !M.colptr) throw cosmo::EngineError{COSMO_B200_ERR_INVALID, nm + ": null colptr"};
  for (int64_t j = 0; j <= ncols; ++j) {
    const int64_t v = ncols ? M.colptr[j] - base : 0;
    if (v < 0 || (j > 0 && v < colptr[j - 1])) throw cosmo::EngineError{COSMO_B200_ERR_INVALID, nm + ": colptr not monotone"};
    colptr[j] = v;
  }
  const int64_t nnz = colptr[ncols];
  if (nnz > 0 && !M.rowval) throw cosmo::EngineError{COSMO_B200_ERR_INVALID, nm + ": null rowval"};
  row.resize(nnz);
  std::vector<int64_t> seen(nrows, -1);
  for (int64_t j = 0; j < ncols; ++j)
    for (int64_t k = colptr[j]; k < colptr[j + 1]; ++k) {
      const int64_t i = M.rowval[k] - base;
      if (i < 0 || i >= nrows) throw cosmo::EngineError{COSMO_B200_ERR_INVALID, nm + ": row index out of range"};
      if (seen[i] == j) throw cosmo::EngineError{COSMO_B200_ERR_INVALID, nm + " has duplicate entries"};
      seen[i] = j;
      row[k] = i;
    }
}

int cosmo_b200_kkt_symbolic(const cosmo_b200_problem* prob, int64_t* perm, int64_t info[8]) {
  if (!prob || !info) { cosmo::g_create_error = "null argument"; return COSMO_B200_ERR_INVALID; }
  try {
    if (prob->n < 0 || prob->m < 0 || (prob->index_base != 0 && prob->index_base != 1))
      throw cosmo::EngineError{COSMO_B200_ERR_INVALID, "bad dimensions or index base"};
    std::vector<int64_t> pc, pr, ac, ar;
    kkt_pattern(prob->P, prob->n, prob->n, prob->index_base, "P", pc, pr);
    kkt_pattern(prob->A, prob->m, prob->n, prob->index_base, "A", ac, ar);
    const cosmo::ldl::Symbolic S = cosmo::ldl::analyse(prob->n, prob->m, pc, pr, ac, ar);
    if (perm) std::copy(S.perm.begin(), S.perm.end(), perm);
    const int64_t out[8] = {S.nnz_L, (int64_t)S.sn_first.size() - 1, S.height, S.widest, S.largest_front,
                            S.factor_bytes, S.workspace_bytes, S.dense};
    std::copy(out, out + 8, info);
    return COSMO_B200_OK;
  } catch (const cosmo::EngineError& e) { cosmo::g_create_error = e.msg; return e.code; }
  catch (const std::bad_alloc&) { cosmo::g_create_error = "host allocation failed"; return COSMO_B200_ERR_ALLOC; }
  catch (...) { cosmo::g_create_error = "unknown error"; return COSMO_B200_ERR_INVALID; }
}

}  // extern "C"
