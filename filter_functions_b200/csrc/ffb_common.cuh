// Shared declarations of libffb200: context, error plumbing, device-memory pool, complex helpers.
#pragma once

#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>
#include <deque>
#include <functional>
#include <map>
#include <string>
#include <tuple>
#include <vector>

#include "../../include/ffb200.h"

// ------------------------------------------------------------------------------------------------
// peer group: the GPUs of one node, one process each, exchanging through NVLink peer memory
// ------------------------------------------------------------------------------------------------
constexpr int FFB_MAX_PEERS = 16;
constexpr int FFB_PEER_SLOTS = 1024;  // doubles one all-reduce can carry

// Kernel-side view of the group (passed by value).  world <= 1: no exchange.
struct PeerReduce {
  unsigned long long window[FFB_MAX_PEERS];  // every rank's exchange window as mapped in THIS process
  int rank = 0, world = 1;
  unsigned seq = 0;          // flag value of this collective (never 0, same on all ranks)
  unsigned timeout_ms = 0;
  int* error = nullptr;      // device flag, set when a peer did not arrive in time
};

struct ffb_comm {
  int rank = 0, world = 1;
  bool connected = false;
  void* window = nullptr;                 // mine (cudaMalloc, exported through CUDA IPC)
  void* peer[FFB_MAX_PEERS] = {};         // peers' windows (peer[rank] == window)
  unsigned seq = 0;                       // collectives issued so far
  bool reduce_infidelity = false;         // all-reduce every infidelity integral before it is returned
  unsigned timeout_ms = 20000;
  int* err_dev = nullptr;
  int* err_host = nullptr;
  // symmetric data window for the all-gather of frequency blocks (grow-only, re-exported on growth)
  void* data = nullptr;
  size_t data_bytes = 0;
  void* peer_data[FFB_MAX_PEERS] = {};
};

// ------------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------------
struct ffb_ctx {
  ffb_comm comm;
  int device = 0;
  int sm_count = 148;
  int cc_major = 0, cc_minor = 0;
  size_t total_mem = 0;
  cudaStream_t own_stream = nullptr;
  cudaStream_t stream = nullptr;  // the stream work is enqueued on (own or external)
  std::string err;
  int64_t launches = 0;
  // 256-entry table of (sin, cos)(k pi / 128) for the table-driven sincos of the control-matrix kernels
  double* trig_table = nullptr;
  // bands and proxies of the last FFB_DISPATCH_LOG_MAX banded control-matrix blocks, written by the plan
  // kernel; ffb_dispatch_log reads them into the records
  int* band_counts = nullptr;
  unsigned band_counts_next = 0;
  // second stream for bulk host<->device copies that overlap kernels (the pulse pipeline, the control
  // matrix, ffb_concatenate_pulses); ordered against `stream` with the two events
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t copy_ev[2] = {nullptr, nullptr};
  // page-locked staging block: the small host inputs of a call are packed here and uploaded by ONE copy
  void* stage_host = nullptr;
  size_t stage_bytes = 0;
  // ... and its twin for small RESULTS that go to ordinary (pageable) caller memory: one device-to-host
  // copy into this block, then plain memcpy to the caller's arrays (a pageable destination costs one
  // blocking driver copy per array otherwise)
  void* stage_out = nullptr;
  size_t stage_out_bytes = 0;
  // eigensolver convergence: a device counter the Jacobi kernels bump for every matrix that did not
  // converge (allocated and zeroed once), and its page-locked host mirror; the synchronous entry points
  // fetch it with their last copies and return FFB_ENOTCONV (numpy.linalg.eigh raises LinAlgError)
  int* conv_dev = nullptr;
  int* conv_host = nullptr;
  // partial sums + ticket counters of the chunked infidelity integral (allocated and zeroed once)
  void* infid_scratch = nullptr;
  // launch bookkeeping that would otherwise cost a driver call per launch: the dynamic shared memory
  // limit already set for a kernel (grow-only) and occupancy query results
  std::map<const void*, size_t> func_smem;
  std::map<std::tuple<const void*, int, size_t>, int> occupancy_cache;

  // grow-only caching pool: freed blocks are kept and handed out again (best fit)
  std::multimap<size_t, void*> free_blocks;
  std::map<void*, size_t> live_blocks;
  size_t pool_bytes = 0;

  // page-locked host blocks handed out by ffb_host_alloc (same caching scheme as the device pool)
  std::multimap<size_t, void*> host_free_blocks;
  std::map<void*, size_t> host_live_blocks;
  size_t host_pool_bytes = 0;

  // device-resident shadows of result arrays (SURVEY.md 8b "dev_handle"): when a host-pointer entry
  // point has written results into page-locked blocks of this context's own pool, the device copy they
  // were downloaded from can be kept, keyed by the host address range it mirrors.  A later call that
  // is handed a host pointer inside such a range reads the device copy instead of uploading the
  // bytes again (ff.infidelity with another spectrum, decay amplitudes, concatenation of cached gates).
  // Dropped when the host block goes back to the pool (the NumPy array was garbage collected), when a
  // call writes into the range, or -- oldest first -- when the shadows exceed `shadow_limit` bytes.
  struct Shadow {
    void* dev = nullptr;
    size_t bytes = 0;                                  // mirrors host [key, key + bytes)
    std::vector<std::pair<size_t, size_t>> valid;      // (offset, length) of the results inside
    uint64_t stamp = 0;
  };
  std::map<char*, Shadow> shadows;
  size_t shadow_bytes = 0, shadow_limit = 0;
  uint64_t shadow_clock = 0;
  bool shadow_next = false;  // keep the results of the next host-pointer call (one-shot)
  int64_t shadow_hits = 0;
  size_t shadow_hit_bytes = 0;

  // timing of the dominant kernel
  bool timing = false;
  double timed_ms = 0.0;
  int64_t timed_launches = 0;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> pending_events;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> event_pool;

  // what the control-matrix calls launched, per frequency block (ffb_dispatch_log)
  std::deque<ffb_dispatch_record> dispatch_log;
  // what each diagonalisation launched (ffb_diag_dispatch_log)
  std::deque<ffb_dispatch_record> diag_dispatch_log;
};

int ffb_fail(ffb_ctx* ctx, int code, const char* fmt, ...);
// FFB_TRACE set and nonzero (read once): host-side timelines and dispatch lines on stderr
bool ffb_trace();

#define FFB_CUDA(ctx, expr)                                                                    \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess)                                                                     \
      return ffb_fail((ctx), _e == cudaErrorMemoryAllocation ? FFB_ENOMEM : FFB_ECUDA,         \
                      "%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e));   \
  } while (0)

#define FFB_TRY(expr)          \
  do {                         \
    int _rc = (expr);          \
    if (_rc != FFB_OK) return _rc; \
  } while (0)

#define FFB_REQUIRE(ctx, cond, ...)                              \
  do {                                                           \
    if (!(cond)) return ffb_fail((ctx), FFB_EINVAL, __VA_ARGS__); \
  } while (0)

// the kernels hold a d x d matrix per warp / thread in shared memory and registers: d <= 32
#define FFB_MAX_DIM 32
#define FFB_CHECK_DIM(ctx, d)                                                                        \
  FFB_REQUIRE((ctx), (d) <= FFB_MAX_DIM, "Hilbert-space dimension d = %d exceeds the supported maximum " \
              "of %d of filter_functions_b200 (README: limits)", (d), FFB_MAX_DIM)

// counts the launch and checks the launch error
#define FFB_LAUNCHED(ctx)         \
  do {                            \
    (ctx)->launches++;            \
    FFB_CUDA((ctx), cudaGetLastError()); \
  } while (0)

int ffb_pool_alloc(ffb_ctx* ctx, size_t bytes, void** ptr);
void ffb_pool_release(ffb_ctx* ctx, void* ptr);

// RAII handle on pool memory; returned to the pool when it goes out of scope. Stream-ordered use is
// safe because everything in a context runs on one stream.
struct DevBuf {
  ffb_ctx* ctx = nullptr;
  void* p = nullptr;
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { reset(); }
  int alloc(ffb_ctx* c, size_t bytes) {
    reset();
    ctx = c;
    return ffb_pool_alloc(c, bytes ? bytes : 8, &p);
  }
  void reset() {
    if (p) ffb_pool_release(ctx, p);
    p = nullptr;
  }
  void* detach() {  // ownership moves to the caller (a shadow)
    void* q = p;
    p = nullptr;
    return q;
  }
  template <typename T>
  T* as() const { return static_cast<T*>(p); }
};

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) / cudaOccupancyMaxActiveBlocksPerMultiprocessor,
// remembered per context (small pulses are bound by the number of driver calls per library call)
int ffb_func_smem_impl(ffb_ctx* ctx, const void* func, size_t smem);
int ffb_occupancy_impl(ffb_ctx* ctx, const void* func, int block_threads, size_t smem, int* blocks);
template <typename K>
int ffb_func_smem(ffb_ctx* ctx, K kern, size_t smem) {
  return ffb_func_smem_impl(ctx, reinterpret_cast<const void*>(kern), smem);
}
template <typename K>
int ffb_occupancy(ffb_ctx* ctx, K kern, int block_threads, size_t smem, int* blocks) {
  return ffb_occupancy_impl(ctx, reinterpret_cast<const void*>(kern), block_threads, smem, blocks);
}
int ffb_h2d(ffb_ctx* ctx, void* dst, const void* src, size_t bytes);
// device shadows of result arrays (ffb_api.cu)
const void* ffb_shadow_lookup(ffb_ctx* ctx, const void* host, size_t bytes);
void ffb_shadow_drop_range(ffb_ctx* ctx, const void* host, size_t bytes);
// `buf` mirrors host [host_lo, host_lo + bytes); `valid` lists the results inside.  Takes the buffer out
// of `buf` if the shadow is kept (host range inside one live block of the host pool, size limits).
bool ffb_shadow_retain(ffb_ctx* ctx, DevBuf& buf, void* host_lo, size_t bytes,
                       const std::vector<std::pair<size_t, size_t>>& valid);
// convergence counter of the eigensolver: device pointer (created on first use); enqueue its download;
// after a stream synchronisation: FFB_ENOTCONV (and reset) if any matrix failed to converge
int ffb_conv_counter(ffb_ctx* ctx, int** dev);
int ffb_conv_fetch(ffb_ctx* ctx);
int ffb_conv_check(ffb_ctx* ctx);
int ffb_d2h(ffb_ctx* ctx, void* dst, const void* src, size_t bytes);

// timing hooks around the dominant kernel
int ffb_time_begin(ffb_ctx* ctx, int* slot);
int ffb_time_end(ffb_ctx* ctx, int slot);

// ------------------------------------------------------------------------------------------------
// internal device-pointer pipeline stages (implemented in the .cu files, all asynchronous)
// ------------------------------------------------------------------------------------------------
int ffbi_diagonalize(ffb_ctx* ctx, int G, int d, int n_cops, const double* c_opers,
                     const double* c_coeffs, const double* dt, double* eigvals, double* eigvecs,
                     double* propagators);
// Optional blocking of the frequency axis of the control-matrix pipeline: the omega-independent
// prologue runs once, then main kernel + finalize per block of frequencies; after the kernels of a
// block are enqueued `after_block(w0, w1)` is called, which lets the caller queue the download of the
// finished block (and its filter function) while the next block is computed.
struct FreqBlocks {
  int n_blocks = 1;
  std::function<int(int, int)> after_block;
};
int ffbi_control_matrix(ffb_ctx* ctx, int G, int d, int n_nops, int n_basis, int n_omega,
                        const double* eigvals, const double* eigvecs, const double* propagators,
                        const double* omega, const double* basis, const double* n_opers,
                        const double* n_coeffs, const double* dt, const double* t, int herm_flags,
                        double* out, const FreqBlocks* blocks = nullptr);
int ffbi_filter_function(ffb_ctx* ctx, int P, int n_nops, int n_basis, int n_omega,
                         const double* B, int generalized, double* F);
// same for a block of n_omega frequencies inside arrays whose rows are `ld` frequencies long
int ffbi_filter_function_ld(ffb_ctx* ctx, int P, int n_nops, int n_basis, int n_omega, size_t ld,
                            const double* B, double* F);
int ffbi_from_atomic(ffb_ctx* ctx, int P, int n_nops, int n_basis, int n_omega,
                     const double* phases, const double* B_atomic, const double* Q, int q_is_complex,
                     int correlations, double* out);
int ffbi_from_atomic_rows(ffb_ctx* ctx, int P, int n_nops, int j0, int jn, int n_basis, int n_omega,
                          const double* phases, const double* B_atomic, const double* Q,
                          int q_is_complex, int correlations, double* out);
int ffbi_from_atomic_dmma(ffb_ctx* ctx, int P, int n_nops, int n_rows, int n_basis, int n_omega,
                          const double* phases, const double* B_atomic, const double* Q,
                          int correlations, double* out);
int ffbi_infidelity(ffb_ctx* ctx, int n_lead, int n_nops, int n_sel, const int* idx_dev,
                    int n_omega, const double* F, const double* spectrum, int spectrum_ndim,
                    int spectrum_is_complex, const double* omega, int d, double* out);
int ffbi_decay_amplitudes(ffb_ctx* ctx, int P, int n_nops, int n_sel, const int* idx_dev,
                          int n_basis, int n_omega, const double* B, const double* spectrum,
                          int spectrum_ndim, int spectrum_is_complex, const double* omega,
                          double* out);
int ffbi_concatenate_many(ffb_ctx* ctx, int n_seq, int L, int d, int n_nops, int n_basis,
                          int n_omega, const int* idx, const double* lib_B, const double* lib_phase,
                          const double* lib_liouville, const double* lib_U, double* U_total,
                          double* out_B, double* out_F);
int ffbi_control_matrix_intermediates(ffb_ctx* ctx, int G, int d, int n_nops, int n_basis,
                                      int n_omega, const double* eigvals, const double* eigvecs,
                                      const double* propagators, const double* omega,
                                      const double* basis, const double* n_opers,
                                      const double* n_coeffs, const double* dt, const double* t,
                                      double* out, double* n_opers_transformed,
                                      double* eigvecs_propagated, double* basis_transformed,
                                      double* phase_factors, double* first_order_integral,
                                      double* step, double* cumulative);
int ffbi_infidelity_derivative(ffb_ctx* ctx, int G, int d, int n_nops, int n_basis, int n_omega,
                               const double* eigvals, const double* eigvecs,
                               const double* propagators, const double* omega, const double* basis,
                               const double* n_opers, const double* n_coeffs, const double* dt,
                               const double* t, const double* c_opers, const double* control_matrix,
                               int n_ctrl, const int* ctrl_idx, int n_sel, const int* sel_idx,
                               const double* spectrum, int spectrum_ndim,
                               const double* n_coeffs_deps, int norm_d, double* out);
int ffbi_control_matrix_periodic(ffb_ctx* ctx, int n_nops, int n_basis, int n_omega, int repeats,
                                 const double* phases, const double* B, const double* L,
                                 int l_is_complex, double* out);
int ffbi_liouville(ffb_ctx* ctx, int n, int d, int n_basis, const double* U, const double* basis,
                   double* out);
int ffbi_cexp(ffb_ctx* ctx, int n, const double* x, double scale, double* out);
int ffbi_cexpm1(ffb_ctx* ctx, int n, const double* x, double* out);
int ffbi_fp64_peak(ffb_ctx* ctx, double* dfma, double* dmma);
// peer group (ffb_comm.cu): the kernel-side descriptor of the NEXT collective (advances the sequence
// number); in-place all-reduce of n doubles in device memory; release of everything the group holds
PeerReduce ffbi_peer_next(ffb_ctx* ctx);
int ffbi_allreduce_sum(ffb_ctx* ctx, double* data_dev, int n);
void ffbi_comm_release(ffb_ctx* ctx);
int ffbi_comm_fetch_error(ffb_ctx* ctx);   // enqueue the download of the time-out flag
int ffbi_comm_check_error(ffb_ctx* ctx);   // after a stream synchronisation

// ------------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------------
struct cplx {
  double re, im;
};

__host__ __device__ __forceinline__ cplx cmul(cplx a, cplx b) {
  return {a.re * b.re - a.im * b.im, a.re * b.im + a.im * b.re};
}
__host__ __device__ __forceinline__ cplx cmulc(cplx a, cplx b) {  // a * conj(b)
  return {a.re * b.re + a.im * b.im, a.im * b.re - a.re * b.im};
}
__host__ __device__ __forceinline__ cplx cadd(cplx a, cplx b) { return {a.re + b.re, a.im + b.im}; }
__host__ __device__ __forceinline__ cplx cconj(cplx a) { return {a.re, -a.im}; }

static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
static inline size_t ceil_div_sz(size_t a, size_t b) { return (a + b - 1) / b; }
