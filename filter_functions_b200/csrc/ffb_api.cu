// C ABI of libffb200 (include/ffb200.h): context, memory pool, host-pointer wrappers.
#include <algorithm>
#include <chrono>
#include <cstdarg>
#include <cstdlib>
#include <cstring>

#include "ffb_common.cuh"

// ------------------------------------------------------------------------------------------------
// error plumbing / pool / staging
// ------------------------------------------------------------------------------------------------
static std::string g_init_error;

int ffb_fail(ffb_ctx* ctx, int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (ctx) ctx->err = buf;
  else g_init_error = buf;
  return code;
}

bool ffb_trace() {
  static const bool on = getenv("FFB_TRACE") && atoi(getenv("FFB_TRACE")) != 0;
  return on;
}

int ffb_pool_alloc(ffb_ctx* ctx, size_t bytes, void** ptr) {
  bytes = (bytes + 511) & ~(size_t)511;
  auto it = ctx->free_blocks.lower_bound(bytes);
  // accept a cached block if it wastes at most 2x
  if (it != ctx->free_blocks.end() && it->first <= 2 * bytes + (1 << 20)) {
    *ptr = it->second;
    ctx->live_blocks[*ptr] = it->first;
    ctx->free_blocks.erase(it);
    return FFB_OK;
  }
  cudaError_t e = cudaMalloc(ptr, bytes);
  if (e != cudaSuccess) {
    // give cached blocks back to the driver and retry once
    (void)cudaGetLastError();
    cudaStreamSynchronize(ctx->stream);
    for (auto& kv : ctx->free_blocks) {
      cudaFree(kv.second);
      ctx->pool_bytes -= kv.first;
    }
    ctx->free_blocks.clear();
    e = cudaMalloc(ptr, bytes);
    if (e != cudaSuccess) {
      (void)cudaGetLastError();
      return ffb_fail(ctx, FFB_ENOMEM, "device allocation of %zu bytes failed: %s", bytes,
                      cudaGetErrorString(e));
    }
  }
  ctx->pool_bytes += bytes;
  ctx->live_blocks[*ptr] = bytes;
  return FFB_OK;
}

void ffb_pool_release(ffb_ctx* ctx, void* ptr) {
  auto it = ctx->live_blocks.find(ptr);
  if (it == ctx->live_blocks.end()) return;
  ctx->free_blocks.emplace(it->second, ptr);
  ctx->live_blocks.erase(it);
}

int ffb_h2d(ffb_ctx* ctx, void* dst, const void* src, size_t bytes) {
  if (bytes == 0) return FFB_OK;
  FFB_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
  return FFB_OK;
}

int ffb_d2h(ffb_ctx* ctx, void* dst, const void* src, size_t bytes) {
  if (bytes == 0) return FFB_OK;
  ffb_shadow_drop_range(ctx, dst, bytes);  // whatever mirrored these host bytes is stale now
  FFB_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  return FFB_OK;
}

// ------------------------------------------------------------------------------------------------
// device shadows of result arrays
// ------------------------------------------------------------------------------------------------
static constexpr size_t SHADOW_MIN_BYTES = (size_t)64 << 10;  // below this an upload costs nothing

static void shadow_erase(ffb_ctx* ctx, std::map<char*, ffb_ctx::Shadow>::iterator it) {
  ffb_pool_release(ctx, it->second.dev);
  ctx->shadow_bytes -= it->second.bytes;
  ctx->shadows.erase(it);
}

const void* ffb_shadow_lookup(ffb_ctx* ctx, const void* host, size_t bytes) {
  if (ctx->shadows.empty() || !host || !bytes) return nullptr;
  char* h = static_cast<char*>(const_cast<void*>(host));
  auto it = ctx->shadows.upper_bound(h);
  if (it == ctx->shadows.begin()) return nullptr;
  --it;
  if (h + bytes > it->first + it->second.bytes) return nullptr;
  const size_t off = (size_t)(h - it->first);
  for (const auto& v : it->second.valid) {
    if (off >= v.first && off + bytes <= v.first + v.second) {
      it->second.stamp = ++ctx->shadow_clock;
      ctx->shadow_hits++;
      ctx->shadow_hit_bytes += bytes;
      return static_cast<char*>(it->second.dev) + off;
    }
  }
  return nullptr;
}

void ffb_shadow_drop_range(ffb_ctx* ctx, const void* host, size_t bytes) {
  if (ctx->shadows.empty() || !host) return;
  char* lo = static_cast<char*>(const_cast<void*>(host));
  char* hi = lo + bytes;
  auto it = ctx->shadows.upper_bound(lo);
  if (it != ctx->shadows.begin()) --it;
  while (it != ctx->shadows.end() && it->first < hi) {
    auto next = std::next(it);
    if (it->first + it->second.bytes > lo) shadow_erase(ctx, it);
    it = next;
  }
}

bool ffb_shadow_retain(ffb_ctx* ctx, DevBuf& buf, void* host_lo, size_t bytes,
                       const std::vector<std::pair<size_t, size_t>>& valid) {
  if (!buf.p || !host_lo || bytes < SHADOW_MIN_BYTES || bytes > ctx->shadow_limit || valid.empty())
    return false;
  // only arrays that live in this context's page-locked pool: their release (ffb_host_free) is the
  // event that ends the shadow's life
  char* h = static_cast<char*>(host_lo);
  auto ub = ctx->host_live_blocks.upper_bound(h);
  if (ub == ctx->host_live_blocks.begin()) return false;
  --ub;
  if (h + bytes > static_cast<char*>(ub->first) + ub->second) return false;
  ffb_shadow_drop_range(ctx, host_lo, bytes);
  while (ctx->shadow_bytes + bytes > ctx->shadow_limit && !ctx->shadows.empty()) {  // oldest first
    auto oldest = ctx->shadows.begin();
    for (auto it = ctx->shadows.begin(); it != ctx->shadows.end(); ++it)
      if (it->second.stamp < oldest->second.stamp) oldest = it;
    shadow_erase(ctx, oldest);
  }
  ffb_ctx::Shadow sh;
  sh.dev = buf.detach();
  sh.bytes = bytes;
  sh.valid = valid;
  sh.stamp = ++ctx->shadow_clock;
  ctx->shadows[h] = sh;
  ctx->shadow_bytes += bytes;
  return true;
}

int ffb_func_smem_impl(ffb_ctx* ctx, const void* func, size_t smem) {
  auto it = ctx->func_smem.find(func);
  if (it != ctx->func_smem.end() && it->second >= smem) return FFB_OK;
  FFB_CUDA(ctx, cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  ctx->func_smem[func] = smem;
  return FFB_OK;
}

int ffb_occupancy_impl(ffb_ctx* ctx, const void* func, int block_threads, size_t smem, int* blocks) {
  const auto key = std::make_tuple(func, block_threads, smem);
  auto it = ctx->occupancy_cache.find(key);
  if (it != ctx->occupancy_cache.end()) {
    *blocks = it->second;
    return FFB_OK;
  }
  FFB_TRY(ffb_func_smem_impl(ctx, func, smem));
  FFB_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks, func, block_threads, smem));
  ctx->occupancy_cache[key] = *blocks;
  return FFB_OK;
}

int ffb_conv_counter(ffb_ctx* ctx, int** dev) {
  if (!ctx->conv_dev) {
    FFB_CUDA(ctx, cudaMalloc(&ctx->conv_dev, sizeof(int)));
    FFB_CUDA(ctx, cudaMemsetAsync(ctx->conv_dev, 0, sizeof(int), ctx->stream));
    FFB_CUDA(ctx, cudaHostAlloc(&ctx->conv_host, sizeof(int), cudaHostAllocDefault));
    *ctx->conv_host = 0;
  }
  *dev = ctx->conv_dev;
  return FFB_OK;
}

int ffb_conv_fetch(ffb_ctx* ctx) {
  if (!ctx->conv_dev) return FFB_OK;
  FFB_CUDA(ctx, cudaMemcpyAsync(ctx->conv_host, ctx->conv_dev, sizeof(int), cudaMemcpyDeviceToHost,
                                ctx->stream));
  return FFB_OK;
}

int ffb_conv_check(ffb_ctx* ctx) {
  if (!ctx->conv_dev || *ctx->conv_host == 0) return FFB_OK;
  const int n = *ctx->conv_host;
  *ctx->conv_host = 0;
  FFB_CUDA(ctx, cudaMemsetAsync(ctx->conv_dev, 0, sizeof(int), ctx->stream));
  return ffb_fail(ctx, FFB_ENOTCONV, "diagonalize: the Jacobi iteration did not converge for %d matrices", n);
}

int ffb_time_begin(ffb_ctx* ctx, int* slot) {
  *slot = -1;
  if (!ctx->timing) return FFB_OK;
  std::pair<cudaEvent_t, cudaEvent_t> ev;
  if (!ctx->event_pool.empty()) {
    ev = ctx->event_pool.back();
    ctx->event_pool.pop_back();
  } else {
    FFB_CUDA(ctx, cudaEventCreate(&ev.first));
    FFB_CUDA(ctx, cudaEventCreate(&ev.second));
  }
  FFB_CUDA(ctx, cudaEventRecord(ev.first, ctx->stream));
  ctx->pending_events.push_back(ev);
  *slot = (int)ctx->pending_events.size() - 1;
  return FFB_OK;
}

int ffb_time_end(ffb_ctx* ctx, int slot) {
  if (slot < 0) return FFB_OK;
  FFB_CUDA(ctx, cudaEventRecord(ctx->pending_events[slot].second, ctx->stream));
  return FFB_OK;
}

// ------------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------------
extern "C" {

const char* ffb_version(void) { return "ffb200 0.1.0 (sm_100a)"; }

int ffb_init(ffb_ctx** out, int device) {
  if (!out) return FFB_EINVAL;
  *out = nullptr;
  int n_dev = 0;
  cudaError_t e = cudaGetDeviceCount(&n_dev);
  if (e != cudaSuccess || n_dev == 0) {
    (void)cudaGetLastError();
    return ffb_fail(nullptr, FFB_ENODEVICE, "no CUDA device available (%s); ffb200 has no CPU fallback",
                    e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
  }
  if (device < 0 || device >= n_dev)
    return ffb_fail(nullptr, FFB_EINVAL, "device %d out of range [0, %d)", device, n_dev);
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) return ffb_fail(nullptr, FFB_ECUDA, "%s", cudaGetErrorString(e));
  if (prop.major != 10)
    return ffb_fail(nullptr, FFB_ENODEVICE,
                    "device %d (%s) has compute capability %d.%d; libffb200 is built for sm_100a only",
                    device, prop.name, prop.major, prop.minor);
  e = cudaSetDevice(device);
  if (e != cudaSuccess) return ffb_fail(nullptr, FFB_ECUDA, "%s", cudaGetErrorString(e));
  ffb_ctx* ctx = new ffb_ctx();
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
  ctx->cc_major = prop.major;
  ctx->cc_minor = prop.minor;
  ctx->total_mem = prop.totalGlobalMem;
  e = cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking);
  if (e != cudaSuccess) {
    delete ctx;
    return ffb_fail(nullptr, FFB_ECUDA, "%s", cudaGetErrorString(e));
  }
  ctx->stream = ctx->own_stream;
  ctx->shadow_limit = prop.totalGlobalMem / 4;
  if (const char* e = getenv("FFB_SHADOW_BYTES")) ctx->shadow_limit = (size_t)strtoull(e, nullptr, 10);
  *out = ctx;
  return FFB_OK;
}

void ffb_destroy(ffb_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  ffbi_comm_release(ctx);
  while (!ctx->shadows.empty()) shadow_erase(ctx, ctx->shadows.begin());
  for (auto& kv : ctx->free_blocks) cudaFree(kv.second);
  for (auto& kv : ctx->live_blocks) cudaFree(kv.first);
  for (auto& ev : ctx->event_pool) {
    cudaEventDestroy(ev.first);
    cudaEventDestroy(ev.second);
  }
  for (auto& ev : ctx->pending_events) {
    cudaEventDestroy(ev.first);
    cudaEventDestroy(ev.second);
  }
  for (auto& kv : ctx->host_free_blocks) cudaFreeHost(kv.second);
  for (auto& kv : ctx->host_live_blocks) cudaFreeHost(kv.first);
  if (ctx->trig_table) cudaFree(ctx->trig_table);
  if (ctx->band_counts) cudaFree(ctx->band_counts);
  if (ctx->stage_host) cudaFreeHost(ctx->stage_host);
  if (ctx->stage_out) cudaFreeHost(ctx->stage_out);
  if (ctx->conv_dev) cudaFree(ctx->conv_dev);
  if (ctx->infid_scratch) cudaFree(ctx->infid_scratch);
  if (ctx->conv_host) cudaFreeHost(ctx->conv_host);
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  for (auto& ev : ctx->copy_ev)
    if (ev) cudaEventDestroy(ev);
  cudaStreamDestroy(ctx->own_stream);
  delete ctx;
}

const char* ffb_last_error(const ffb_ctx* ctx) {
  return ctx ? ctx->err.c_str() : g_init_error.c_str();
}

int ffb_set_stream(ffb_ctx* ctx, void* cuda_stream, int external) {
  if (!ctx) return FFB_EINVAL;
  FFB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  ctx->stream = external ? static_cast<cudaStream_t>(cuda_stream) : ctx->own_stream;
  return FFB_OK;
}

int ffb_sync(ffb_ctx* ctx) {
  if (!ctx) return FFB_EINVAL;
  FFB_TRY(ffb_conv_fetch(ctx));  // device-resident callers learn about a non-converged eigensolver here
  FFB_TRY(ffbi_comm_fetch_error(ctx));  // ... and about a peer that never arrived
  FFB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  FFB_TRY(ffbi_comm_check_error(ctx));
  return ffb_conv_check(ctx);
}

int64_t ffb_launch_count(const ffb_ctx* ctx) { return ctx ? ctx->launches : 0; }

int ffb_device_info(ffb_ctx* ctx, int* sm_count, int* cc_major, int* cc_minor, size_t* total_mem) {
  if (!ctx) return FFB_EINVAL;
  if (sm_count) *sm_count = ctx->sm_count;
  if (cc_major) *cc_major = ctx->cc_major;
  if (cc_minor) *cc_minor = ctx->cc_minor;
  if (total_mem) *total_mem = ctx->total_mem;
  return FFB_OK;
}

int ffb_measure_fp64_peak(ffb_ctx* ctx, double* dfma_tflops, double* dmma_tflops) {
  if (!ctx) return FFB_EINVAL;
  FFB_CUDA(ctx, cudaSetDevice(ctx->device));
  return ffbi_fp64_peak(ctx, dfma_tflops, dmma_tflops);
}

int ffb_kernel_timing_enable(ffb_ctx* ctx, int enable) {
  if (!ctx) return FFB_EINVAL;
  ctx->timing = enable != 0;
  return FFB_OK;
}

int ffb_kernel_timing_read(ffb_ctx* ctx, double* total_ms, int64_t* launches, int reset) {
  if (!ctx) return FFB_EINVAL;
  FFB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  for (auto& ev : ctx->pending_events) {
    float ms = 0.f;
    FFB_CUDA(ctx, cudaEventElapsedTime(&ms, ev.first, ev.second));
    ctx->timed_ms += ms;
    ctx->timed_launches++;
    ctx->event_pool.push_back(ev);
  }
  ctx->pending_events.clear();
  if (total_ms) *total_ms = ctx->timed_ms;
  if (launches) *launches = ctx->timed_launches;
  if (reset) {
    ctx->timed_ms = 0.0;
    ctx->timed_launches = 0;
  }
  return FFB_OK;
}

namespace {
int copy_log(std::deque<ffb_dispatch_record>& log, ffb_dispatch_record* out, int capacity) {
  int n = 0;
  if (out)
    for (const auto& rec : log) {
      if (n >= capacity) break;
      out[n++] = rec;
    }
  log.clear();
  return n;
}
}  // namespace

int ffb_dispatch_log(ffb_ctx* ctx, ffb_dispatch_record* out, int capacity) {
  if (!ctx) return FFB_EINVAL;
  // banded blocks: the plan kernel counted their bands on the device (n_bands = -(ring slot + 1) until read)
  bool pending = false;
  for (const auto& rec : ctx->dispatch_log) pending = pending || rec.n_bands < 0;
  if (pending && out) {
    std::vector<int> counts((size_t)2 * FFB_DISPATCH_LOG_MAX);
    FFB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    FFB_CUDA(ctx, cudaMemcpy(counts.data(), ctx->band_counts, counts.size() * sizeof(int), cudaMemcpyDeviceToHost));
    for (auto& rec : ctx->dispatch_log) {
      if (rec.n_bands >= 0) continue;
      const int slot = -rec.n_bands - 1;
      rec.n_bands = counts[2 * slot];
      rec.n_proxies = counts[2 * slot + 1];
    }
  }
  return copy_log(ctx->dispatch_log, out, capacity);
}

int ffb_diag_dispatch_log(ffb_ctx* ctx, ffb_dispatch_record* out, int capacity) {
  if (!ctx) return FFB_EINVAL;
  return copy_log(ctx->diag_dispatch_log, out, capacity);
}

// ------------------------------------------------------------------------------------------------
// raw device memory
// ------------------------------------------------------------------------------------------------
int ffb_dev_alloc(ffb_ctx* ctx, size_t bytes, void** ptr) {
  if (!ctx || !ptr) return FFB_EINVAL;
  FFB_CUDA(ctx, cudaSetDevice(ctx->device));
  return ffb_pool_alloc(ctx, bytes ? bytes : 8, ptr);
}

int ffb_dev_free(ffb_ctx* ctx, void* ptr) {
  if (!ctx) return FFB_EINVAL;
  ffb_pool_release(ctx, ptr);
  return FFB_OK;
}

int ffb_host_alloc(ffb_ctx* ctx, size_t bytes, void** ptr) {
  if (!ctx || !ptr) return FFB_EINVAL;
  FFB_CUDA(ctx, cudaSetDevice(ctx->device));
  bytes = (std::max<size_t>(bytes, 8) + 4095) & ~(size_t)4095;
  auto it = ctx->host_free_blocks.lower_bound(bytes);
  if (it != ctx->host_free_blocks.end() && it->first <= 2 * bytes + (1 << 20)) {
    *ptr = it->second;
    ctx->host_live_blocks[*ptr] = it->first;
    ctx->host_free_blocks.erase(it);
    return FFB_OK;
  }
  // keep the amount of page-locked memory bounded: drop cached blocks beyond 4 GiB
  if (ctx->host_pool_bytes + bytes > ((size_t)4 << 30)) {
    for (auto& kv : ctx->host_free_blocks) {
      cudaFreeHost(kv.second);
      ctx->host_pool_bytes -= kv.first;
    }
    ctx->host_free_blocks.clear();
  }
  cudaError_t e = cudaHostAlloc(ptr, bytes, cudaHostAllocDefault);
  if (e != cudaSuccess) {
    (void)cudaGetLastError();
    return ffb_fail(ctx, FFB_ENOMEM, "page-locked allocation of %zu bytes failed: %s", bytes,
                    cudaGetErrorString(e));
  }
  ctx->host_pool_bytes += bytes;
  ctx->host_live_blocks[*ptr] = bytes;
  return FFB_OK;
}

int ffb_host_free(ffb_ctx* ctx, void* ptr) {
  if (!ctx) return FFB_EINVAL;
  auto it = ctx->host_live_blocks.find(ptr);
  if (it == ctx->host_live_blocks.end()) return FFB_OK;
  ffb_shadow_drop_range(ctx, ptr, it->second);  // the arrays in this block are gone: so are their mirrors
  ctx->host_free_blocks.emplace(it->second, ptr);
  ctx->host_live_blocks.erase(it);
  return FFB_OK;
}

int ffb_shadow_enable_next(ffb_ctx* ctx, int enable) {
  if (!ctx) return FFB_EINVAL;
  static const bool allowed = !(getenv("FFB_SHADOWS") && atoi(getenv("FFB_SHADOWS")) == 0);
  ctx->shadow_next = allowed && enable != 0;
  return FFB_OK;
}

int ffb_shadow_upload(ffb_ctx* ctx, const void* host, size_t bytes) {
  if (!ctx || !host || !bytes) return FFB_EINVAL;
  FFB_CUDA(ctx, cudaSetDevice(ctx->device));
  static const bool allowed = !(getenv("FFB_SHADOWS") && atoi(getenv("FFB_SHADOWS")) == 0);
  if (!allowed) return FFB_OK;
  DevBuf buf;
  FFB_TRY(buf.alloc(ctx, bytes));
  FFB_TRY(ffb_h2d(ctx, buf.p, host, bytes));
  FFB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  ffb_shadow_retain(ctx, buf, const_cast<void*>(host), bytes, {{0, bytes}});  // may decline (size, pool)
  return FFB_OK;
}

int ffb_shadow_query(ffb_ctx* ctx, const void* host, size_t bytes) {
  if (!ctx) return 0;
  const int64_t hits = ctx->shadow_hits;
  const size_t hit_bytes = ctx->shadow_hit_bytes;
  const bool found = ffb_shadow_lookup(ctx, host, bytes) != nullptr;
  ctx->shadow_hits = hits;  // a query is not a use
  ctx->shadow_hit_bytes = hit_bytes;
  return found ? 1 : 0;
}

int ffb_shadow_drop(ffb_ctx* ctx, const void* host, size_t bytes) {
  if (!ctx) return FFB_EINVAL;
  ffb_shadow_drop_range(ctx, host, bytes);
  return FFB_OK;
}

int ffb_shadow_stats(ffb_ctx* ctx, int* count, size_t* bytes, int64_t* hits, size_t* hit_bytes) {
  if (!ctx) return FFB_EINVAL;
  if (count) *count = (int)ctx->shadows.size();
  if (bytes) *bytes = ctx->shadow_bytes;
  if (hits) *hits = ctx->shadow_hits;
  if (hit_bytes) *hit_bytes = ctx->shadow_hit_bytes;
  return FFB_OK;
}

int ffb_memcpy_h2d(ffb_ctx* ctx, void* dst_dev, const void* src_host, size_t bytes) {
  if (!ctx) return FFB_EINVAL;
  FFB_TRY(ffb_h2d(ctx, dst_dev, src_host, bytes));
  FFB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return FFB_OK;
}

int ffb_memcpy_d2h(ffb_ctx* ctx, void* dst_host, const void* src_dev, size_t bytes) {
  if (!ctx) return FFB_EINVAL;
  FFB_TRY(ffb_d2h(ctx, dst_host, src_dev, bytes));
  FFB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return FFB_OK;
}

// ------------------------------------------------------------------------------------------------
// device-pointer entry points
// ------------------------------------------------------------------------------------------------
int ffb_dev_diagonalize(ffb_ctx* ctx, int G, int d, int n_cops, const double* c_opers,
                        const double* c_coeffs, const double* dt, double* eigvals, double* eigvecs,
                        double* propagators) {
  if (!ctx) return FFB_EINVAL;
  return ffbi_diagonalize(ctx, G, d, n_cops, c_opers, c_coeffs, dt, eigvals, eigvecs, propagators);
}

int ffb_dev_control_matrix_from_scratch(ffb_ctx* ctx, int G, int d, int n_nops, int n_basis,
                                        int n_omega, const double* eigvals, const double* eigvecs,
                                        const double* propagators, const double* omega,
                                        const double* basis, const double* n_opers,
                                        const double* n_coeffs, const double* dt, const double* t,
                                        int herm_flags, double* out) {
  if (!ctx) return FFB_EINVAL;
  return ffbi_control_matrix(ctx, G, d, n_nops, n_basis, n_omega, eigvals, eigvecs, propagators,
                             omega, basis, n_opers, n_coeffs, dt, t, herm_flags, out);
}

int ffb_dev_filter_function(ffb_ctx* ctx, int P, int n_nops, int n_basis, int n_omega,
                            const double* B, int generalized, double* F) {
  if (!ctx) return FFB_EINVAL;
  return ffbi_filter_function(ctx, P, n_nops, n_basis, n_omega, B, generalized, F);
}

int ffb_dev_control_matrix_from_atomic(ffb_ctx* ctx, int P, int n_nops, int n_basis, int n_omega,
                                       const double* phases, const double* B_atomic,
                                       const double* Q_liouville, int q_is_complex,
                                       int correlations, double* out) {
  if (!ctx) return FFB_EINVAL;
  return ffbi_from_atomic(ctx, P, n_nops, n_basis, n_omega, phases, B_atomic, Q_liouville,
                          q_is_complex, correlations, out);
}

int ffb_dev_infidelity(ffb_ctx* ctx, int n_lead, int n_nops, int n_sel, const int* idx,
                       int n_omega, const double* F, const double* spectrum, int spectrum_ndim,
                       int spectrum_is_complex, const double* omega, int d, double* out) {
  if (!ctx) return FFB_EINVAL;
  return ffbi_infidelity(ctx, n_lead, n_nops, n_sel, idx, n_omega, F, spectrum, spectrum_ndim,
                         spectrum_is_complex, omega, d, out);
}

int ffb_dev_decay_amplitudes(ffb_ctx* ctx, int P, int n_nops, int n_sel, const int* idx,
                             int n_basis, int n_omega, const double* B, const double* spectrum,
                             int spectrum_ndim, int spectrum_is_complex, const double* omega,
                             double* out) {
  if (!ctx) return FFB_EINVAL;
  return ffbi_decay_amplitudes(ctx, P, n_nops, n_sel, idx, n_basis, n_omega, B, spectrum,
                               spectrum_ndim, spectrum_is_complex, omega, out);
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// host-pointer entry points
// ------------------------------------------------------------------------------------------------
namespace {

// exact Hermiticity test of a stack of d x d complex matrices (host side, O(n d^2))
bool all_hermitian(const double* m, int n, int d) {
  for (int i = 0; i < n; ++i) {
    const double* a = m + (size_t)i * 2 * d * d;
    for (int r = 0; r < d; ++r) {
      for (int c = r; c < d; ++c) {
        if (a[2 * (r * d + c)] != a[2 * (c * d + r)]) return false;
        if (a[2 * (r * d + c) + 1] != -a[2 * (c * d + r) + 1]) return false;
      }
    }
  }
  return true;
}

// basis element 0 exactly a real multiple of the identity?
bool first_is_identity(const double* basis, int d) {
  const double c = basis[0];
  for (int r = 0; r < d; ++r)
    for (int q = 0; q < d; ++q) {
      if (basis[2 * (r * d + q)] != (r == q ? c : 0.0)) return false;
      if (basis[2 * (r * d + q) + 1] != 0.0) return false;
    }
  return true;
}

// Hermiticity and identity flags of the noise operators and the basis (FFB_HERM_*, FFB_BASIS_IDENTITY0)
int herm_flags(const double* n_opers, int n_nops, const double* basis, int n_basis, int d) {
  return (all_hermitian(n_opers, n_nops, d) ? FFB_HERM_NOPERS : 0) |
         (all_hermitian(basis, n_basis, d) ? FFB_HERM_BASIS : 0) |
         (n_basis >= 1 && first_is_identity(basis, d) ? FFB_BASIS_IDENTITY0 : 0);
}

// elements of a spectrum of shape (n_omega,), (n_sel, n_omega) or (n_sel, n_sel, n_omega)
size_t spectrum_elems(int ndim, int n_sel, int n_omega) {
  return (ndim == 1 ? 1 : ndim == 2 ? (size_t)n_sel : (size_t)n_sel * n_sel) * n_omega;
}

int enter(ffb_ctx* ctx) {
  if (!ctx) return FFB_EINVAL;
  FFB_CUDA(ctx, cudaSetDevice(ctx->device));
  return FFB_OK;
}

// All host inputs of one call -> ONE page-locked staging block -> as few host-to-device copies as the
// sizes allow.  A pageable cudaMemcpyAsync costs ~10 us of driver time per call and blocks the host for
// the larger ones; a pulse has 8-9 input arrays of 0.1-500 KB each.  The staging block belongs to the
// context and is reused by the next call, so an entry point calls upload() exactly once: a second
// upload() would overwrite staged bytes whose copy may still be in flight.  (Every host-pointer entry
// point is synchronous on return, so the next call finds the block free.)
struct PackedUpload {
  static constexpr size_t ALIGN = 256;
  static constexpr size_t PACK_LIMIT = (size_t)512 << 10;  // larger parts are copied from where they lie
  static constexpr size_t RUN_BYTES = (size_t)128 << 10;   // a run of packed parts is sent at this size
  std::vector<const void*> src, mirror;
  std::vector<size_t> bytes, offset;
  size_t packed = 0, large = 0;  // bytes through the staging block, bytes copied from where they lie
  DevBuf dev;
  ffb_ctx* ctx;
  explicit PackedUpload(ffb_ctx* c) : ctx(c) {}
  int add(const void* host, size_t n) {
    // a part that is mirrored on the device already (a cached result array) is not sent again
    const void* m = ffb_shadow_lookup(ctx, host, n);
    size_t& end = !m && n > PACK_LIMIT ? large : packed;
    src.push_back(host);
    mirror.push_back(m);
    bytes.push_back(m ? 0 : n);
    offset.push_back(end);
    if (!m) end += (n + ALIGN - 1) & ~(ALIGN - 1);
    return (int)src.size() - 1;
  }
  // device layout: the staging block's layout, then the large parts
  char* at(size_t i) const { return dev.as<char>() + offset[i] + (bytes[i] > PACK_LIMIT ? packed : 0); }
  int upload() {
    if (ctx->stage_bytes < packed) {
      if (ctx->stage_host) FFB_CUDA(ctx, cudaFreeHost(ctx->stage_host));
      ctx->stage_host = nullptr;
      ctx->stage_bytes = 0;
      const size_t want = std::max<size_t>(2 * packed, (size_t)1 << 20);
      FFB_CUDA(ctx, cudaHostAlloc(&ctx->stage_host, want, cudaHostAllocDefault));
      ctx->stage_bytes = want;
    }
    char* stage = static_cast<char*>(ctx->stage_host);
    FFB_TRY(dev.alloc(ctx, packed + large));
    char* d0 = dev.as<char>();
    // runs of consecutive small parts travel in one copy out of the staging block, a large part in its
    // own copy straight from the caller's array (which is page-locked already when it is one of the
    // library's result arrays)
    size_t run_begin = 0, run_end = 0;
    auto flush = [&]() -> int {
      if (run_end > run_begin) FFB_TRY(ffb_h2d(ctx, d0 + run_begin, stage + run_begin, run_end - run_begin));
      run_begin = run_end = 0;
      return FFB_OK;
    };
    for (size_t i = 0; i < src.size(); ++i) {
      if (!bytes[i]) continue;
      if (bytes[i] > PACK_LIMIT) {
        FFB_TRY(ffb_h2d(ctx, at(i), src[i], bytes[i]));
        continue;
      }
      std::memcpy(stage + offset[i], src[i], bytes[i]);
      if (run_end == run_begin) run_begin = offset[i];
      run_end = offset[i] + bytes[i];
      if (run_end - run_begin >= RUN_BYTES) FFB_TRY(flush());  // send what is packed while the rest is packed
    }
    return flush();
  }
  template <typename T = double>
  const T* d(int i) const {
    return static_cast<const T*>(mirror[i] ? mirror[i] : static_cast<const void*>(at(i)));
  }
};

// `to` waits for the work enqueued on `from` so far (through the context's copy event `ev`)
int after(ffb_ctx* ctx, int ev, cudaStream_t from, cudaStream_t to) {
  FFB_CUDA(ctx, cudaEventRecord(ctx->copy_ev[ev], from));
  FFB_CUDA(ctx, cudaStreamWaitEvent(to, ctx->copy_ev[ev], 0));
  return FFB_OK;
}

// enqueue on the copy stream the strided download of frequencies [w0, w1) of every row of a
// (rows, n_omega) complex result
int download_freqs(ffb_ctx* ctx, double* host, const double* dev, size_t rows, int n_omega, int w0, int w1) {
  const size_t pitch = (size_t)n_omega * 16, off = (size_t)w0 * 16;
  FFB_CUDA(ctx, cudaMemcpy2DAsync(reinterpret_cast<char*>(host) + off, pitch,
                                  reinterpret_cast<const char*>(dev) + off, pitch, (size_t)(w1 - w0) * 16,
                                  rows, cudaMemcpyDeviceToHost, ctx->copy_stream));
  return FFB_OK;
}

// microseconds since construction, for the FFB_TRACE timelines
struct TraceClock {
  const std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
  double operator()() const {
    return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t0).count();
  }
};

// number of frequency blocks of a pipeline that returns out_bytes of frequency-dependent results
// (measured on B200, e2e ms with 1 / 2 / 4 / 8 blocks: config 2 (3.4 MB) 1.37 / 1.38 / 1.44 / 1.55, d4
// (21 MB) 17.65 / 17.29 / 17.73 / 18.07, config 3 (105 MB) 18.74 / 18.39 / 17.46 / 17.48 -- a block pays
// off from ~10 MB of results per block)
int pipeline_blocks(size_t out_bytes, int n_omega) {
  int n = (int)std::min<size_t>(4, std::max<size_t>(1, out_bytes / ((size_t)10 << 20)));
  n = std::max(1, std::min(n, n_omega / 2048));
  if (const char* e = getenv("FFB_PIPELINE_BLOCKS")) n = std::max(1, atoi(e));
  return n;
}

int ensure_copy_stream(ffb_ctx* ctx) {
  if (ctx->copy_stream) return FFB_OK;
  FFB_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
  for (auto& ev : ctx->copy_ev) FFB_CUDA(ctx, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  return FFB_OK;
}

// the copy stream may read buffers that go back to the pool at scope exit: drain it first (declare
// AFTER the buffers, so that it is destroyed BEFORE them), also on the error paths
struct CopyStreamDrain {
  ffb_ctx* ctx;
  ~CopyStreamDrain() {
    if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
  }
};

// The results of one call in ONE device block.  If all result pointers of the caller lie in one
// page-locked block of the library's own pool (ffb_host_alloc; that is how the Python shell allocates
// them, _lib.empty_many), the device block MIRRORS that layout, and results that are neighbours there
// (less than 256 bytes of alignment padding apart) travel in one device-to-host copy: a small pulse
// is bound by the number of driver calls, not by bytes (config 1: 8 copies -> 2).
struct OutputBlock {
  static constexpr size_t ALIGN = 256;
  struct Item {
    char* host;
    size_t bytes, off;
  };
  static constexpr size_t STAGED_LIMIT = (size_t)256 << 10;
  std::vector<Item> items;
  std::vector<const Item*> staged_items;  // downloaded into the context's staging block, not yet delivered
  DevBuf dev;
  bool mirrored = false;
  bool staged = false;  // small results to pageable memory: one copy into ctx->stage_out + memcpy
  size_t total_bytes = 0;
  char* host_base = nullptr;
  int add(void* host, size_t bytes) {
    items.push_back({static_cast<char*>(host), bytes, 0});
    return (int)items.size() - 1;
  }
  // keep the device block as the shadow of the listed results (they must have been downloaded)
  bool retain(ffb_ctx* ctx, std::initializer_list<int> which) {
    if (!mirrored) return false;
    std::vector<std::pair<size_t, size_t>> valid;
    size_t hi = 0;
    for (int i : which)
      if (i >= 0 && items[i].host && items[i].bytes) {
        valid.emplace_back(items[i].off, items[i].bytes);
        hi = std::max(hi, items[i].off + items[i].bytes);
      }
    return ffb_shadow_retain(ctx, dev, host_base, hi, valid);
  }
  int alloc(ffb_ctx* ctx) {
    for (const Item& it : items)
      if (it.host && it.bytes) ffb_shadow_drop_range(ctx, it.host, it.bytes);
    // one pool block that contains every requested result?
    char* lo = nullptr;
    char* hi = nullptr;
    mirrored = true;
    const void* block = nullptr;
    for (const Item& it : items) {
      if (!it.host || !it.bytes) continue;
      auto ub = ctx->host_live_blocks.upper_bound(it.host);
      if (ub == ctx->host_live_blocks.begin()) { mirrored = false; break; }
      --ub;
      char* b0 = static_cast<char*>(ub->first);
      if (it.host + it.bytes > b0 + ub->second || (block && block != ub->first) ||
          (size_t)(it.host - b0) % ALIGN != 0) {
        mirrored = false;
        break;
      }
      block = ub->first;
      lo = lo ? std::min(lo, it.host) : it.host;
      hi = hi ? std::max(hi, it.host + it.bytes) : it.host + it.bytes;
    }
    if (!block) mirrored = false;
    size_t total = 0;
    if (mirrored) {  // overlap check: sorted by address, no two results may share bytes
      std::vector<const Item*> order;
      for (const Item& it : items)
        if (it.host && it.bytes) order.push_back(&it);
      std::sort(order.begin(), order.end(), [](const Item* a, const Item* b) { return a->host < b->host; });
      for (size_t i = 1; i < order.size(); ++i)
        if (order[i]->host < order[i - 1]->host + order[i - 1]->bytes) mirrored = false;
    }
    if (mirrored) {  // results scattered over a large block: mirroring would waste device memory
      size_t sum = 0;
      for (const Item& it : items) sum += it.bytes;
      if ((size_t)(hi - lo) > 2 * sum + ((size_t)1 << 20)) mirrored = false;
    }
    if (mirrored) {
      host_base = lo;
      total = ((size_t)(hi - lo) + ALIGN - 1) & ~(ALIGN - 1);
      for (Item& it : items)
        if (it.host && it.bytes) it.off = (size_t)(it.host - lo);
    }
    for (Item& it : items) {  // not requested (or no mirroring): packed behind
      if (mirrored && it.host && it.bytes) continue;
      it.off = total;
      total += (it.bytes + ALIGN - 1) & ~(ALIGN - 1);
    }
    total_bytes = total;
    staged = !mirrored && total <= STAGED_LIMIT;
    if (staged && ctx->stage_out_bytes < total) {
      if (ctx->stage_out) FFB_CUDA(ctx, cudaFreeHost(ctx->stage_out));
      ctx->stage_out = nullptr;
      ctx->stage_out_bytes = 0;
      FFB_CUDA(ctx, cudaHostAlloc(&ctx->stage_out, STAGED_LIMIT, cudaHostAllocDefault));
      ctx->stage_out_bytes = STAGED_LIMIT;
    }
    return dev.alloc(ctx, total);
  }
  // after the stream the downloads were enqueued on has been synchronised
  void finish(ffb_ctx* ctx) {
    for (const Item* it : staged_items)
      std::memcpy(it->host, static_cast<const char*>(ctx->stage_out) + it->off, it->bytes);
    staged_items.clear();
  }
  template <typename T = double>
  T* d(int i) const {
    return reinterpret_cast<T*>(static_cast<char*>(dev.p) + items[i].off);
  }
  // enqueue the download of the listed results on `stream`
  int download(ffb_ctx* ctx, std::initializer_list<int> which, cudaStream_t stream) {
    std::vector<const Item*> order;
    for (int i : which)
      if (i >= 0 && items[i].host && items[i].bytes) order.push_back(&items[i]);
    if (order.empty()) return FFB_OK;
    if (staged) {  // one copy of the span that holds the requested results
      size_t lo = order[0]->off, hi = lo;
      for (const Item* it : order) {
        lo = std::min(lo, it->off);
        hi = std::max(hi, it->off + it->bytes);
        staged_items.push_back(it);
      }
      FFB_CUDA(ctx, cudaMemcpyAsync(static_cast<char*>(ctx->stage_out) + lo, static_cast<char*>(dev.p) + lo,
                                    hi - lo, cudaMemcpyDeviceToHost, stream));
      return FFB_OK;
    }
    if (!mirrored) {
      for (const Item* it : order)
        FFB_CUDA(ctx, cudaMemcpyAsync(it->host, static_cast<char*>(dev.p) + it->off, it->bytes,
                                      cudaMemcpyDeviceToHost, stream));
      return FFB_OK;
    }
    std::sort(order.begin(), order.end(), [](const Item* a, const Item* b) { return a->off < b->off; });
    size_t r0 = order[0]->off, r1 = r0 + order[0]->bytes;
    auto flush = [&]() -> int {
      FFB_CUDA(ctx, cudaMemcpyAsync(host_base + r0, static_cast<char*>(dev.p) + r0, r1 - r0,
                                    cudaMemcpyDeviceToHost, stream));
      return FFB_OK;
    };
    for (size_t i = 1; i < order.size(); ++i) {
      if (order[i]->off < r1 + ALIGN) {  // neighbours: only alignment padding in between
        r1 = order[i]->off + order[i]->bytes;
      } else {
        FFB_TRY(flush());
        r0 = order[i]->off;
        r1 = r0 + order[i]->bytes;
      }
    }
    return flush();
  }
};

}  // namespace

extern "C" {

int ffb_diagonalize(ffb_ctx* ctx, int G, int d, int n_cops, const double* c_opers,
                    const double* c_coeffs, const double* dt, double* eigvals, double* eigvecs,
                    double* propagators) {
  FFB_TRY(enter(ctx));
  FFB_REQUIRE(ctx, c_opers && dt && eigvals && eigvecs && propagators, "diagonalize: null pointer");
  FFB_CHECK_DIM(ctx, d);
  FFB_REQUIRE(ctx, G >= 1 && d >= 1 && d <= 32, "diagonalize: G=%d, d=%d unsupported", G, d);
  const size_t dd = (size_t)d * d;
  PackedUpload in(ctx);
  DevBuf ev, V, Q;
  const size_t n_mats = c_coeffs ? (size_t)n_cops : (size_t)G;
  const int i_co = in.add(c_opers, n_mats * dd * 16);
  const int i_cc = c_coeffs ? in.add(c_coeffs, (size_t)n_cops * G * 8) : -1;
  const int i_dt = in.add(dt, (size_t)G * 8);
  FFB_TRY(in.upload());
  FFB_TRY(ev.alloc(ctx, (size_t)G * d * 8));
  FFB_TRY(V.alloc(ctx, (size_t)G * dd * 16));
  FFB_TRY(Q.alloc(ctx, (size_t)(G + 1) * dd * 16));
  FFB_TRY(ffbi_diagonalize(ctx, G, d, n_cops, in.d(i_co), c_coeffs ? in.d(i_cc) : nullptr, in.d(i_dt),
                           ev.as<double>(), V.as<double>(), Q.as<double>()));
  FFB_TRY(ffb_d2h(ctx, eigvals, ev.p, (size_t)G * d * 8));
  FFB_TRY(ffb_d2h(ctx, eigvecs, V.p, (size_t)G * dd * 16));
  FFB_TRY(ffb_d2h(ctx, propagators, Q.p, (size_t)(G + 1) * dd * 16));
  FFB_TRY(ffb_conv_fetch(ctx));
  FFB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return ffb_conv_check(ctx);
}

int ffb_control_matrix_from_scratch(ffb_ctx* ctx, int G, int d, int n_nops, int n_basis,
                                    int n_omega, const double* eigvals, const double* eigvecs,
                                    const double* propagators, const double* omega,
                                    const double* basis, const double* n_opers,
                                    const double* n_coeffs, const double* dt, const double* t,
                                    double* out) {
  FFB_TRY(enter(ctx));
  FFB_REQUIRE(ctx, eigvals && eigvecs && propagators && omega && basis && n_opers && n_coeffs &&
                       dt && t && out, "control matrix: null pointer");
  FFB_CHECK_DIM(ctx, d);
  FFB_REQUIRE(ctx, G >= 1 && d >= 1 && d <= 32 && n_nops >= 1 && n_basis >= 1 && n_omega >= 1,
              "control matrix: bad shape");
  const bool keep = ctx->shadow_next;
  ctx->shadow_next = false;
  const size_t dd = (size_t)d * d;
  const int herm = herm_flags(n_opers, n_nops, basis, n_basis, d);
  FFB_TRY(ensure_copy_stream(ctx));
  ffb_shadow_drop_range(ctx, out, (size_t)n_nops * n_basis * n_omega * 16);
  const TraceClock since;
  PackedUpload in(ctx);
  DevBuf B;
  CopyStreamDrain drain{ctx};
  const int i_ev = in.add(eigvals, (size_t)G * d * 8);
  const int i_V = in.add(eigvecs, (size_t)G * dd * 16);
  const int i_Q = in.add(propagators, (size_t)G * dd * 16);  // Q_G (the last one) is not needed
  const int i_om = in.add(omega, (size_t)n_omega * 8);
  const int i_bs = in.add(basis, (size_t)n_basis * dd * 16);
  const int i_no = in.add(n_opers, (size_t)n_nops * dd * 16);
  const int i_nc = in.add(n_coeffs, (size_t)n_nops * G * 8);
  const int i_dt = in.add(dt, (size_t)G * 8);
  const int i_ts = in.add(t, (size_t)(G + 1) * 8);
  FFB_TRY(in.upload());
  const size_t out_bytes = (size_t)n_nops * n_basis * n_omega * 16;
  FFB_TRY(B.alloc(ctx, out_bytes));
  // the rows of a finished block of frequencies are downloaded while the next block is computed
  FreqBlocks fb;
  fb.n_blocks = pipeline_blocks(out_bytes, n_omega);
  fb.after_block = [&](int w0, int w1) -> int {
    FFB_TRY(after(ctx, 1, ctx->stream, ctx->copy_stream));
    return download_freqs(ctx, out, B.as<double>(), (size_t)n_nops * n_basis, n_omega, w0, w1);
  };
  FFB_TRY(ffbi_control_matrix(ctx, G, d, n_nops, n_basis, n_omega, in.d(i_ev), in.d(i_V), in.d(i_Q),
                              in.d(i_om), in.d(i_bs), in.d(i_no), in.d(i_nc), in.d(i_dt), in.d(i_ts),
                              herm, B.as<double>(), &fb));
  const double us_enqueued = since();
  FFB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  const double us_main = since();
  FFB_CUDA(ctx, cudaStreamSynchronize(ctx->copy_stream));
  if (ffb_trace())
    fprintf(stderr, "[ffb trace] control matrix: all work enqueued %.0f us, main stream done %.0f us, "
            "copy stream done %.0f us (%d blocks)\n", us_enqueued, us_main, since(), fb.n_blocks);
  if (keep) ffb_shadow_retain(ctx, B, out, out_bytes, {{0, out_bytes}});
  return FFB_OK;
}

int ffb_control_matrix_intermediates(ffb_ctx* ctx, int G, int d, int n_nops, int n_basis,
                                     int n_omega, const double* eigvals, const double* eigvecs,
                                     const double* propagators, const double* omega,
                                     const double* basis, const double* n_opers,
                                     const double* n_coeffs, const double* dt, const double* t,
                                     double* out, double* n_opers_transformed,
                                     double* eigvecs_propagated, double* basis_transformed,
                                     double* phase_factors, double* first_order_integral,
                                     double* control_matrix_step,
                                     double* control_matrix_step_cumulative) {
  FFB_TRY(enter(ctx));
  FFB_REQUIRE(ctx, eigvals && eigvecs && propagators && omega && basis && n_opers && n_coeffs &&
                       dt && t && out && n_opers_transformed && eigvecs_propagated &&
                       basis_transformed && phase_factors && first_order_integral &&
                       control_matrix_step && (G == 1 || control_matrix_step_cumulative),
              "control matrix intermediates: null pointer");
  FFB_CHECK_DIM(ctx, d);
  FFB_REQUIRE(ctx, G >= 1 && d >= 1 && d <= 32 && n_nops >= 1 && n_basis >= 1 && n_omega >= 1,
              "control matrix intermediates: bad shape");
  const size_t dd = (size_t)d * d;
  PackedUpload in(ctx);
  DevBuf B, Bt, Up, Ct, Ph, In, St, Cu;
  const int i_ev = in.add(eigvals, (size_t)G * d * 8);
  const int i_V = in.add(eigvecs, (size_t)G * dd * 16);
  const int i_Q = in.add(propagators, (size_t)G * dd * 16);
  const int i_om = in.add(omega, (size_t)n_omega * 8);
  const int i_bs = in.add(basis, (size_t)n_basis * dd * 16);
  const int i_no = in.add(n_opers, (size_t)n_nops * dd * 16);
  const int i_nc = in.add(n_coeffs, (size_t)n_nops * G * 8);
  const int i_dt = in.add(dt, (size_t)G * 8);
  const int i_ts = in.add(t, (size_t)(G + 1) * 8);
  FFB_TRY(in.upload());
  const size_t per_step = (size_t)n_nops * n_basis * n_omega * 16;
  const size_t b_bt = (size_t)n_nops * G * dd * 16, b_up = (size_t)G * dd * 16,
               b_ct = (size_t)G * n_basis * dd * 16, b_ph = (size_t)G * n_omega * 16,
               b_in = (size_t)G * n_omega * dd * 16, b_st = (size_t)G * per_step,
               b_cu = (size_t)(G - 1) * per_step;
  FFB_TRY(B.alloc(ctx, per_step));
  FFB_TRY(Bt.alloc(ctx, b_bt));
  FFB_TRY(Up.alloc(ctx, b_up));
  FFB_TRY(Ct.alloc(ctx, b_ct));
  FFB_TRY(Ph.alloc(ctx, b_ph));
  FFB_TRY(In.alloc(ctx, b_in));
  FFB_TRY(St.alloc(ctx, b_st));
  FFB_TRY(Cu.alloc(ctx, b_cu));
  FFB_TRY(ffbi_control_matrix_intermediates(
      ctx, G, d, n_nops, n_basis, n_omega, in.d(i_ev), in.d(i_V), in.d(i_Q), in.d(i_om), in.d(i_bs),
      in.d(i_no), in.d(i_nc), in.d(i_dt), in.d(i_ts), B.as<double>(), Bt.as<double>(), Up.as<double>(),
      Ct.as<double>(), Ph.as<double>(), In.as<double>(), St.as<double>(), Cu.as<double>()));
  FFB_TRY(ffb_d2h(ctx, out, B.p, per_step));
  FFB_TRY(ffb_d2h(ctx, n_opers_transformed, Bt.p, b_bt));
  FFB_TRY(ffb_d2h(ctx, eigvecs_propagated, Up.p, b_up));
  FFB_TRY(ffb_d2h(ctx, basis_transformed, Ct.p, b_ct));
  FFB_TRY(ffb_d2h(ctx, phase_factors, Ph.p, b_ph));
  FFB_TRY(ffb_d2h(ctx, first_order_integral, In.p, b_in));
  FFB_TRY(ffb_d2h(ctx, control_matrix_step, St.p, b_st));
  if (G > 1) FFB_TRY(ffb_d2h(ctx, control_matrix_step_cumulative, Cu.p, b_cu));
  FFB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return FFB_OK;
}

int ffb_filter_function(ffb_ctx* ctx, int P, int n_nops, int n_basis, int n_omega, const double* B,
                        int generalized, double* F) {
  FFB_TRY(enter(ctx));
  FFB_REQUIRE(ctx, B && F, "filter function: null pointer");
  FFB_REQUIRE(ctx, P >= 1 && n_nops >= 1 && n_basis >= 1 && n_omega >= 1,
              "filter function: bad shape");
  PackedUpload in(ctx);
  DevBuf Fd;
  const size_t L = (size_t)P * n_nops;
  const size_t f_bytes = L * L * (generalized ? (size_t)n_basis * n_basis : 1) * n_omega * 16;
  const int i_B = in.add(B, L * n_basis * n_omega * 16);
  FFB_TRY(in.upload());
  FFB_TRY(Fd.alloc(ctx, f_bytes));
  FFB_TRY(ffbi_filter_function(ctx, P, n_nops, n_basis, n_omega, in.d(i_B), generalized,
                               Fd.as<double>()));
  FFB_TRY(ffb_d2h(ctx, F, Fd.p, f_bytes));
  FFB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return FFB_OK;
}

int ffb_control_matrix_from_atomic(ffb_ctx* ctx, int P, int n_nops, int n_basis, int n_omega,
                                   const double* phases, const double* B_atomic,
                                   const double* Q_liouville, int q_is_complex, int correlations,
                                   double* out) {
  FFB_TRY(enter(ctx));
  FFB_REQUIRE(ctx, B_atomic && out && (P == 1 || (phases && Q_liouville)),
              "from_atomic: null pointer");
  FFB_REQUIRE(ctx, P >= 1 && n_nops >= 1 && n_basis >= 1 && n_omega >= 1, "from_atomic: bad shape");
  PackedUpload in(ctx);
  DevBuf O;
  const size_t pulse_bytes = (size_t)n_nops * n_basis * n_omega * 16;
  const int i_ph = P > 1 ? in.add(phases, (size_t)(P - 1) * n_omega * 16) : -1;
  const int i_Q = P > 1 ? in.add(Q_liouville, (size_t)(P - 1) * n_basis * n_basis * (q_is_complex ? 16 : 8))
                        : -1;
  const int i_Ba = in.add(B_atomic, P * pulse_bytes);
  FFB_TRY(in.upload());
  const size_t out_bytes = (correlations ? P : 1) * pulse_bytes;
  FFB_TRY(O.alloc(ctx, out_bytes));
  FFB_TRY(ffbi_from_atomic(ctx, P, n_nops, n_basis, n_omega, P > 1 ? in.d(i_ph) : nullptr, in.d(i_Ba),
                           P > 1 ? in.d(i_Q) : nullptr, q_is_complex, correlations, O.as<double>()));
  FFB_TRY(ffb_d2h(ctx, out, O.p, out_bytes));
  FFB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return FFB_OK;
}

int ffb_control_matrix_periodic(ffb_ctx* ctx, int n_nops, int n_basis, int n_omega, int repeats,
                                const double* phases, const double* B, const double* L,
                                int l_is_complex, double* out) {
  FFB_TRY(enter(ctx));
  FFB_REQUIRE(ctx, phases && B && L && out, "periodic control matrix: null pointer");
  FFB_REQUIRE(ctx, n_nops >= 1 && n_basis >= 1 && n_omega >= 1 && repeats >= 1,
              "periodic control matrix: bad shape");
  PackedUpload in(ctx);
  DevBuf O;
  const size_t b_bytes = (size_t)n_nops * n_basis * n_omega * 16;
  const int i_ph = in.add(phases, (size_t)n_omega * 16);
  const int i_B = in.add(B, b_bytes);
  const int i_L = in.add(L, (size_t)n_basis * n_basis * (l_is_complex ? 16 : 8));
  FFB_TRY(in.upload());
  FFB_TRY(O.alloc(ctx, b_bytes));
  FFB_TRY(ffbi_control_matrix_periodic(ctx, n_nops, n_basis, n_omega, repeats, in.d(i_ph), in.d(i_B),
                                       in.d(i_L), l_is_complex, O.as<double>()));
  FFB_TRY(ffb_d2h(ctx, out, O.p, b_bytes));
  FFB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return FFB_OK;
}

int ffb_infidelity(ffb_ctx* ctx, int n_lead, int n_nops, int n_sel, const int* idx, int n_omega,
                   const double* F, const double* spectrum, int spectrum_ndim,
                   int spectrum_is_complex, const double* omega, int d, double* out) {
  FFB_TRY(enter(ctx));
  FFB_REQUIRE(ctx, idx && F && spectrum && omega && out, "infidelity: null pointer");
  FFB_REQUIRE(ctx, spectrum_ndim >= 1 && spectrum_ndim <= 3, "infidelity: spectrum_ndim=%d",
              spectrum_ndim);
  for (int i = 0; i < n_sel; ++i)
    FFB_REQUIRE(ctx, idx[i] >= 0 && idx[i] < n_nops, "infidelity: idx[%d]=%d out of range", i, idx[i]);
  DevBuf res;
  // a filter function that is still mirrored on the device (the pulse's cached array) is not sent at all
  PackedUpload in(ctx);
  const int i_F = in.add(F, (size_t)n_lead * n_nops * n_nops * n_omega * 16);
  const int i_S = in.add(spectrum,
                         spectrum_elems(spectrum_ndim, n_sel, n_omega) * (spectrum_is_complex ? 16 : 8));
  const int i_om = in.add(omega, (size_t)n_omega * 8);
  const int i_ix = in.add(idx, (size_t)n_sel * sizeof(int));
  FFB_TRY(in.upload());
  const size_t n_out = (size_t)n_lead * (spectrum_ndim == 3 ? (size_t)n_sel * n_sel : n_sel);
  FFB_TRY(res.alloc(ctx, n_out * 8));
  FFB_TRY(ffbi_infidelity(ctx, n_lead, n_nops, n_sel, in.d<int>(i_ix), n_omega, in.d(i_F), in.d(i_S),
                          spectrum_ndim, spectrum_is_complex, in.d(i_om), d, res.as<double>()));
  FFB_TRY(ffb_d2h(ctx, out, res.p, n_out * 8));
  FFB_TRY(ffbi_comm_fetch_error(ctx));
  FFB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return ffbi_comm_check_error(ctx);
}

int ffb_infidelity_derivative(ffb_ctx* ctx, int G, int d, int n_cops, int n_nops, int n_basis,
                              int n_omega, const double* c_opers, const double* c_coeffs,
                              const double* eigvals, const double* eigvecs,
                              const double* propagators, const double* omega, const double* basis,
                              const double* n_opers, const double* n_coeffs, const double* dt,
                              const double* t, const double* control_matrix, int n_ctrl,
                              const int* ctrl_idx, int n_sel, const int* sel_idx,
                              const double* spectrum, int spectrum_ndim,
                              const double* n_coeffs_deps, int norm_d, double* out) {
  FFB_TRY(enter(ctx));
  const bool diag = !eigvals;
  FFB_REQUIRE(ctx, c_opers && omega && basis && n_opers && n_coeffs && dt && t && ctrl_idx && sel_idx &&
                       spectrum && out && (diag ? c_coeffs && !eigvecs && !propagators
                                                : eigvecs && propagators),
              "infidelity derivative: null pointer");
  FFB_REQUIRE(ctx, d >= 1 && d <= 8,
              "infidelity derivative: Hilbert-space dimension d = %d exceeds the supported maximum of 8 "
              "of filter_functions_b200 (README: limits)", d);
  FFB_REQUIRE(ctx, G >= 1 && n_cops >= 1 && n_nops >= 1 && n_basis >= 1 && n_omega >= 1 && n_ctrl >= 1 &&
                       n_sel >= 1 && norm_d >= 1,
              "infidelity derivative: bad shape");
  FFB_REQUIRE(ctx, spectrum_ndim == 1 || spectrum_ndim == 2, "infidelity derivative: spectrum_ndim=%d",
              spectrum_ndim);
  for (int i = 0; i < n_ctrl; ++i)
    FFB_REQUIRE(ctx, ctrl_idx[i] >= 0 && ctrl_idx[i] < n_cops,
                "infidelity derivative: ctrl_idx[%d]=%d out of range", i, ctrl_idx[i]);
  for (int i = 0; i < n_sel; ++i)
    FFB_REQUIRE(ctx, sel_idx[i] >= 0 && sel_idx[i] < n_nops,
                "infidelity derivative: sel_idx[%d]=%d out of range", i, sel_idx[i]);
  const size_t dd = (size_t)d * d;
  // one packed upload; arrays the pulse keeps mirrored on the device (its cached eigensystem and
  // control matrix) are read from there
  PackedUpload in(ctx);
  const int i_co = in.add(c_opers, (size_t)n_cops * dd * 16);
  const int i_cc = diag ? in.add(c_coeffs, (size_t)n_cops * G * 8) : -1;
  const int i_ev = diag ? -1 : in.add(eigvals, (size_t)G * d * 8);
  const int i_V = diag ? -1 : in.add(eigvecs, (size_t)G * dd * 16);
  const int i_Q = diag ? -1 : in.add(propagators, (size_t)G * dd * 16);
  const int i_om = in.add(omega, (size_t)n_omega * 8);
  const int i_bs = in.add(basis, (size_t)n_basis * dd * 16);
  const int i_no = in.add(n_opers, (size_t)n_nops * dd * 16);
  const int i_nc = in.add(n_coeffs, (size_t)n_nops * G * 8);
  const int i_dt = in.add(dt, (size_t)G * 8);
  const int i_ts = in.add(t, (size_t)(G + 1) * 8);
  const int i_B = control_matrix ? in.add(control_matrix, (size_t)n_nops * n_basis * n_omega * 16) : -1;
  const int i_ci = in.add(ctrl_idx, (size_t)n_ctrl * sizeof(int));
  const int i_si = in.add(sel_idx, (size_t)n_sel * sizeof(int));
  const int i_sp = in.add(spectrum, spectrum_elems(spectrum_ndim, n_sel, n_omega) * 8);
  const int i_dp = n_coeffs_deps ? in.add(n_coeffs_deps, (size_t)n_nops * n_ctrl * G * 8) : -1;
  FFB_TRY(in.upload());
  DevBuf ev, V, Q, B, res;
  const double *ev_d, *V_d, *Q_d;
  if (diag) {
    FFB_TRY(ev.alloc(ctx, (size_t)G * d * 8));
    FFB_TRY(V.alloc(ctx, (size_t)G * dd * 16));
    FFB_TRY(Q.alloc(ctx, (size_t)(G + 1) * dd * 16));
    FFB_TRY(ffbi_diagonalize(ctx, G, d, n_cops, in.d(i_co), in.d(i_cc), in.d(i_dt), ev.as<double>(),
                             V.as<double>(), Q.as<double>()));
    ev_d = ev.as<double>();
    V_d = V.as<double>();
    Q_d = Q.as<double>();
  } else {
    ev_d = in.d(i_ev);
    V_d = in.d(i_V);
    Q_d = in.d(i_Q);
  }
  const double* B_d;
  if (control_matrix) {
    B_d = in.d(i_B);
  } else {
    FFB_TRY(B.alloc(ctx, (size_t)n_nops * n_basis * n_omega * 16));
    FFB_TRY(ffbi_control_matrix(ctx, G, d, n_nops, n_basis, n_omega, ev_d, V_d, Q_d, in.d(i_om),
                                in.d(i_bs), in.d(i_no), in.d(i_nc), in.d(i_dt), in.d(i_ts),
                                herm_flags(n_opers, n_nops, basis, n_basis, d), B.as<double>()));
    B_d = B.as<double>();
  }
  const size_t n_out = (size_t)n_sel * G * n_ctrl;
  FFB_TRY(res.alloc(ctx, n_out * 8));
  FFB_TRY(ffbi_infidelity_derivative(
      ctx, G, d, n_nops, n_basis, n_omega, ev_d, V_d, Q_d, in.d(i_om), in.d(i_bs), in.d(i_no),
      in.d(i_nc), in.d(i_dt), in.d(i_ts), in.d(i_co), B_d, n_ctrl, in.d<int>(i_ci), n_sel, in.d<int>(i_si),
      in.d(i_sp), spectrum_ndim, n_coeffs_deps ? in.d(i_dp) : nullptr, norm_d, res.as<double>()));
  FFB_TRY(ffb_d2h(ctx, out, res.p, n_out * 8));
  if (diag) FFB_TRY(ffb_conv_fetch(ctx));
  FFB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return diag ? ffb_conv_check(ctx) : FFB_OK;
}

int ffb_decay_amplitudes(ffb_ctx* ctx, int P, int n_nops, int n_sel, const int* idx, int n_basis,
                         int n_omega, const double* B, const double* spectrum, int spectrum_ndim,
                         int spectrum_is_complex, const double* omega, double* out) {
  FFB_TRY(enter(ctx));
  FFB_REQUIRE(ctx, idx && B && spectrum && omega && out, "decay amplitudes: null pointer");
  FFB_REQUIRE(ctx, spectrum_ndim >= 1 && spectrum_ndim <= 3, "decay amplitudes: spectrum_ndim=%d",
              spectrum_ndim);
  FFB_REQUIRE(ctx, P >= 1 && n_nops >= 1 && n_sel >= 1 && n_basis >= 1 && n_omega >= 1,
              "decay amplitudes: bad shape");
  for (int i = 0; i < n_sel; ++i)
    FFB_REQUIRE(ctx, idx[i] >= 0 && idx[i] < n_nops, "decay amplitudes: idx[%d]=%d out of range", i,
                idx[i]);
  PackedUpload in(ctx);
  DevBuf res;
  const int i_B = in.add(B, (size_t)P * n_nops * n_basis * n_omega * 16);
  const int i_S = in.add(spectrum,
                         spectrum_elems(spectrum_ndim, n_sel, n_omega) * (spectrum_is_complex ? 16 : 8));
  const int i_om = in.add(omega, (size_t)n_omega * 8);
  const int i_ix = in.add(idx, (size_t)n_sel * sizeof(int));
  FFB_TRY(in.upload());
  const size_t n_pairs = spectrum_ndim == 3 ? (size_t)n_sel * n_sel : n_sel;
  const size_t n_out = (size_t)P * P * n_pairs * n_basis * n_basis;
  FFB_TRY(res.alloc(ctx, n_out * 8));
  FFB_TRY(ffbi_decay_amplitudes(ctx, P, n_nops, n_sel, in.d<int>(i_ix), n_basis, n_omega, in.d(i_B),
                                in.d(i_S), spectrum_ndim, spectrum_is_complex, in.d(i_om),
                                res.as<double>()));
  FFB_TRY(ffb_d2h(ctx, out, res.p, n_out * 8));
  FFB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return FFB_OK;
}

int ffb_concatenate_many(ffb_ctx* ctx, int n_seq, int L, int n_lib, int d, int n_nops, int n_basis,
                         int n_omega, const int* indices, const double* lib_control_matrix,
                         const double* lib_total_phases, const double* lib_liouville,
                         const double* lib_propagator, const double* basis, const double* spectrum,
                         int spectrum_ndim, int spectrum_is_complex, const double* omega,
                         double* total_propagator, double* total_propagator_liouville,
                         double* control_matrix, double* filter_function, double* infidelity,
                         const double* tau, double* total_phases) {
  FFB_TRY(enter(ctx));
  FFB_REQUIRE(ctx, !total_phases || (tau && omega),
              "concatenate_many: total phases requested without tau and omega");
  FFB_REQUIRE(ctx, indices && lib_control_matrix && lib_total_phases && lib_liouville &&
                       lib_propagator, "concatenate_many: null input pointer");
  FFB_REQUIRE(ctx, n_seq >= 1 && L >= 1 && n_lib >= 1 && d >= 1 && n_nops >= 1 && n_basis >= 1 &&
                       n_omega >= 1, "concatenate_many: bad shape");
  FFB_REQUIRE(ctx, !infidelity || (spectrum && omega),
              "concatenate_many: infidelity requested without spectrum and omega");
  FFB_REQUIRE(ctx, !total_propagator_liouville || basis,
              "concatenate_many: Liouville representation requested without basis");
  const bool keep = ctx->shadow_next;
  ctx->shadow_next = false;
  for (size_t i = 0; i < (size_t)n_seq * L; ++i)
    FFB_REQUIRE(ctx, indices[i] < n_lib, "concatenate_many: index %d at position %zu out of range "
                "[0, %d)", indices[i], i, n_lib);
  const size_t dd = (size_t)d * d, nn = (size_t)n_basis * n_basis;
  // inputs in one packed upload, results in one (mirrored) device block: a single-sequence call -- the
  // tail of every ff.concatenate -- is bound by driver calls and blocking copies, not by bytes
  PackedUpload in(ctx);
  const int i_om = omega ? in.add(omega, (size_t)n_omega * 8) : -1;
  const int i_ix = in.add(indices, (size_t)n_seq * L * sizeof(int));
  const int i_lb = in.add(lib_control_matrix, (size_t)n_lib * n_nops * n_basis * n_omega * 16);
  const int i_lp = in.add(lib_total_phases, (size_t)n_lib * n_omega * 16);
  const int i_ll = in.add(lib_liouville, (size_t)n_lib * nn * 8);
  const int i_lu = in.add(lib_propagator, (size_t)n_lib * dd * 16);
  int i_sp = -1, i_bs = -1;
  size_t n_inf = 0;
  if (infidelity) {
    FFB_REQUIRE(ctx, spectrum_ndim >= 1 && spectrum_ndim <= 3, "concatenate_many: spectrum_ndim=%d",
                spectrum_ndim);
    i_sp = in.add(spectrum, spectrum_elems(spectrum_ndim, n_nops, n_omega) * (spectrum_is_complex ? 16 : 8));
    n_inf = (size_t)n_seq * (spectrum_ndim == 3 ? (size_t)n_nops * n_nops : n_nops);
  }
  if (total_propagator_liouville) i_bs = in.add(basis, (size_t)n_basis * dd * 16);
  FFB_TRY(in.upload());
  const size_t b_bytes = (size_t)n_seq * n_nops * n_basis * n_omega * 16;
  const size_t f_bytes = (size_t)n_seq * n_nops * n_nops * n_omega * 16;
  const bool need_F = filter_function || infidelity;
  OutputBlock out;
  const int o_U = out.add(total_propagator, (size_t)n_seq * dd * 16);
  const int o_L = total_propagator_liouville ? out.add(total_propagator_liouville, (size_t)n_seq * nn * 16) : -1;
  const int o_ph = total_phases ? out.add(total_phases, (size_t)n_seq * n_omega * 16) : -1;
  const int o_B = out.add(control_matrix, b_bytes);
  const int o_F = need_F ? out.add(filter_function, f_bytes) : -1;
  const int o_I = infidelity ? out.add(infidelity, n_inf * 8) : -1;
  FFB_TRY(out.alloc(ctx));
  FFB_TRY(ffbi_concatenate_many(ctx, n_seq, L, d, n_nops, n_basis, n_omega, in.d<int>(i_ix), in.d(i_lb),
                                in.d(i_lp), in.d(i_ll), in.d(i_lu), out.d(o_U), out.d(o_B),
                                need_F ? out.d(o_F) : nullptr));
  if (infidelity)
    FFB_TRY(ffbi_infidelity(ctx, n_seq, n_nops, n_nops, nullptr, n_omega, out.d(o_F), in.d(i_sp),
                            spectrum_ndim, spectrum_is_complex, in.d(i_om), d, out.d(o_I)));
  if (total_propagator_liouville)
    FFB_TRY(ffbi_liouville(ctx, n_seq, d, n_basis, out.d(o_U), in.d(i_bs), out.d(o_L)));
  if (total_phases)
    for (int s = 0; s < n_seq; ++s)  // tau is a host value, as in the cold pulse pipeline
      FFB_TRY(ffbi_cexp(ctx, n_omega, in.d(i_om), tau[s], out.d(o_ph) + (size_t)s * n_omega * 2));
  FFB_TRY(out.download(ctx, {o_U, o_L, o_ph, o_B, o_F, o_I}, ctx->stream));
  FFB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  out.finish(ctx);
  if (keep) out.retain(ctx, {o_U, o_ph, o_B, filter_function ? o_F : -1});
  return FFB_OK;
}

int ffb_concatenate_pulses(ffb_ctx* ctx, int P, int d, int n_nops, int n_basis, int n_omega,
                           const int* row_of, const double* const* cached, const int* G,
                           const double* const* eigvals, const double* const* eigvecs,
                           const double* const* propagators, const double* const* dt,
                           const double* const* t, const double* const* n_coeffs,
                           const double* n_opers, const double* basis, const double* omega,
                           const double* phases, const double* liouville, int correlations,
                           int filter_function_kind, double* control_matrix,
                           double* filter_function) {
  FFB_TRY(enter(ctx));
  FFB_REQUIRE(ctx, row_of && cached && G && eigvals && eigvecs && propagators && dt && t &&
                       n_coeffs && n_opers && basis && omega && (P == 1 || (phases && liouville)),
              "concatenate_pulses: null input pointer");
  FFB_CHECK_DIM(ctx, d);
  FFB_REQUIRE(ctx, P >= 1 && d >= 1 && d <= 32 && n_nops >= 1 && n_basis >= 1 && n_omega >= 1,
              "concatenate_pulses: bad shape");
  FFB_REQUIRE(ctx, filter_function_kind >= 0 && filter_function_kind <= 2 &&
                       (filter_function_kind == 0 || filter_function),
              "concatenate_pulses: filter_function_kind=%d", filter_function_kind);
  const TraceClock since;
  const int64_t hits0 = ctx->shadow_hits;
  const bool keep_shadow = ctx->shadow_next;
  ctx->shadow_next = false;
  double* const control_matrix_host = control_matrix;
  const size_t dd = (size_t)d * d;
  const size_t row_bytes = (size_t)n_basis * n_omega * 16;
  const size_t pulse_bytes = (size_t)n_nops * row_bytes;
  const bool basis_herm = all_hermitian(basis, n_basis, d);
  if (control_matrix) ffb_shadow_drop_range(ctx, control_matrix, (size_t)(correlations ? P : 1) * pulse_bytes);
  for (int p = 0; p < P; ++p)
    for (int j = 0; j < n_nops; ++j)
      FFB_REQUIRE(ctx, row_of[(size_t)p * n_nops + j] < 0 || cached[p],
                  "concatenate_pulses: pulse %d has cached rows but no array", p);

  // every input in one packed upload, before any launch: omega, the basis, the contraction's phases and
  // Liouville propagators, and for each pulse with missing rows its eigensystem, time steps and the
  // noise operators and coefficients of those rows (seven parts from fill[p] on, in the order
  // ffbi_control_matrix takes them)
  PackedUpload in(ctx);
  const int i_om = in.add(omega, (size_t)n_omega * 8);
  const int i_bs = in.add(basis, (size_t)n_basis * dd * 16);
  const int i_ph = P > 1 ? in.add(phases, (size_t)(P - 1) * n_omega * 16) : -1;
  const int i_Q = P > 1 ? in.add(liouville, (size_t)(P - 1) * n_basis * n_basis * 8) : -1;
  std::vector<std::vector<int>> missing_rows(P);
  std::vector<int> fill(P, -1), herm(P, 0);
  {
    std::vector<std::vector<double>> keep;  // host staging of the subsets, read by in.upload()
    for (int p = 0; p < P; ++p) {
      std::vector<int>& missing = missing_rows[p];
      for (int j = 0; j < n_nops; ++j)
        if (row_of[(size_t)p * n_nops + j] < 0) missing.push_back(j);
      if (missing.empty()) continue;
      const int m = (int)missing.size(), Gp = G[p];
      FFB_REQUIRE(ctx, Gp >= 1 && eigvals[p] && eigvecs[p] && propagators[p] && dt[p] && t[p] &&
                           n_coeffs[p], "concatenate_pulses: pulse %d lacks its diagonalisation", p);
      keep.emplace_back((size_t)m * dd * 2);
      keep.emplace_back((size_t)m * Gp);
      std::vector<double>& ops = keep[keep.size() - 2];
      std::vector<double>& cf = keep[keep.size() - 1];
      for (int i = 0; i < m; ++i) {
        std::memcpy(ops.data() + (size_t)i * dd * 2, n_opers + (size_t)missing[i] * dd * 2, dd * 16);
        std::memcpy(cf.data() + (size_t)i * Gp, n_coeffs[p] + (size_t)missing[i] * Gp, (size_t)Gp * 8);
      }
      herm[p] = (all_hermitian(ops.data(), m, d) ? FFB_HERM_NOPERS : 0) | (basis_herm ? FFB_HERM_BASIS : 0);
      fill[p] = in.add(eigvals[p], (size_t)Gp * d * 8);
      in.add(eigvecs[p], (size_t)Gp * dd * 16);
      in.add(propagators[p], (size_t)Gp * dd * 16);
      in.add(ops.data(), (size_t)m * dd * 16);
      in.add(cf.data(), (size_t)m * Gp * 8);
      in.add(dt[p], (size_t)Gp * 8);
      in.add(t[p], (size_t)(Gp + 1) * 8);
    }
    FFB_TRY(in.upload());
  }
  // Full stack (P pulse slots) when it takes at most a quarter of the device memory: all from-scratch
  // fills are enqueued first, the cached rows are uploaded on the copy stream WHILE the fills run, and
  // one from_atomic launch consumes the stack.  Otherwise (and never for 'correlations', whose result
  // has the size of the stack anyway) two slots [running sum, current pulse]: the sum is updated in
  // place pulse by pulse (from_atomic with P = 2; every thread block of the from_atomic kernels reads
  // exactly the accumulator elements it later writes).
  bool full_stack = correlations != 0 || (size_t)P * pulse_bytes <= ctx->total_mem / 4;
  if (const char* e = getenv("FFB_CONCAT_STACK")) full_stack = correlations != 0 || atoi(e) != 0;
  const int slots = full_stack ? P : std::min(P, 2);
  DevBuf stack, scratch, result;
  FFB_TRY(stack.alloc(ctx, (size_t)slots * pulse_bytes));
  if (full_stack) FFB_TRY(result.alloc(ctx, (size_t)(correlations ? P : 1) * pulse_bytes));
  if (full_stack) {  // the copy stream must not touch pool memory before earlier work is done with it
    FFB_TRY(ensure_copy_stream(ctx));
    FFB_TRY(after(ctx, 0, ctx->stream, ctx->copy_stream));
  }
  cudaStream_t up_stream = full_stack ? ctx->copy_stream : ctx->stream;

  auto upload_cached = [&](int p, char* dst) -> int {
    const int* rows = row_of + (size_t)p * n_nops;
    for (int j = 0; j < n_nops; ++j) {
      if (rows[j] < 0) continue;
      // consecutive rows of the cached array that map to consecutive merged rows go in one copy
      int run = 1;
      while (j + run < n_nops && rows[j + run] == rows[j] + run) ++run;
      // rows that are still mirrored on the device (the pulse's control matrix was computed by this
      // context and its array is alive) are copied device-to-device: no PCIe traffic
      const char* src_host = reinterpret_cast<const char*>(cached[p]) + (size_t)rows[j] * row_bytes;
      const void* mirror = ffb_shadow_lookup(ctx, src_host, (size_t)run * row_bytes);
      FFB_CUDA(ctx, cudaMemcpyAsync(dst + (size_t)j * row_bytes, mirror ? mirror : src_host,
                                    (size_t)run * row_bytes,
                                    mirror ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice,
                                    up_stream));
      j += run - 1;
    }
    return FFB_OK;
  };

  for (int p = 0; p < P; ++p) {
    const int slot = full_stack ? p : std::min(p, 1);
    char* dst = stack.as<char>() + (size_t)slot * pulse_bytes;
    if (!full_stack) FFB_TRY(upload_cached(p, dst));
    const std::vector<int>& missing = missing_rows[p];
    if (!missing.empty()) {
      const int m = (int)missing.size(), i0 = fill[p];
      // one contiguous run of missing rows is written in place, otherwise through scratch
      const bool contiguous = missing.back() - missing.front() + 1 == m;
      double* target = reinterpret_cast<double*>(dst + (size_t)missing.front() * row_bytes);
      if (!contiguous) {
        FFB_TRY(scratch.alloc(ctx, (size_t)m * row_bytes));
        target = scratch.as<double>();
      }
      FFB_TRY(ffbi_control_matrix(ctx, G[p], d, m, n_basis, n_omega, in.d(i0), in.d(i0 + 1), in.d(i0 + 2),
                                  in.d(i_om), in.d(i_bs), in.d(i0 + 3), in.d(i0 + 4), in.d(i0 + 5),
                                  in.d(i0 + 6), herm[p], target));
      if (!contiguous) {
        for (int i = 0; i < m; ++i) {
          int run = 1;
          while (i + run < m && missing[i + run] == missing[i] + run) ++run;
          FFB_CUDA(ctx, cudaMemcpyAsync(dst + (size_t)missing[i] * row_bytes,
                                        scratch.as<char>() + (size_t)i * row_bytes,
                                        (size_t)run * row_bytes, cudaMemcpyDeviceToDevice,
                                        ctx->stream));
          i += run - 1;
        }
      }
    }
    if (!full_stack && p >= 1) {
      FFB_TRY(ffbi_from_atomic(ctx, 2, n_nops, n_basis, n_omega, in.d(i_ph) + (size_t)(p - 1) * n_omega * 2,
                               stack.as<double>(), in.d(i_Q) + (size_t)(p - 1) * n_basis * n_basis, 0, 0,
                               stack.as<double>()));
    }
  }
  const double us_fills = since();
  const double* B_dev = stack.as<double>();
  if (full_stack) {
    // cached rows: issued after the fills were enqueued, so that even a pageable source (staged by the
    // driver while the host thread waits) overlaps them
    for (int p = 0; p < P; ++p) FFB_TRY(upload_cached(p, stack.as<char>() + (size_t)p * pulse_bytes));
    FFB_TRY(after(ctx, 1, ctx->copy_stream, ctx->stream));
    B_dev = result.as<double>();
    // total control matrix: a few row chunks, each downloaded on the copy stream while the next one
    // is computed (the download of the whole result takes about as long as computing it)
    const int n_chunks = (correlations || !control_matrix) ? 1 : std::min(n_nops, 6);
    for (int c = 0; c < n_chunks; ++c) {
      const int j0 = (int)((long long)c * n_nops / n_chunks);
      const int j1 = (int)((long long)(c + 1) * n_nops / n_chunks);
      FFB_TRY(ffbi_from_atomic_rows(ctx, P, n_nops, j0, j1 - j0, n_basis, n_omega,
                                    P > 1 ? in.d(i_ph) : nullptr, stack.as<double>(),
                                    P > 1 ? in.d(i_Q) : nullptr, 0, correlations, result.as<double>()));
      if (n_chunks > 1) {
        FFB_TRY(after(ctx, 0, ctx->stream, ctx->copy_stream));
        FFB_CUDA(ctx, cudaMemcpyAsync(reinterpret_cast<char*>(control_matrix) + (size_t)j0 * row_bytes,
                                      reinterpret_cast<const char*>(B_dev) + (size_t)j0 * row_bytes,
                                      (size_t)(j1 - j0) * row_bytes, cudaMemcpyDeviceToHost,
                                      ctx->copy_stream));
      }
    }
    if (n_chunks > 1) control_matrix = nullptr;  // already on its way
  }
  const int lead = correlations ? P : 1;
  DevBuf F;
  size_t f_bytes = 0;
  if (filter_function_kind) {
    const size_t L = (size_t)lead * n_nops;
    f_bytes = L * L * (filter_function_kind == 2 ? (size_t)n_basis * n_basis : 1) * n_omega * 16;
    FFB_TRY(F.alloc(ctx, f_bytes));
  }
  if (control_matrix && full_stack && filter_function_kind) {
    // download the control matrix on the copy stream while the filter function is computed
    FFB_TRY(after(ctx, 0, ctx->stream, ctx->copy_stream));
    FFB_CUDA(ctx, cudaMemcpyAsync(control_matrix, B_dev, (size_t)lead * pulse_bytes,
                                  cudaMemcpyDeviceToHost, ctx->copy_stream));
  } else if (control_matrix) {
    FFB_TRY(ffb_d2h(ctx, control_matrix, B_dev, (size_t)lead * pulse_bytes));
  }
  if (filter_function_kind) {
    FFB_TRY(ffbi_filter_function(ctx, lead, n_nops, n_basis, n_omega, B_dev,
                                 filter_function_kind == 2, F.as<double>()));
    FFB_TRY(ffb_d2h(ctx, filter_function, F.p, f_bytes));
  }
  const double us_enqueued = since();
  if (full_stack) FFB_CUDA(ctx, cudaStreamSynchronize(ctx->copy_stream));
  const double us_copy = since();
  FFB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (ffb_trace())
    fprintf(stderr, "[ffb trace] concatenate_pulses: P=%d, fills enqueued %.0f us, all enqueued %.0f us, "
            "copy stream done %.0f us, main stream done %.0f us; %lld cached row runs read from device "
            "shadows; %s stack\n", P, us_fills, us_enqueued, us_copy, since(),
            (long long)(ctx->shadow_hits - hits0), full_stack ? "full" : "two-slot");
  if (keep_shadow) {
    if (full_stack && control_matrix_host)
      ffb_shadow_retain(ctx, result, control_matrix_host, (size_t)lead * pulse_bytes,
                        {{0, (size_t)lead * pulse_bytes}});
    if (filter_function_kind) ffb_shadow_retain(ctx, F, filter_function, f_bytes, {{0, f_bytes}});
  }
  return FFB_OK;
}

int ffb_liouville_representation(ffb_ctx* ctx, int n, int d, int n_basis, const double* U,
                                 const double* basis, double* out) {
  FFB_TRY(enter(ctx));
  FFB_REQUIRE(ctx, U && basis && out, "liouville: null pointer");
  FFB_REQUIRE(ctx, n >= 1 && d >= 1 && n_basis >= 1, "liouville: bad shape");
  PackedUpload in(ctx);
  DevBuf O;
  const size_t dd = (size_t)d * d;
  const int i_U = in.add(U, (size_t)n * dd * 16);
  const int i_bs = in.add(basis, (size_t)n_basis * dd * 16);
  FFB_TRY(in.upload());
  const size_t out_bytes = (size_t)n * n_basis * n_basis * 16;
  FFB_TRY(O.alloc(ctx, out_bytes));
  FFB_TRY(ffbi_liouville(ctx, n, d, n_basis, in.d(i_U), in.d(i_bs), O.as<double>()));
  FFB_TRY(ffb_d2h(ctx, out, O.p, out_bytes));
  FFB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return FFB_OK;
}

int ffb_cexp(ffb_ctx* ctx, int n, const double* x, double scale, double* out) {
  FFB_TRY(enter(ctx));
  FFB_REQUIRE(ctx, x && out && n >= 1, "cexp: bad arguments");
  PackedUpload in(ctx);
  DevBuf O;
  const int i_x = in.add(x, (size_t)n * 8);
  FFB_TRY(in.upload());
  FFB_TRY(O.alloc(ctx, (size_t)n * 16));
  FFB_TRY(ffbi_cexp(ctx, n, in.d(i_x), scale, O.as<double>()));
  FFB_TRY(ffb_d2h(ctx, out, O.p, (size_t)n * 16));
  FFB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return FFB_OK;
}

int ffb_cexpm1(ffb_ctx* ctx, int n, const double* x, double* out) {
  FFB_TRY(enter(ctx));
  FFB_REQUIRE(ctx, x && out && n >= 1, "cexpm1: bad arguments");
  PackedUpload in(ctx);
  DevBuf O;
  const int i_x = in.add(x, (size_t)n * 8);
  FFB_TRY(in.upload());
  FFB_TRY(O.alloc(ctx, (size_t)n * 16));
  FFB_TRY(ffbi_cexpm1(ctx, n, in.d(i_x), O.as<double>()));
  FFB_TRY(ffb_d2h(ctx, out, O.p, (size_t)n * 16));
  FFB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return FFB_OK;
}

int ffb_pulse_filter_function(ffb_ctx* ctx, int G, int d, int n_cops, int n_nops, int n_basis,
                              int n_omega, const double* c_opers, const double* c_coeffs,
                              const double* n_opers, const double* n_coeffs, const double* dt,
                              const double* t, const double* basis, const double* omega,
                              const double* spectrum, int spectrum_ndim, int spectrum_is_complex,
                              double* eigvals, double* eigvecs, double* propagators,
                              double* control_matrix, double* filter_function,
                              double* infidelity, double* total_phases,
                              double* total_propagator_liouville) {
  FFB_TRY(enter(ctx));
  FFB_REQUIRE(ctx, c_opers && c_coeffs && n_opers && n_coeffs && dt && basis && omega,
              "pulse pipeline: null input pointer");
  FFB_CHECK_DIM(ctx, d);
  FFB_REQUIRE(ctx, G >= 1 && d >= 1 && d <= 32 && n_cops >= 1 && n_nops >= 1 && n_basis >= 1 &&
                       n_omega >= 1, "pulse pipeline: bad shape");
  FFB_REQUIRE(ctx, !infidelity || spectrum, "pulse pipeline: infidelity requested without spectrum");
  const bool keep = ctx->shadow_next;
  ctx->shadow_next = false;
  const size_t dd = (size_t)d * d;
  const int herm = herm_flags(n_opers, n_nops, basis, n_basis, d);
  FFB_TRY(ensure_copy_stream(ctx));
  // FFB_TRACE=1: host-side timestamps of the pipeline stages on stderr (where does e2e time go?)
  const TraceClock since;
  double us_packed = 0, us_enqueued = 0, us_main = 0;
  std::string marks;
  auto mark = [&](const char* what) {
    if (!ffb_trace()) return;
    char buf[64];
    snprintf(buf, sizeof(buf), " %s@%.0f", what, since());
    marks += buf;
  };
  PackedUpload in(ctx);
  const int i_co = in.add(c_opers, (size_t)n_cops * dd * 16);
  const int i_cc = in.add(c_coeffs, (size_t)n_cops * G * 8);
  const int i_dt = in.add(dt, (size_t)G * 8);
  const int i_no = in.add(n_opers, (size_t)n_nops * dd * 16);
  const int i_nc = in.add(n_coeffs, (size_t)n_nops * G * 8);
  // t == NULL: t = [0, cumsum(dt)] with the sequential summation of np.cumsum (pulse_sequence.py:540-552)
  std::vector<double> t_own;
  if (!t) {
    t_own.resize((size_t)G + 1);
    double acc = 0.0;
    t_own[0] = 0.0;
    for (int g = 0; g < G; ++g) {
      acc += dt[g];
      t_own[(size_t)g + 1] = acc;
    }
    t = t_own.data();
  }
  const int i_ts = in.add(t, (size_t)(G + 1) * 8);
  const int i_bs = in.add(basis, (size_t)n_basis * dd * 16);
  const int i_om = in.add(omega, (size_t)n_omega * 8);
  int i_sp = -1;
  size_t n_inf = 0;
  if (infidelity) {
    FFB_REQUIRE(ctx, spectrum_ndim >= 1 && spectrum_ndim <= 3, "pulse pipeline: spectrum_ndim=%d",
                spectrum_ndim);
    i_sp = in.add(spectrum, spectrum_elems(spectrum_ndim, n_nops, n_omega) * (spectrum_is_complex ? 16 : 8));
    n_inf = spectrum_ndim == 3 ? (size_t)n_nops * n_nops : n_nops;
  }
  FFB_TRY(in.upload());
  us_packed = since();
  const size_t b_bytes = (size_t)n_nops * n_basis * n_omega * 16;
  const size_t f_bytes = (size_t)n_nops * n_nops * n_omega * 16;
  OutputBlock out;
  CopyStreamDrain drain{ctx};  // after `out`: destroyed (drained) before its device block is released
  const int o_ev = out.add(eigvals, (size_t)G * d * 8);
  const int o_V = out.add(eigvecs, (size_t)G * dd * 16);
  const int o_Q = out.add(propagators, (size_t)(G + 1) * dd * 16);
  const int o_ph = total_phases ? out.add(total_phases, (size_t)n_omega * 16) : -1;
  const int o_li = total_propagator_liouville
                       ? out.add(total_propagator_liouville, (size_t)n_basis * n_basis * 16) : -1;
  const int o_B = out.add(control_matrix, b_bytes);
  const int o_F = out.add(filter_function, f_bytes);
  const int o_I = infidelity ? out.add(infidelity, n_inf * 8) : -1;
  FFB_TRY(out.alloc(ctx));
  mark("alloc");
  cudaStream_t cs = ctx->copy_stream;

  // stage 1: everything that does not depend on the control matrix
  FFB_TRY(ffbi_diagonalize(ctx, G, d, n_cops, in.d(i_co), in.d(i_cc), in.d(i_dt), out.d(o_ev),
                           out.d(o_V), out.d(o_Q)));
  if (total_phases)
    FFB_TRY(ffbi_cexp(ctx, n_omega, in.d(i_om), t[G], out.d(o_ph)));  // tau = t[G] (host value)
  if (total_propagator_liouville)
    FFB_TRY(ffbi_liouville(ctx, 1, d, n_basis, out.d(o_Q) + (size_t)G * dd * 2, in.d(i_bs),
                           out.d(o_li)));
  mark("stage1");
  // ... is downloaded on the copy stream WHILE the control-matrix kernel runs -- unless it is so
  // little that the two extra driver calls of the hand-over cost more than the overlap saves
  const size_t early_bytes = (size_t)G * d * 8 + (size_t)(2 * G + 1) * dd * 16 + (size_t)n_omega * 16;
  const size_t out_bytes = (control_matrix ? b_bytes : 0) + (filter_function ? f_bytes : 0);
  const bool overlap = early_bytes + out_bytes >= ((size_t)256 << 10);
  if (overlap) {
    FFB_TRY(after(ctx, 0, ctx->stream, cs));
    FFB_TRY(out.download(ctx, {o_ev, o_V, o_Q, o_ph, o_li}, cs));
  }

  // stage 2: control matrix and filter function in blocks of frequencies; the rows of a finished block
  // are downloaded (strided 2-D copies) while the next block is computed, so that only the last
  // block's download is left after the last kernel (PCIe is the tail of this call: config 3 returns
  // 105 MB, 1.9 ms at 56 GB/s)
  FreqBlocks fb;
  fb.n_blocks = pipeline_blocks(out_bytes, n_omega);
  fb.after_block = [&](int w0, int w1) -> int {
    FFB_TRY(ffbi_filter_function_ld(ctx, 1, n_nops, n_basis, w1 - w0, (size_t)n_omega,
                                    out.d(o_B) + 2 * (size_t)w0, out.d(o_F) + 2 * (size_t)w0));
    if (fb.n_blocks == 1) return FFB_OK;  // one block: whole arrays, copied below
    FFB_TRY(after(ctx, 1, ctx->stream, cs));
    if (control_matrix)
      FFB_TRY(download_freqs(ctx, control_matrix, out.d(o_B), (size_t)n_nops * n_basis, n_omega, w0, w1));
    if (filter_function)
      FFB_TRY(download_freqs(ctx, filter_function, out.d(o_F), (size_t)n_nops * n_nops, n_omega, w0, w1));
    return FFB_OK;
  };
  FFB_TRY(ffbi_control_matrix(ctx, G, d, n_nops, n_basis, n_omega, out.d(o_ev), out.d(o_V),
                              out.d(o_Q), in.d(i_om), in.d(i_bs), in.d(i_no), in.d(i_nc),
                              in.d(i_dt), in.d(i_ts), herm, out.d(o_B), &fb));
  mark("ctrlmat");
  if (overlap && fb.n_blocks == 1) {  // B and F in one copy while the integral runs
    FFB_TRY(after(ctx, 1, ctx->stream, cs));
    FFB_TRY(out.download(ctx, {o_B, o_F}, cs));
  }
  if (infidelity)
    FFB_TRY(ffbi_infidelity(ctx, 1, n_nops, n_nops, nullptr, n_omega, out.d(o_F), in.d(i_sp),
                            spectrum_ndim, spectrum_is_complex, in.d(i_om), d, out.d(o_I)));
  mark("integral");
  if (overlap) {
    FFB_TRY(out.download(ctx, {o_I}, ctx->stream));
  } else {  // small pulse: everything on one stream, as few copies as the layout allows
    FFB_TRY(out.download(ctx, {o_ev, o_V, o_Q, o_ph, o_li, o_B, o_F, o_I}, ctx->stream));
  }
  FFB_TRY(ffb_conv_fetch(ctx));
  if (infidelity) FFB_TRY(ffbi_comm_fetch_error(ctx));
  us_enqueued = since();
  FFB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  us_main = since();
  if (overlap || fb.n_blocks > 1) FFB_CUDA(ctx, cudaStreamSynchronize(cs));  // anything on the copy stream?
  out.finish(ctx);
  FFB_TRY(ffb_conv_check(ctx));
  FFB_TRY(ffbi_comm_check_error(ctx));
  if (ffb_trace())
    fprintf(stderr, "[ffb trace] pulse pipeline: inputs packed+upload enqueued %.0f us, all work enqueued "
            "%.0f us, main stream done %.0f us, copy stream done %.0f us;%s\n", us_packed, us_enqueued,
            us_main, since(), marks.c_str());
  // the eigensystem, control matrix and filter function stay mirrored on the device for the consumers
  // of the pulse's cache (the infidelity and the Liouville matrix are post-processed on the host)
  if (keep) out.retain(ctx, {o_ev, o_V, o_Q, o_ph, control_matrix ? o_B : -1, filter_function ? o_F : -1});
  return FFB_OK;
}

}  // extern "C"
