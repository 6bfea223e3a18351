// K3 / K5 -- filter functions from control matrices and the infidelity integral.
//
// Replaces numeric.calculate_filter_function (numeric.py:1413-1467),
// numeric.calculate_pulse_correlation_filter_function (numeric.py:1821-1883) and the integrand +
// trapezoid of numeric.infidelity (numeric.py:2318-2320, :259-374, util.py:880-906).
//
// These stages are HBM/L2-bound streaming reductions: omega is the fastest axis of every array, so a
// warp reads 32 consecutive complex128 values (512 B) per row and the basis axis is reduced in
// registers.
#include <algorithm>
#include <cstdlib>

#include "ffb_common.cuh"
#include "ffb_device.cuh"
#include "ffb_peer.cuh"

namespace {

// F[(l), (r), w] = sum_k conj(B[l,k,w]) B[r,k,w];  l, r run over (pulse, noise operator) rows.
// Output index (P = n_pulses, l = (g,a), r = (h,b)): (((g*P + h)*n_nops + a)*n_nops + b)*n_omega + w
template <int RT>
__global__ void __launch_bounds__(256)
ff_fidelity_kernel(int P, int n_nops, int n_basis, int n_omega, size_t ld,
                   const double2* __restrict__ B, double2* __restrict__ F) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= n_omega) return;
  const int L = P * n_nops;
  const int l = blockIdx.y;
  const int r0 = blockIdx.z * RT;
  double2 acc[RT];
#pragma unroll
  for (int i = 0; i < RT; ++i) acc[i] = make_double2(0.0, 0.0);
  const double2* Bl = B + (size_t)l * n_basis * ld + w;  // rows are ld frequencies apart
  for (int k = 0; k < n_basis; ++k) {
    const double2 x = Bl[(size_t)k * ld];
#pragma unroll
    for (int i = 0; i < RT; ++i) {
      const int r = r0 + i;
      if (r < L) {
        const double2 y = B[((size_t)r * n_basis + k) * ld + w];
        // conj(x) * y.  The imaginary part is formed from two ROUNDED products (no FMA contraction), as
        // NumPy forms it: exchanging x and y then flips its sign exactly, so F[r, l] == conj(F[l, r]) bit
        // for bit and the diagonal is exactly real -- properties the reference's results have and its
        // users test for (tests/test_precision.py:549, tests/test_core.py:861 of the reference)
        acc[i].x += x.x * y.x + x.y * y.y;
        acc[i].y += __dsub_rn(__dmul_rn(x.x, y.y), __dmul_rn(x.y, y.x));
      }
    }
  }
  const int g = l / n_nops, a = l % n_nops;
#pragma unroll
  for (int i = 0; i < RT; ++i) {
    const int r = r0 + i;
    if (r < L) {
      const int h = r / n_nops, b = r % n_nops;
      F[((((size_t)g * P + h) * n_nops + a) * n_nops + b) * ld + w] = acc[i];
    }
  }
}

// One-pass Gram variant for long basis sums (n_basis >= 32: d >= 6).  The kernel above re-reads every row
// of B once per group of RT right rows through L2 (config 5, L = 18, n_basis = 256: 18 GB of L2 reads for
// 737 MB of data, 1.6 ms = 7 % of the HBM rate).  Here a CTA owns GRAM_W = 16 frequencies and a PAIR OF
// ROW PANELS (PL = TL * NT rows each; one panel covers all of config 5's 18 rows), streams the panels' rows
// ONCE through a cp.async ring in shared memory ([stage][k][row][16 frequencies]) and every warp accumulates
// one TL x TL register tile of the Gram matrix: 2 TL shared-memory loads per TL^2 complex multiply-adds.
// The two half-warps of a warp take the even and the odd basis elements of a stage for the same 16
// frequencies and are added up by one shuffle at the end (16 instead of 32 frequencies per CTA: twice
// the CTAs, so the last wave wastes half as much).  Only tiles on or above the diagonal are computed, the
// mirror image is written as the conjugate (F is exactly Hermitian, its diagonal exactly real, as in the
// reference where conj(x) x has no imaginary part).  Algorithmic bytes: 16 (L n_basis + L^2) per frequency,
// read / written once; 4 L (L + 1) / 2 n_basis FP64 multiply-adds per frequency -- for L = 18 the FP64
// pipe, not HBM, is the nearer roof (94 us against 120 us).
constexpr int GRAM_W = 16;       // frequencies per CTA
constexpr int GRAM_KC = 8;       // basis elements per stage (4 per half-warp)
__host__ __device__ constexpr int gram_stages(bool tri) { return tri ? 4 : 3; }   // pairs of panels: 64 KB per stage

// acc[i][j] += conj(x_i) y_j for the basis elements kk = 2 m + half of one stage
template <int TL, bool DIAG, bool WHOLE>
__device__ __forceinline__ void gram_stage(const double2* __restrict__ sa, const double2* __restrict__ sb,
                                           int rows_per_k, int n_k, double2 (&acc)[TL][TL]) {
  // WHOLE: all GRAM_KC / 2 basis elements of the stage exist -- no guards, so that the loads of element
  // m + 1 are scheduled under the multiply-adds of element m
#pragma unroll
  for (int m = 0; m < GRAM_KC / 2; ++m) {
    if (WHOLE || m < n_k) {
      double2 x[TL], y[TL];
#pragma unroll
      for (int i = 0; i < TL; ++i) x[i] = sa[(size_t)(2 * m * rows_per_k + i) * GRAM_W];
#pragma unroll
      for (int j = 0; j < TL; ++j) y[j] = sb[(size_t)(2 * m * rows_per_k + j) * GRAM_W];
#pragma unroll
      for (int i = 0; i < TL; ++i)
#pragma unroll
        for (int j = DIAG ? i : 0; j < TL; ++j) {
          acc[i][j].x = fma(x[i].x, y[j].x, acc[i][j].x);
          acc[i][j].x = fma(x[i].y, y[j].y, acc[i][j].x);
          acc[i][j].y = fma(x[i].x, y[j].y, acc[i][j].y);
          acc[i][j].y = fma(-x[i].y, y[j].x, acc[i][j].y);
        }
    }
  }
}

template <int TL, int NT, bool TRI>
__global__ void __launch_bounds__((TRI ? NT * (NT + 1) / 2 : NT * NT) * 32)
ff_gram_kernel(int P, int n_nops, int n_basis, int n_omega, size_t ld, int n_panels,
               const double2* __restrict__ B, double2* __restrict__ F) {
  constexpr int PL = TL * NT;                 // rows per panel
  // warps: one per register tile of the panel pair; TRI (a single panel): the tiles on or above the
  // diagonal only
  constexpr int NW = TRI ? NT * (NT + 1) / 2 : NT * NT;
  constexpr int SLOTS = ((TRI ? 1 : 2) * PL + NW - 1) / NW;   // rows a warp copies per basis element
  constexpr int GRAM_STAGES = gram_stages(TRI);
  extern __shared__ __align__(16) unsigned char gram_smem[];
  const int L = P * n_nops;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int wl = lane & (GRAM_W - 1), half = lane >> 4;
  // panel pair (pa <= pb) of this CTA
  int pa = 0, pb = blockIdx.y;
  while (pb >= n_panels - pa) {
    pb -= n_panels - pa;
    ++pa;
  }
  pb += pa;
  const bool diag_pair = pa == pb;
  const int rows_per_k = (diag_pair ? 1 : 2) * PL;
  const int w0 = blockIdx.x * GRAM_W;
  const int w = min(w0 + wl, n_omega - 1);   // lanes beyond the grid repeat the last frequency
  const size_t stage_elems = (size_t)GRAM_KC * rows_per_k * GRAM_W;
  double2* const ring = reinterpret_cast<double2*>(gram_smem);
  const int n_chunks = (n_basis + GRAM_KC - 1) / GRAM_KC;

  // copies: the warp's rows rr = warp, warp + NW, ... of every basis element; the half-warps take the even
  // and the odd elements.  src[s] walks along the basis axis, one stage (GRAM_KC elements) per call.
  const double2* src[SLOTS];
  int dst[SLOTS];
#pragma unroll
  for (int s = 0; s < SLOTS; ++s) {
    const int rr = warp + s * NW;
    const int l = min((rr < PL ? pa * PL + rr : pb * PL + rr - PL), L - 1);   // padding rows repeat the last row
    src[s] = B + ((size_t)l * n_basis + half) * ld + w;
    dst[s] = rr < rows_per_k ? (half * rows_per_k + rr) * GRAM_W + wl : -1;
  }
  int k_next = 0;   // first basis element of the next stage to be copied
  auto load_stage = [&](int chunk) {
    double2* const st = ring + (size_t)(chunk % GRAM_STAGES) * stage_elems;
    const bool full = k_next + GRAM_KC <= n_basis;
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) {
      if (dst[s] >= 0) {
#pragma unroll
        for (int m = 0; m < GRAM_KC / 2; ++m) {
          // the tail stage repeats the last basis element (never summed)
          const ptrdiff_t koff = full ? 2 * m : min(k_next + 2 * m + half, n_basis - 1) - k_next - half;
          cp_async16(st + dst[s] + (size_t)(2 * m * rows_per_k) * GRAM_W, src[s] + koff * (ptrdiff_t)ld);
        }
      }
      src[s] += (size_t)GRAM_KC * ld;
    }
    k_next += GRAM_KC;
  };

  int ta = warp / NT, tb = warp % NT;
  if (TRI) {
    ta = 0;
    tb = warp;
    while (tb >= NT - ta) {
      tb -= NT - ta;
      ++ta;
    }
    tb += ta;
  }
  const bool active = !diag_pair || ta <= tb;
  const bool diag_tile = diag_pair && ta == tb;
  double2 acc[TL][TL];
#pragma unroll
  for (int i = 0; i < TL; ++i)
#pragma unroll
    for (int j = 0; j < TL; ++j) acc[i][j] = make_double2(0.0, 0.0);

  for (int c = 0; c < GRAM_STAGES - 1; ++c) {
    if (c < n_chunks) load_stage(c);
    cp_async_commit();
  }
  for (int c = 0; c < n_chunks; ++c) {
    cp_async_wait<GRAM_STAGES - 2>();
    __syncthreads();   // chunk c has landed for everybody; everybody is done with chunk c - 1
    if (c + GRAM_STAGES - 1 < n_chunks) load_stage(c + GRAM_STAGES - 1);
    cp_async_commit();
    if (active) {
      const double2* const st = ring + (size_t)(c % GRAM_STAGES) * stage_elems + (size_t)half * rows_per_k * GRAM_W + wl;
      const double2* const sa = st + (size_t)(ta * TL) * GRAM_W;
      const double2* const sb = st + (size_t)((diag_pair ? 0 : PL) + tb * TL) * GRAM_W;
      // basis elements of this stage that exist for this half-warp
      const int left = n_basis - c * GRAM_KC - half;
      const int n_k = left >= GRAM_KC - 1 ? GRAM_KC / 2 : (left + 1) / 2;
      if (n_k == GRAM_KC / 2) {
        if (diag_tile) gram_stage<TL, true, true>(sa, sb, rows_per_k, n_k, acc);
        else gram_stage<TL, false, true>(sa, sb, rows_per_k, n_k, acc);
      } else {
        if (diag_tile) gram_stage<TL, true, false>(sa, sb, rows_per_k, n_k, acc);
        else gram_stage<TL, false, false>(sa, sb, rows_per_k, n_k, acc);
      }
    }
  }
  if (!active) return;
  // even + odd basis elements
#pragma unroll
  for (int i = 0; i < TL; ++i)
#pragma unroll
    for (int j = 0; j < TL; ++j) {
      acc[i][j].x += __shfl_xor_sync(0xffffffffu, acc[i][j].x, 16);
      acc[i][j].y += __shfl_xor_sync(0xffffffffu, acc[i][j].y, 16);
    }
  if (w0 + wl >= n_omega) return;
  auto f_index = [&](int l, int r) -> size_t {
    const int g = l / n_nops, a = l % n_nops, h = r / n_nops, b = r % n_nops;
    return ((((size_t)g * P + h) * n_nops + a) * n_nops + b) * ld + w;
  };
  // half-warp 0 writes the tile, half-warp 1 its mirror image
#pragma unroll
  for (int i = 0; i < TL; ++i)
#pragma unroll
    for (int j = 0; j < TL; ++j) {
      const int l = pa * PL + ta * TL + i, r = pb * PL + tb * TL + j;
      if (l >= L || r >= L || (diag_tile && j < i)) continue;
      if (l == r) {
        if (half == 0) F[f_index(l, l)] = make_double2(acc[i][j].x, 0.0);
      } else if (half == 0) {
        F[f_index(l, r)] = acc[i][j];
      } else {
        F[f_index(r, l)] = make_double2(acc[i][j].x, -acc[i][j].y);
      }
    }
}

template <int TL, int NT, bool TRI>
int launch_gram(ffb_ctx* ctx, int P, int n_nops, int n_basis, int n_omega, size_t ld, const double* B,
                double* F) {
  constexpr int PL = TL * NT;
  const int L = P * n_nops;
  const int n_panels = ceil_div(L, PL);
  const size_t smem = (size_t)gram_stages(TRI) * (TRI ? 1 : 2) * GRAM_KC * PL * GRAM_W * 16;
  FFB_TRY(ffb_func_smem(ctx, ff_gram_kernel<TL, NT, TRI>, smem));
  dim3 grid(ceil_div(n_omega, GRAM_W), n_panels * (n_panels + 1) / 2);
  ff_gram_kernel<TL, NT, TRI><<<grid, (TRI ? NT * (NT + 1) / 2 : NT * NT) * 32, smem, ctx->stream>>>(
      P, n_nops, n_basis, n_omega, ld, n_panels, reinterpret_cast<const double2*>(B),
      reinterpret_cast<double2*>(F));
  FFB_LAUNCHED(ctx);
  return FFB_OK;
}

// Single panel (L <= 18 rows: every first-order filter function with up to 18 noise operators).  The
// 6 x 6 tile of the kernel above needs 244 registers, which leaves 6 warps per SM -- 1.5 per scheduler, and
// an FP64 instruction keeps its scheduler's dispatch port for 2 cycles: the FP64 pipe sat at 32 %
// (profiles/r02_ncu_ff_gram.txt).  Here a warp owns a 6 x 3 tile (x: 6 rows, y: 3 rows; ~130 registers),
// so that all 12 tiles on or above the diagonal of an 18-row panel are resident as 12 warps, 3 per
// scheduler; tiles the diagonal crosses skip the pairs below it at compile time (kinds LEFT / RIGHT),
// and the warp -> tile table spreads the three kinds evenly over the schedulers (warp % 4).
enum { GRAM_FULL = 0, GRAM_LEFT = 1, GRAM_RIGHT = 2 };

template <int KIND, bool WHOLE, int KC, int GW>
__device__ __forceinline__ void gram18_stage(const double2* __restrict__ sa, const double2* __restrict__ sb,
                                             int rows_per_k, int n_k, double2 (&acc)[6][3]) {
  // WHOLE: all KC / NPH basis elements of the stage exist -- no guards, so that the loads of element
  // m + 1 are scheduled under the multiply-adds of element m
#pragma unroll
  constexpr int NPH = 32 / GW;
  for (int m = 0; m < KC / NPH; ++m) {
    if (WHOLE || m < n_k) {
      double2 x[6], y[3];
#pragma unroll
      for (int i = 0; i < 6; ++i) x[i] = sa[(size_t)(NPH * m * rows_per_k + i) * GW];
#pragma unroll
      for (int j = 0; j < 3; ++j) y[j] = sb[(size_t)(NPH * m * rows_per_k + j) * GW];
#pragma unroll
      for (int i = 0; i < 6; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) {
          if (KIND == GRAM_LEFT && i > j) continue;
          if (KIND == GRAM_RIGHT && i > j + 3) continue;
          acc[i][j].x = fma(x[i].x, y[j].x, acc[i][j].x);
          acc[i][j].x = fma(x[i].y, y[j].y, acc[i][j].x);
          acc[i][j].y = fma(x[i].x, y[j].y, acc[i][j].y);
          acc[i][j].y = fma(-x[i].y, y[j].x, acc[i][j].y);
        }
    }
  }
}

// (ta, tb) of the warps of an 18-row panel: per scheduler F F L | F F L | F R L | F R R
__constant__ unsigned char GRAM18_TILES[12][2] = {{0, 2}, {0, 4}, {1, 4}, {1, 5}, {0, 3}, {0, 5},
                                                  {0, 1}, {1, 3}, {0, 0}, {1, 2}, {2, 4}, {2, 5}};

template <int NTA, int KC, int STAGES, int GW>
__global__ void __launch_bounds__(NTA * (NTA + 1) * 32, 1)
ff_gram18_kernel(int P, int n_nops, int n_basis, int n_omega, size_t ld, const double2* __restrict__ B,
                 double2* __restrict__ F) {
  constexpr int PL = 6 * NTA;
  constexpr int NW = NTA * (NTA + 1);
  constexpr int SLOTS = (PL + NW - 1) / NW;
  extern __shared__ __align__(16) unsigned char gram_smem[];
  const int L = P * n_nops;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int NPH = 32 / GW;               // phases of the basis sum inside a warp (GW frequencies each)
  const int wl = lane & (GW - 1), half = lane / GW;
  const int w0 = blockIdx.x * GW;
  const int w = min(w0 + wl, n_omega - 1);
  constexpr size_t stage_elems = (size_t)KC * PL * GW;
  double2* const ring = reinterpret_cast<double2*>(gram_smem);
  const int n_chunks = (n_basis + KC - 1) / KC;
  const ptrdiff_t ld2 = NPH * (ptrdiff_t)ld;

  const double2* src[SLOTS];
  int dst[SLOTS];
#pragma unroll
  for (int s = 0; s < SLOTS; ++s) {
    const int rr = warp + s * NW;
    src[s] = B + ((size_t)min(rr, L - 1) * n_basis + half) * ld + w;   // padding rows repeat the last row
    dst[s] = rr < PL ? (half * PL + rr) * GW + wl : -1;
  }
  int k_next = 0;
  auto load_stage = [&](int chunk) {
    double2* const st = ring + (size_t)(chunk % STAGES) * stage_elems;
    if (k_next + KC <= n_basis) {
#pragma unroll
      for (int s = 0; s < SLOTS; ++s)
        if (dst[s] >= 0) {
          const double2* q = src[s];
#pragma unroll
          for (int m = 0; m < KC / NPH; ++m, q += ld2)
            cp_async16(st + dst[s] + (size_t)(NPH * m * PL) * GW, q);
        }
    } else {   // tail stage: repeats the last basis element (never summed)
#pragma unroll
      for (int s = 0; s < SLOTS; ++s)
        if (dst[s] >= 0) {
#pragma unroll
          for (int m = 0; m < KC / NPH; ++m) {
            const ptrdiff_t koff = min(k_next + NPH * m + half, n_basis - 1) - k_next - half;
            cp_async16(st + dst[s] + (size_t)(NPH * m * PL) * GW, src[s] + koff * (ptrdiff_t)ld);
          }
        }
    }
#pragma unroll
    for (int s = 0; s < SLOTS; ++s) src[s] += (ptrdiff_t)KC * (ptrdiff_t)ld;
    k_next += KC;
  };

  int ta, tb;
  if (NTA == 3) {
    ta = GRAM18_TILES[warp][0];
    tb = GRAM18_TILES[warp][1];
  } else {   // tiles (ta, tb >= 2 ta) in order
    ta = 0;
    tb = warp;
    while (tb >= 2 * (NTA - ta)) {
      tb -= 2 * (NTA - ta);
      ++ta;
    }
    tb += 2 * ta;
  }
  const int kind = tb == 2 * ta ? GRAM_LEFT : tb == 2 * ta + 1 ? GRAM_RIGHT : GRAM_FULL;
  double2 acc[6][3];
#pragma unroll
  for (int i = 0; i < 6; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) acc[i][j] = make_double2(0.0, 0.0);

  for (int c = 0; c < STAGES - 1; ++c) {
    if (c < n_chunks) load_stage(c);
    cp_async_commit();
  }
  for (int c = 0; c < n_chunks; ++c) {
    cp_async_wait<STAGES - 2>();
    __syncthreads();   // chunk c has landed for everybody; everybody is done with chunk c - 1
    if (c + STAGES - 1 < n_chunks) load_stage(c + STAGES - 1);
    cp_async_commit();
    const double2* const st = ring + (size_t)(c % STAGES) * stage_elems + (size_t)half * PL * GW + wl;
    const double2* const sa = st + (size_t)(ta * 6) * GW;
    const double2* const sb = st + (size_t)(tb * 3) * GW;
    const int left = n_basis - c * KC - half;   // elements kk = NPH m + half of this chunk that exist
    const int n_k = left >= KC - NPH + 1 ? KC / NPH : max(0, (left + NPH - 1) / NPH);
    if (n_k == KC / NPH) {
      if (kind == GRAM_FULL) gram18_stage<GRAM_FULL, true, KC, GW>(sa, sb, PL, n_k, acc);
      else if (kind == GRAM_LEFT) gram18_stage<GRAM_LEFT, true, KC, GW>(sa, sb, PL, n_k, acc);
      else gram18_stage<GRAM_RIGHT, true, KC, GW>(sa, sb, PL, n_k, acc);
    } else {
      if (kind == GRAM_FULL) gram18_stage<GRAM_FULL, false, KC, GW>(sa, sb, PL, n_k, acc);
      else if (kind == GRAM_LEFT) gram18_stage<GRAM_LEFT, false, KC, GW>(sa, sb, PL, n_k, acc);
      else gram18_stage<GRAM_RIGHT, false, KC, GW>(sa, sb, PL, n_k, acc);
    }
  }
#pragma unroll
  for (int i = 0; i < 6; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) {
#pragma unroll
      for (int off = 16; off >= GW; off >>= 1) {   // the NPH partial sums, in a fixed order
        acc[i][j].x += __shfl_xor_sync(0xffffffffu, acc[i][j].x, off);
        acc[i][j].y += __shfl_xor_sync(0xffffffffu, acc[i][j].y, off);
      }
    }
  if (w0 + wl >= n_omega) return;
  auto f_index = [&](int l, int r) -> size_t {
    const int g = l / n_nops, a = l % n_nops, h = r / n_nops, b = r % n_nops;
    return ((((size_t)g * P + h) * n_nops + a) * n_nops + b) * ld + w;
  };
  // phase 0 writes the tile, phase 1 its mirror image
#pragma unroll
  for (int i = 0; i < 6; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const int l = ta * 6 + i, r = tb * 3 + j;
      if (l > r || r >= L) continue;
      if (l == r) {
        if (half == 0) F[f_index(l, l)] = make_double2(acc[i][j].x, 0.0);
      } else if (half == 0) {
        F[f_index(l, r)] = acc[i][j];
      } else if (half == 1) {
        F[f_index(r, l)] = make_double2(acc[i][j].x, -acc[i][j].y);
      }
    }
}

template <int NTA>
int launch_gram18(ffb_ctx* ctx, int P, int n_nops, int n_basis, int n_omega, size_t ld, const double* B,
                  double* F) {
  // 16 basis elements per stage, double buffered (72 KB per stage for 18 rows: enough bytes in flight per SM
  // to cover the HBM latency; the per-stage bookkeeping and the block barrier are paid half as often)
  // (8 frequencies per CTA -- four quarter-warps sharing the basis sum, 8.4 waves instead of 4.2 -- was
  // measured slower: 0.283 vs 0.251 ms on config 5; the per-CTA prologue / epilogue is paid twice as often)
  constexpr int GW = GRAM_W, KC = 16, STAGES = 2;
  const size_t smem = (size_t)STAGES * KC * 6 * NTA * GW * 16;
  FFB_TRY((ffb_func_smem(ctx, ff_gram18_kernel<NTA, KC, STAGES, GW>, smem)));
  ff_gram18_kernel<NTA, KC, STAGES, GW><<<ceil_div(n_omega, GW), NTA * (NTA + 1) * 32, smem, ctx->stream>>>(
      P, n_nops, n_basis, n_omega, ld, reinterpret_cast<const double2*>(B), reinterpret_cast<double2*>(F));
  FFB_LAUNCHED(ctx);
  return FFB_OK;
}

// the Gram kernel pays when the basis sum is long and there are several rows to pair up
bool gram_eligible(int L, int n_basis) {
  static const bool off = getenv("FFB_FF_GRAM") && atoi(getenv("FFB_FF_GRAM")) == 0;
  return !off && n_basis >= 32 && L >= 4 && L <= 4096;
}

int run_gram(ffb_ctx* ctx, int P, int n_nops, int n_basis, int n_omega, size_t ld, const double* B,
             double* F) {
  const int L = P * n_nops;
  // one panel: 4 x 4 tiles on or above the diagonal (3 / 6 / 10 warps) up to 16 rows -- HBM-bound there --,
  // 6 x 3 tiles (12 warps) for 17 or 18 rows; pairs of 16-row panels beyond
  if (L <= 8) return launch_gram<4, 2, true>(ctx, P, n_nops, n_basis, n_omega, ld, B, F);
  if (L <= 12) return launch_gram<4, 3, true>(ctx, P, n_nops, n_basis, n_omega, ld, B, F);
  if (L <= 16) return launch_gram<4, 4, true>(ctx, P, n_nops, n_basis, n_omega, ld, B, F);
  if (L <= 18) return launch_gram18<3>(ctx, P, n_nops, n_basis, n_omega, ld, B, F);
  return launch_gram<4, 4, false>(ctx, P, n_nops, n_basis, n_omega, ld, B, F);
}

// F[(l), (r), k, m, w] = conj(B[l,k,w]) B[r,m,w]   (write-bound outer product)
__global__ void __launch_bounds__(256)
ff_generalized_kernel(int P, int n_nops, int n_basis, int n_omega, const double2* __restrict__ B,
                      double2* __restrict__ F) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= n_omega) return;
  const int l = blockIdx.y / n_basis, k = blockIdx.y % n_basis;
  const int r = blockIdx.z;
  const double2 x = B[((size_t)l * n_basis + k) * n_omega + w];
  const int g = l / n_nops, a = l % n_nops;
  const int h = r / n_nops, b = r % n_nops;
  double2* dst = F + ((((((size_t)g * P + h) * n_nops + a) * n_nops + b) * n_basis + k) * n_basis) *
                         (size_t)n_omega + w;
  const double2* Br = B + (size_t)r * n_basis * n_omega + w;
  for (int m = 0; m < n_basis; ++m) {
    const double2 y = Br[(size_t)m * n_omega];
    dst[(size_t)m * n_omega] = make_double2(x.x * y.x + x.y * y.y,
                                            __dsub_rn(__dmul_rn(x.x, y.y), __dmul_rn(x.y, y.x)));
  }
}

// One block per output element: trapezoid of Re(F S) over omega, warp-shuffle + shared reduction in a
// fixed order (deterministic).
__global__ void __launch_bounds__(1024)
infidelity_kernel(int n_nops, int n_sel, const int* __restrict__ idx, int n_omega,
                  const double2* __restrict__ F, const double* __restrict__ spectrum,
                  int spectrum_ndim, int spectrum_is_complex, const double* __restrict__ omega,
                  double norm, double* __restrict__ out, PeerReduce peers) {
  __shared__ double warp_sums[32];
  const int o = blockIdx.x;  // output index
  int lead, a, b;
  if (spectrum_ndim == 3) {
    lead = o / (n_sel * n_sel);
    a = (o / n_sel) % n_sel;
    b = o % n_sel;
  } else {
    lead = o / n_sel;
    a = b = o % n_sel;
  }
  const int ia = idx ? idx[a] : a, ib = idx ? idx[b] : b;  // idx == nullptr: all operators, in order
  const double2* Frow = F + (((size_t)lead * n_nops + ia) * n_nops + ib) * n_omega;
  size_t s_off = 0;
  if (spectrum_ndim == 2) s_off = (size_t)a * n_omega;
  if (spectrum_ndim == 3) s_off = ((size_t)a * n_sel + b) * n_omega;
  auto integrand = [&](int i) -> double {
    const double2 f = Frow[i];
    if (spectrum_is_complex) {
      const double2 s = reinterpret_cast<const double2*>(spectrum)[s_off + i];
      return f.x * s.x - f.y * s.y;
    }
    return f.x * spectrum[s_off + i];
  };
  double sum = 0.0;
  for (int i = threadIdx.x; i < n_omega - 1; i += blockDim.x) {
    sum += (integrand(i + 1) + integrand(i)) * (omega[i + 1] - omega[i]);
  }
  for (int off = 16; off > 0; off >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, off);
  if ((threadIdx.x & 31) == 0) warp_sums[threadIdx.x >> 5] = sum;
  __syncthreads();
  if (threadIdx.x == 0) {
    double total = 0.0;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) total += warp_sums[i];
    // frequency-sharded run: the partial integral of this rank's block is exchanged with the peers
    // over NVLink right here (peers.world == 1 otherwise)
    out[o] = peer_allreduce_slot(peers, o, total / 2.0 / norm);
  }
}

// Few outputs on a long frequency grid (one pulse: 3-36 integrals over 1e4-5e4 frequencies): one block
// per output leaves the machine idle and walks the grid with one block's worth of loads in flight
// (9 us for config 2).  Here an output is cut into chunks of INFID_CHUNK intervals, one block each; a
// block writes its partial sum and takes a ticket, and the block that draws the last ticket adds the
// partial sums up IN CHUNK ORDER (deterministic) and resets the ticket counter for the next launch.
constexpr int INFID_CHUNK = 1024;
constexpr int INFID_MAX_CHUNKS = 64;
constexpr int INFID_MAX_OUT = 64;  // more outputs than this fill the machine with one block each
__global__ void __launch_bounds__(256)
infidelity_chunked_kernel(int n_nops, int n_sel, const int* __restrict__ idx, int n_omega,
                          const double2* __restrict__ F, const double* __restrict__ spectrum,
                          int spectrum_ndim, int spectrum_is_complex,
                          const double* __restrict__ omega, double norm, int n_chunks,
                          double* __restrict__ partial, unsigned* __restrict__ tickets,
                          double* __restrict__ out, PeerReduce peers) {
  __shared__ double warp_sums[8];
  __shared__ bool last;
  const int o = blockIdx.x, chunk = blockIdx.y;
  int lead, a, b;
  if (spectrum_ndim == 3) {
    lead = o / (n_sel * n_sel);
    a = (o / n_sel) % n_sel;
    b = o % n_sel;
  } else {
    lead = o / n_sel;
    a = b = o % n_sel;
  }
  const int ia = idx ? idx[a] : a, ib = idx ? idx[b] : b;
  const double2* Frow = F + (((size_t)lead * n_nops + ia) * n_nops + ib) * n_omega;
  size_t s_off = 0;
  if (spectrum_ndim == 2) s_off = (size_t)a * n_omega;
  if (spectrum_ndim == 3) s_off = ((size_t)a * n_sel + b) * n_omega;
  auto integrand = [&](int i) -> double {
    const double2 f = Frow[i];
    if (spectrum_is_complex) {
      const double2 s = reinterpret_cast<const double2*>(spectrum)[s_off + i];
      return f.x * s.x - f.y * s.y;
    }
    return f.x * spectrum[s_off + i];
  };
  const int per = (n_omega - 1 + n_chunks - 1) / n_chunks;  // intervals per chunk
  const int i0 = chunk * per, i1 = min(n_omega - 1, i0 + per);
  double sum = 0.0;
  for (int i = i0 + threadIdx.x; i < i1; i += blockDim.x)
    sum += (integrand(i + 1) + integrand(i)) * (omega[i + 1] - omega[i]);
  for (int off = 16; off > 0; off >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, off);
  if ((threadIdx.x & 31) == 0) warp_sums[threadIdx.x >> 5] = sum;
  __syncthreads();
  if (threadIdx.x == 0) {
    double total = 0.0;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) total += warp_sums[i];
    partial[(size_t)o * n_chunks + chunk] = total;
    __threadfence();
    last = atomicAdd(&tickets[o], 1u) == (unsigned)(n_chunks - 1);
    if (last) {
      __threadfence();
      double all = 0.0;
      for (int c = 0; c < n_chunks; ++c)
        all += reinterpret_cast<volatile double*>(partial)[(size_t)o * n_chunks + c];
      tickets[o] = 0;  // ready for the next launch (launches on one stream are ordered)
      out[o] = peer_allreduce_slot(peers, o, all / 2.0 / norm);  // sum over the frequency shards
    }
  }
}

}  // namespace

int ffbi_filter_function(ffb_ctx* ctx, int P, int n_nops, int n_basis, int n_omega,
                         const double* B, int generalized, double* F) {
  FFB_REQUIRE(ctx, P >= 1 && n_nops >= 1 && n_basis >= 1 && n_omega >= 1,
              "filter function: bad shape (P=%d, n_nops=%d, n_basis=%d, n_omega=%d)", P, n_nops,
              n_basis, n_omega);
  const int L = P * n_nops;
  FFB_REQUIRE(ctx, L <= 65535 && (!generalized || (long long)L * n_basis <= 65535 * 1LL),
              "filter function: too many rows (%d x %d)", L, n_basis);
  const int wt = ceil_div(n_omega, 256);
  if (!generalized && gram_eligible(L, n_basis))
    return run_gram(ctx, P, n_nops, n_basis, n_omega, (size_t)n_omega, B, F);
  if (!generalized) {
    constexpr int RT = 4;
    dim3 grid(wt, L, ceil_div(L, RT));
    ff_fidelity_kernel<RT><<<grid, 256, 0, ctx->stream>>>(
        P, n_nops, n_basis, n_omega, (size_t)n_omega, reinterpret_cast<const double2*>(B),
        reinterpret_cast<double2*>(F));
  } else {
    dim3 grid(wt, L * n_basis, L);
    ff_generalized_kernel<<<grid, 256, 0, ctx->stream>>>(
        P, n_nops, n_basis, n_omega, reinterpret_cast<const double2*>(B),
        reinterpret_cast<double2*>(F));
  }
  FFB_LAUNCHED(ctx);
  return FFB_OK;
}

int ffbi_filter_function_ld(ffb_ctx* ctx, int P, int n_nops, int n_basis, int n_omega, size_t ld,
                            const double* B, double* F) {
  FFB_REQUIRE(ctx, P >= 1 && n_nops >= 1 && n_basis >= 1 && n_omega >= 1 && ld >= (size_t)n_omega,
              "filter function: bad shape (P=%d, n_nops=%d, n_basis=%d, n_omega=%d)", P, n_nops,
              n_basis, n_omega);
  const int L = P * n_nops;
  FFB_REQUIRE(ctx, L <= 65535, "filter function: too many rows (%d)", L);
  if (gram_eligible(L, n_basis)) return run_gram(ctx, P, n_nops, n_basis, n_omega, ld, B, F);
  constexpr int RT = 4;
  dim3 grid(ceil_div(n_omega, 256), L, ceil_div(L, RT));
  ff_fidelity_kernel<RT><<<grid, 256, 0, ctx->stream>>>(
      P, n_nops, n_basis, n_omega, ld, reinterpret_cast<const double2*>(B),
      reinterpret_cast<double2*>(F));
  FFB_LAUNCHED(ctx);
  return FFB_OK;
}

int ffbi_infidelity(ffb_ctx* ctx, int n_lead, int n_nops, int n_sel, const int* idx_dev,
                    int n_omega, const double* F, const double* spectrum, int spectrum_ndim,
                    int spectrum_is_complex, const double* omega, int d, double* out) {
  FFB_REQUIRE(ctx, spectrum_ndim >= 1 && spectrum_ndim <= 3, "infidelity: spectrum_ndim=%d",
              spectrum_ndim);
  FFB_REQUIRE(ctx, n_lead >= 1 && n_sel >= 1 && n_omega >= 1 && d >= 1,
              "infidelity: bad shape (n_lead=%d, n_sel=%d, n_omega=%d, d=%d)", n_lead, n_sel,
              n_omega, d);
  const int n_out = n_lead * (spectrum_ndim == 3 ? n_sel * n_sel : n_sel);
  const double norm = 2.0 * 3.141592653589793238462643383279502884 * d;
  // frequency-sharded run (ffb_comm_reduce_infidelity): the exchange is the epilogue of the kernel when
  // the outputs fit one exchange window, a stand-alone all-reduce behind it otherwise
  const bool reduce = ctx->comm.reduce_infidelity && ctx->comm.connected && ctx->comm.world > 1;
  const bool fused = reduce && n_out <= FFB_PEER_SLOTS;
  static const bool chunked_ok = !(getenv("FFB_INFIDELITY_CHUNKED") && atoi(getenv("FFB_INFIDELITY_CHUNKED")) == 0);
  if (chunked_ok && n_out <= INFID_MAX_OUT && n_omega - 1 >= 2 * INFID_CHUNK) {
    const int n_chunks = std::min(INFID_MAX_CHUNKS, ceil_div(n_omega - 1, INFID_CHUNK));
    if (!ctx->infid_scratch) {  // partial sums and ticket counters, allocated (and zeroed) once
      FFB_CUDA(ctx, cudaMalloc(&ctx->infid_scratch,
                               (size_t)INFID_MAX_OUT * (INFID_MAX_CHUNKS * sizeof(double) + sizeof(unsigned))));
      FFB_CUDA(ctx, cudaMemsetAsync(ctx->infid_scratch, 0,
                                    (size_t)INFID_MAX_OUT * (INFID_MAX_CHUNKS * sizeof(double) + sizeof(unsigned)),
                                    ctx->stream));
    }
    double* partial = static_cast<double*>(ctx->infid_scratch);
    unsigned* tickets = reinterpret_cast<unsigned*>(partial + (size_t)INFID_MAX_OUT * INFID_MAX_CHUNKS);
    infidelity_chunked_kernel<<<dim3(n_out, n_chunks), 256, 0, ctx->stream>>>(
        n_nops, n_sel, idx_dev, n_omega, reinterpret_cast<const double2*>(F), spectrum, spectrum_ndim,
        spectrum_is_complex, omega, norm, n_chunks, partial, tickets, out,
        fused ? ffbi_peer_next(ctx) : PeerReduce());
    FFB_LAUNCHED(ctx);
    return FFB_OK;
  }
  const int threads = n_omega > 4096 ? 1024 : 256;
  infidelity_kernel<<<n_out, threads, 0, ctx->stream>>>(
      n_nops, n_sel, idx_dev, n_omega, reinterpret_cast<const double2*>(F), spectrum,
      spectrum_ndim, spectrum_is_complex, omega, norm, out, fused ? ffbi_peer_next(ctx) : PeerReduce());
  FFB_LAUNCHED(ctx);
  if (reduce && !fused) FFB_TRY(ffbi_allreduce_sum(ctx, out, n_out));
  return FFB_OK;
}
