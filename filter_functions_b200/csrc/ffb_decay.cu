// K6 -- decay amplitudes (numeric.calculate_decay_amplitudes, numeric.py:1194-1337 of the reference):
//     Gamma^{(gh)}_{ab,kl} = 1/(2 pi) trapezoid_w Re( conj(B^{(g)}_{ak}(w)) S_{ab}(w) B^{(h)}_{bl}(w) )
// The reference materialises the integrand '...ko,...o,...lo->...klo' (numeric.py:344-347), an array of
// n_basis^2 n_omega doubles per noise-operator pair (7.4 GB for BASELINE config 3), and then calls
// util.integrate (util.py:880-906).
//
// B200 formulation.  The trapezoid rule is a weighted sum, sum_i f_i u_i with
// u_i = ((w_{i+1} - w_i) + (w_i - w_{i-1})) / 2 (one-sided at the ends), so Gamma is a REAL GEMM over the
// interleaved (re, im) storage of the control matrix:
//     Gamma_kl = sum_{(w,c)} A[k,(w,c)] Y[(w,c),l],   Y[(w,c),l] = raw doubles of B_b[l, w],
//     A[k,(w,0)] = Re(u S conj(B_a[k,w])),  A[k,(w,1)] = -Im(u S conj(B_a[k,w]))
// with K = 2 n_omega.  It runs on the FP64 tensor path (DMMA.8x8x4): M = 8 values of k, N = 8 values of
// l, K = 4 doubles = 2 frequencies.  The summation index may be permuted freely as long as both
// operands use the same permutation, so a lane (r = lane / 4, q = lane % 4) loads the 32 contiguous
// bytes (2 complex frequencies) at w0 + 2 q of its row and feeds them to 4 consecutive DMMAs: every
// load is a full sector, nothing is staged through shared memory and the integrand never exists.
// Arithmetic intensity is n_basis / 4 flop/B: HBM-bound for d <= 4, FP64-bound for d = 16.
//
// The frequency axis is cut into chunks (grid.x) whose partial sums are reduced in a fixed order by
// reduce_kernel (deterministic, no atomics), which also applies the 1 / (2 pi).
#include "ffb_common.cuh"
#include "ffb_device.cuh"

namespace {

// WS[s, w] = u_w S[s, w]: trapezoid weight times spectrum (complex if the spectrum is)
__global__ void __launch_bounds__(256)
weights_kernel(int n_omega, int n_srows, const double* __restrict__ omega,
               const double* __restrict__ spectrum, int is_complex, double* __restrict__ ws) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= n_omega) return;
  double u = 0.0;
  if (n_omega > 1) {
    const double left = w > 0 ? omega[w] - omega[w - 1] : 0.0;
    const double right = w + 1 < n_omega ? omega[w + 1] - omega[w] : 0.0;
    u = 0.5 * (left + right);
  }
  for (int s = 0; s < n_srows; ++s) {
    const size_t e = (size_t)s * n_omega + w;
    if (is_complex) {
      ws[2 * e] = u * spectrum[2 * e];
      ws[2 * e + 1] = u * spectrum[2 * e + 1];
    } else {
      ws[e] = u * spectrum[e];
    }
  }
}

struct DecayParams {
  const double2* B;   // (P, n_nops, n_basis, n_omega)
  const double* ws;   // (n_srows, n_omega) f64 or c128
  const int* idx;     // (n_sel)
  double* partial;    // (n_chunks, n_z, n_basis, n_basis)
  int P, n_nops, n_sel, n_basis, n_omega;
  int spectrum_ndim;  // 1, 2, 3
  int n_pairs;        // n_sel or n_sel^2
  int n_ltiles;       // CTA tiles along l
  int chunk;          // frequencies per chunk, multiple of 8 * WO
};

// Warp tile: TM x TN DMMA tiles (8 TM values of k, 8 TN values of l).  CTA: WK x WL warps tile (k, l),
// WO warps split the chunk's frequencies (small bases) and are reduced through shared memory.
template <int TM, int TN, int WK, int WL, int WO, bool CPLX>
__global__ void __launch_bounds__(WK * WL * WO * 32)
decay_kernel(const DecayParams p) {
  __shared__ double red[WO > 1 ? WK * WL * WO * TM * TN * 64 : 1];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int r = lane >> 2, q = lane & 3;
  const int wo = warp % WO, wl = (warp / WO) % WL, wk = warp / (WO * WL);
  const int kt = blockIdx.y / p.n_ltiles, lt = blockIdx.y % p.n_ltiles;
  const int k0 = (kt * WK + wk) * TM * 8, l0 = (lt * WL + wl) * TN * 8;
  // z -> (g, h, pair); pair -> (a, b, spectrum row)
  const int z = blockIdx.z;
  const int pair = z % p.n_pairs;
  const int gh = z / p.n_pairs;
  const int g = gh / p.P, h = gh % p.P;
  int a, b, srow;
  if (p.spectrum_ndim == 3) {
    a = pair / p.n_sel;
    b = pair % p.n_sel;
    srow = pair;
  } else {
    a = b = pair;
    srow = p.spectrum_ndim == 2 ? pair : 0;
  }
  const size_t row_stride = (size_t)p.n_omega;
  const double2* Ba = p.B + ((size_t)(g * p.n_nops + p.idx[a]) * p.n_basis) * row_stride;
  const double2* Bb = p.B + ((size_t)(h * p.n_nops + p.idx[b]) * p.n_basis) * row_stride;
  const double* ws = p.ws + (size_t)srow * p.n_omega * (CPLX ? 2 : 1);

  double acc[TM][TN][2];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

  const int begin = blockIdx.x * p.chunk;
  const int end = min(p.n_omega, begin + p.chunk);
  const double2 zero2 = make_double2(0.0, 0.0);
  for (int w0 = begin + wo * 8; w0 < end; w0 += 8 * WO) {
    const int w = w0 + 2 * q;
    const bool ok0 = w < end, ok1 = w + 1 < end;
    double2 u0, u1;  // weights of the lane's two frequencies (y unused for real spectra)
    if (CPLX) {
      u0 = ok0 ? reinterpret_cast<const double2*>(ws)[w] : zero2;
      u1 = ok1 ? reinterpret_cast<const double2*>(ws)[w + 1] : zero2;
    } else {
      u0 = make_double2(ok0 ? ws[w] : 0.0, 0.0);
      u1 = make_double2(ok1 ? ws[w + 1] : 0.0, 0.0);
    }
    double av[TM][4], bv[TN][4];
#pragma unroll
    for (int i = 0; i < TM; ++i) {
      const int k = k0 + i * 8 + r;
      const bool kv = k < p.n_basis;
      const double2 x0 = (kv && ok0) ? Ba[(size_t)k * row_stride + w] : zero2;
      const double2 x1 = (kv && ok1) ? Ba[(size_t)k * row_stride + w + 1] : zero2;
      if (CPLX) {  // u S conj(x): real part, minus imaginary part
        av[i][0] = u0.x * x0.x + u0.y * x0.y;
        av[i][1] = u0.x * x0.y - u0.y * x0.x;
        av[i][2] = u1.x * x1.x + u1.y * x1.y;
        av[i][3] = u1.x * x1.y - u1.y * x1.x;
      } else {
        av[i][0] = u0.x * x0.x;
        av[i][1] = u0.x * x0.y;
        av[i][2] = u1.x * x1.x;
        av[i][3] = u1.x * x1.y;
      }
    }
#pragma unroll
    for (int j = 0; j < TN; ++j) {
      const int l = l0 + j * 8 + r;
      const bool lv = l < p.n_basis;
      const double2 y0 = (lv && ok0) ? Bb[(size_t)l * row_stride + w] : zero2;
      const double2 y1 = (lv && ok1) ? Bb[(size_t)l * row_stride + w + 1] : zero2;
      bv[j][0] = y0.x;
      bv[j][1] = y0.y;
      bv[j][2] = y1.x;
      bv[j][3] = y1.y;
    }
#pragma unroll
    for (int s = 0; s < 4; ++s)
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) dmma884(acc[i][j][0], acc[i][j][1], av[i][s], bv[j][s]);
  }

  // ---- epilogue: C fragment (row r, columns 2q, 2q+1) -> partial[chunk][z][k][l]
  double* out = p.partial + ((size_t)blockIdx.x * gridDim.z + z) * p.n_basis * p.n_basis;
  if (WO > 1) {
    double* mine = red + (size_t)warp * TM * TN * 64;
#pragma unroll
    for (int i = 0; i < TM; ++i)
#pragma unroll
      for (int j = 0; j < TN; ++j) {
        mine[(i * TN + j) * 64 + lane * 2] = acc[i][j][0];
        mine[(i * TN + j) * 64 + lane * 2 + 1] = acc[i][j][1];
      }
    __syncthreads();
    if (wo == 0) {
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) {
          double s0 = 0.0, s1 = 0.0;
#pragma unroll
          for (int o = 0; o < WO; ++o) {  // warps (wk, wl, o) are consecutive
            const double* src = red + (size_t)(warp + o) * TM * TN * 64 + (i * TN + j) * 64;
            s0 += src[lane * 2];
            s1 += src[lane * 2 + 1];
          }
          acc[i][j][0] = s0;
          acc[i][j][1] = s1;
        }
    }
  }
  if (wo == 0) {
#pragma unroll
    for (int i = 0; i < TM; ++i) {
      const int k = k0 + i * 8 + r;
#pragma unroll
      for (int j = 0; j < TN; ++j) {
        const int l = l0 + j * 8 + 2 * q;
        if (k < p.n_basis) {
          if (l < p.n_basis) out[(size_t)k * p.n_basis + l] = acc[i][j][0];
          if (l + 1 < p.n_basis) out[(size_t)k * p.n_basis + l + 1] = acc[i][j][1];
        }
      }
    }
  }
}

__global__ void __launch_bounds__(256)
reduce_kernel(int n_chunks, size_t n_out, double scale, const double* __restrict__ partial,
              double* __restrict__ out) {
  const size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n_out) return;
  double s = 0.0;
  for (int c = 0; c < n_chunks; ++c) s += partial[(size_t)c * n_out + e];
  out[e] = s * scale;
}

template <int TM, int TN, int WK, int WL, int WO>
int launch_decay(ffb_ctx* ctx, DecayParams p, int n_z, int cplx, double* out) {
  constexpr int threads = WK * WL * WO * 32;
  const int n_ktiles = ceil_div(p.n_basis, 8 * TM * WK);
  p.n_ltiles = ceil_div(p.n_basis, 8 * TN * WL);
  const long long base = (long long)n_ktiles * p.n_ltiles * n_z;
  // chunks: enough CTAs for ~4 per SM, at least 4 iterations per warp, partials bounded by 256 MiB
  const int min_chunk = 8 * WO * 4;
  long long n_chunks = std::max<long long>(1, (4LL * ctx->sm_count + base - 1) / base);
  n_chunks = std::min<long long>(n_chunks, std::max(1, p.n_omega / min_chunk));
  const size_t n_out = (size_t)n_z * p.n_basis * p.n_basis;
  n_chunks = std::min<long long>(n_chunks, std::max<size_t>(1, ((size_t)256 << 20) / (n_out * 8)));
  p.chunk = ceil_div(ceil_div(p.n_omega, (int)n_chunks), 8 * WO) * 8 * WO;
  const int chunks = ceil_div(p.n_omega, p.chunk);
  FFB_REQUIRE(ctx, n_z <= 65535 && n_ktiles * p.n_ltiles <= 65535,
              "decay amplitudes: too many operator pairs (%d) or basis tiles (%d)", n_z,
              n_ktiles * p.n_ltiles);
  DevBuf partial;
  FFB_TRY(partial.alloc(ctx, (size_t)chunks * n_out * 8));
  p.partial = partial.as<double>();
  dim3 grid(chunks, n_ktiles * p.n_ltiles, n_z);
  if (cplx) decay_kernel<TM, TN, WK, WL, WO, true><<<grid, threads, 0, ctx->stream>>>(p);
  else decay_kernel<TM, TN, WK, WL, WO, false><<<grid, threads, 0, ctx->stream>>>(p);
  FFB_LAUNCHED(ctx);
  const double scale = 1.0 / (2.0 * 3.141592653589793238462643383279502884);
  reduce_kernel<<<(unsigned)ceil_div_sz(n_out, 256), 256, 0, ctx->stream>>>(
      chunks, n_out, scale, partial.as<double>(), out);
  FFB_LAUNCHED(ctx);
  return FFB_OK;
}

}  // namespace

int ffbi_decay_amplitudes(ffb_ctx* ctx, int P, int n_nops, int n_sel, const int* idx_dev,
                          int n_basis, int n_omega, const double* B, const double* spectrum,
                          int spectrum_ndim, int spectrum_is_complex, const double* omega,
                          double* out) {
  FFB_REQUIRE(ctx, spectrum_ndim >= 1 && spectrum_ndim <= 3, "decay amplitudes: spectrum_ndim=%d",
              spectrum_ndim);
  FFB_REQUIRE(ctx, P >= 1 && n_nops >= 1 && n_sel >= 1 && n_basis >= 1 && n_omega >= 1,
              "decay amplitudes: bad shape (P=%d, n_nops=%d, n_sel=%d, n_basis=%d, n_omega=%d)", P,
              n_nops, n_sel, n_basis, n_omega);
  const int n_pairs = spectrum_ndim == 3 ? n_sel * n_sel : n_sel;
  const int n_srows = spectrum_ndim == 1 ? 1 : n_pairs;
  const int n_z = P * P * n_pairs;
  DevBuf ws;
  FFB_TRY(ws.alloc(ctx, (size_t)n_srows * n_omega * (spectrum_is_complex ? 16 : 8)));
  weights_kernel<<<ceil_div(n_omega, 256), 256, 0, ctx->stream>>>(
      n_omega, n_srows, omega, spectrum, spectrum_is_complex, ws.as<double>());
  FFB_LAUNCHED(ctx);
  DecayParams p;
  p.B = reinterpret_cast<const double2*>(B);
  p.ws = ws.as<double>();
  p.idx = idx_dev;
  p.partial = nullptr;
  p.P = P;
  p.n_nops = n_nops;
  p.n_sel = n_sel;
  p.n_basis = n_basis;
  p.n_omega = n_omega;
  p.spectrum_ndim = spectrum_ndim;
  p.n_pairs = n_pairs;
  p.n_ltiles = 1;
  p.chunk = 0;
  if (n_basis <= 8) return launch_decay<1, 1, 1, 1, 4>(ctx, p, n_z, spectrum_is_complex, out);
  if (n_basis <= 16) return launch_decay<2, 2, 1, 1, 4>(ctx, p, n_z, spectrum_is_complex, out);
  if (n_basis <= 32) return launch_decay<4, 4, 1, 1, 4>(ctx, p, n_z, spectrum_is_complex, out);
  return launch_decay<4, 4, 2, 2, 1>(ctx, p, n_z, spectrum_is_complex, out);
}
