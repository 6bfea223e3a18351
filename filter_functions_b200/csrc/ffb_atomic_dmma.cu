// K4b -- calculate_control_matrix_from_atomic (numeric.py:621-704 of the reference) for LARGE operator
// bases (n_basis >= 32, i.e. d >= 6; config 5: d = 16, n_basis = 256) on the FP64 tensor path.
//
//     out[j, l, w] = B^{(0)}[j, l, w] + sum_{g >= 1} sum_k  Q^{(g-1)}[k, l] * phi_{g-1}(w) B^{(g)}[j, k, w]
//
// Per noise operator j this is a real (n_basis x n_basis) x complex (n_basis x n_omega) GEMM per
// constituent pulse: 4 n_basis^2 flops against 16 n_basis bytes per (pulse, j, w) -- n_basis / 4 flop/B,
// FP64-bound from n_basis ~ 32 (SURVEY.md 8d), which is where the thread-per-frequency kernel of
// ffb_concat.cu (HBM-bound regime, d <= 4) stops being adequate.
//
// Mapping on DMMA.8x8x4: M = 8 output basis indices l, N = 8 frequencies, K = 4 input basis indices k.
//   A fragment (lane 4 r + q): Q[k0 + q][l0 + r]  -- pre-arranged in fragment order by
//       qstream_kernel, streamed through shared memory with a double-buffered cp.async pipeline and
//       shared by all warps of the CTA (each warp owns 8 other frequencies);
//   B fragment (lane 4 r + q): phi(w0 + r) B^{(g)}[j, k0 + q, w0 + r] -- one 16-byte cp.async per lane
//       (8 lanes cover 128 contiguous bytes) into the warp's own shared-memory tile, one stage ahead
//       of its use; phase factor applied in registers, real and imaginary part feed two accumulator
//       sets;
//   C fragment: out[l0 + r][w0 + 2 q + {0, 1}] -- initialised from B^{(0)}, stored as 32 contiguous
//       bytes per lane.
// A warp keeps LT l-tiles (8 LT basis indices) x 8 frequencies in registers and sweeps k for all
// constituent pulses.
#include <cstdlib>

#include "ffb_common.cuh"
#include "ffb_device.cuh"

namespace {

// qstream[g][ls][s][lt][lane] = Q_g[4 s + lane % 4][(ls * LT + lt) * 8 + lane / 4]   (0 outside)
__global__ void __launch_bounds__(256)
qstream_kernel(int n_q, int n_basis, int n_ls, int n_ksteps, int LT, const double* __restrict__ Q,
               double* __restrict__ qstream) {
  const size_t total = (size_t)n_q * n_ls * n_ksteps * LT * 32;
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (size_t)gridDim.x * blockDim.x) {
    const int lane = (int)(idx % 32);
    size_t rem = idx / 32;
    const int lt = (int)(rem % LT);
    rem /= LT;
    const int s = (int)(rem % n_ksteps);
    rem /= n_ksteps;
    const int ls = (int)(rem % n_ls);
    const int g = (int)(rem / n_ls);
    const int k = 4 * s + (lane & 3);
    const int l = (ls * LT + lt) * 8 + (lane >> 2);
    qstream[idx] = (k < n_basis && l < n_basis) ? Q[((size_t)g * n_basis + k) * n_basis + l] : 0.0;
  }
}

struct AtomicParams {
  const double2* phases;   // (P-1, n_omega)
  const double2* Bat;      // (P, n_nops, n_basis, n_omega)
  const double* qstream;
  double2* out;            // (n_nops, n_basis, n_omega) or (P, ...) with correlations
  int P, n_nops, n_basis, n_omega;
  int n_ls, n_ksteps, KS;  // l splits, k-steps per pulse, k-steps per stage
};

// cp.async with zero fill: copies 16 bytes if `valid`, writes 16 zero bytes otherwise
__device__ __forceinline__ void cp_async16_zfill(void* smem_dst, const void* gmem_src, bool valid) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  const int n = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(s), "l"(gmem_src), "r"(n));
}

// Both operands are staged in shared memory by cp.async, one stage (KS k-steps) ahead of the DMMAs:
//   A part  [KS][LT][32] doubles   -- Q in fragment order, shared by the CTA's warps
//   X part  [NW][KS][32] double2   -- each warp's own B^{(g)} tile (8 frequencies x 4 KS basis rows)
template <int LT, int NW, bool CORR>
__global__ void __launch_bounds__(NW * 32, (LT >= 16 ? 2 : 3))
from_atomic_dmma_kernel(const AtomicParams p) {
  extern __shared__ __align__(16) double smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int q = lane & 3, r = lane >> 2;
  const int j = blockIdx.y, ls = blockIdx.z;
  const int w_tile = (blockIdx.x * NW + warp) * 8;
  const int w_b = w_tile + r;           // frequency of this lane's B-fragment element
  const bool w_ok = w_b < p.n_omega;
  const int w_ld = w_ok ? w_b : 0;      // clamped (address stays valid, value zero-filled)
  const int w_c = w_tile + 2 * q;       // first of the two frequencies of the C fragment
  const size_t row_stride = (size_t)p.n_omega;
  const size_t pulse_stride = (size_t)p.n_nops * p.n_basis * row_stride;
  const double2* Bj = p.Bat + (size_t)j * p.n_basis * row_stride;
  const int a_doubles = p.KS * LT * 32;
  const int stage_doubles = a_doubles + NW * p.KS * 64;

  double acc_re[LT][2], acc_im[LT][2];
  // ---- g = 0: identity propagator, unit phase
#pragma unroll
  for (int lt = 0; lt < LT; ++lt) {
    const int l = (ls * LT + lt) * 8 + r;
    double2 v0 = make_double2(0.0, 0.0), v1 = v0;
    if (l < p.n_basis) {
      if (w_c < p.n_omega) v0 = Bj[(size_t)l * row_stride + w_c];
      if (w_c + 1 < p.n_omega) v1 = Bj[(size_t)l * row_stride + w_c + 1];
    }
    acc_re[lt][0] = v0.x; acc_re[lt][1] = v1.x;
    acc_im[lt][0] = v0.y; acc_im[lt][1] = v1.y;
  }

  // ---- flattened sequence of stages over (g, k chunk); g counts from 0 = first propagator
  const int spg = (p.n_ksteps + p.KS - 1) / p.KS;  // stages per pulse
  const int n_stages = (p.P - 1) * spg;
  auto stage_load = [&](int i, double* buf) {
    const int g = i / spg, st = i % spg;
    const int s0 = st * p.KS;
    const int ks = min(p.KS, p.n_ksteps - s0);
    const double* src = p.qstream + (((size_t)g * p.n_ls + ls) * p.n_ksteps + s0) * LT * 32;
    const int len = ks * LT * 32;
    for (int e = threadIdx.x * 2; e < len; e += NW * 32 * 2) cp_async16(buf + e, src + e);
    const double2* Bg = Bj + (size_t)(g + 1) * pulse_stride;
    double2* xdst = reinterpret_cast<double2*>(buf + a_doubles) + (size_t)warp * p.KS * 32 + lane;
    for (int s = 0; s < ks; ++s) {
      const int k = 4 * (s0 + s) + q;
      const bool ok = w_ok && k < p.n_basis;
      cp_async16_zfill(xdst + s * 32, Bg + (size_t)(ok ? k : 0) * row_stride + w_ld, ok);
    }
  };
  if (n_stages > 0) {
    stage_load(0, smem);
    cp_async_commit();
  }
  double2 ph = make_double2(0.0, 0.0);
  for (int i = 0; i < n_stages; ++i) {
    const double* cur = smem + (i & 1) * stage_doubles;
    if (i + 1 < n_stages) {
      stage_load(i + 1, smem + ((i + 1) & 1) * stage_doubles);
      cp_async_commit();
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    const int g = i / spg, st = i % spg;
    const int ks = min(p.KS, p.n_ksteps - st * p.KS);
    if (st == 0) {
      ph = w_ok ? p.phases[(size_t)g * row_stride + w_b] : make_double2(0.0, 0.0);
      if (CORR) {  // summand of the previous pulse is complete (g = 0: the first pulse itself)
        double2* dst = p.out + (size_t)g * pulse_stride + (size_t)j * p.n_basis * row_stride;
#pragma unroll
        for (int lt = 0; lt < LT; ++lt) {
          const int l = (ls * LT + lt) * 8 + r;
          if (l < p.n_basis) {
            if (w_c < p.n_omega)
              dst[(size_t)l * row_stride + w_c] = make_double2(acc_re[lt][0], acc_im[lt][0]);
            if (w_c + 1 < p.n_omega)
              dst[(size_t)l * row_stride + w_c + 1] = make_double2(acc_re[lt][1], acc_im[lt][1]);
          }
          acc_re[lt][0] = acc_re[lt][1] = 0.0;
          acc_im[lt][0] = acc_im[lt][1] = 0.0;
        }
      }
    }
    const double2* xs = reinterpret_cast<const double2*>(cur + a_doubles) + (size_t)warp * p.KS * 32 + lane;
    const double* as = cur + lane;
    for (int s = 0; s < ks; ++s) {
      const double2 x = xs[s * 32];
      const double xr = ph.x * x.x - ph.y * x.y;
      const double xi = ph.x * x.y + ph.y * x.x;
#pragma unroll
      for (int lt = 0; lt < LT; ++lt) {
        const double a = as[(s * LT + lt) * 32];
        dmma884(acc_re[lt][0], acc_re[lt][1], a, xr);
        dmma884(acc_im[lt][0], acc_im[lt][1], a, xi);
      }
    }
    __syncthreads();  // everyone is done with `cur` before it is refilled two stages later
  }
  {
    double2* dst = p.out + (size_t)(CORR ? p.P - 1 : 0) * pulse_stride + (size_t)j * p.n_basis * row_stride;
#pragma unroll
    for (int lt = 0; lt < LT; ++lt) {
      const int l = (ls * LT + lt) * 8 + r;
      if (l < p.n_basis) {
        if (w_c < p.n_omega)
          dst[(size_t)l * row_stride + w_c] = make_double2(acc_re[lt][0], acc_im[lt][0]);
        if (w_c + 1 < p.n_omega)
          dst[(size_t)l * row_stride + w_c + 1] = make_double2(acc_re[lt][1], acc_im[lt][1]);
      }
    }
  }
}

template <int LT, int NW>
int launch(ffb_ctx* ctx, AtomicParams p, int n_rows, int correlations) {
  const size_t smem = (size_t)2 * (p.KS * LT * 32 + NW * p.KS * 64) * sizeof(double);
  dim3 grid(ceil_div(p.n_omega, NW * 8), n_rows, p.n_ls);
  if (correlations) {
    auto kern = from_atomic_dmma_kernel<LT, NW, true>;
    FFB_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, NW * 32, smem, ctx->stream>>>(p);
  } else {
    auto kern = from_atomic_dmma_kernel<LT, NW, false>;
    FFB_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, NW * 32, smem, ctx->stream>>>(p);
  }
  FFB_LAUNCHED(ctx);
  return FFB_OK;
}

}  // namespace

int ffbi_from_atomic_dmma(ffb_ctx* ctx, int P, int n_nops, int n_rows, int n_basis, int n_omega,
                          const double* phases, const double* B_atomic, const double* Q,
                          int correlations, double* out) {
  const int l_tiles = ceil_div(n_basis, 8);
  int LT = l_tiles >= 16 ? 16 : l_tiles >= 8 ? 8 : 4;
  if (const char* e = getenv("FFB_FA_LT")) LT = atoi(e);
  AtomicParams p;
  p.phases = reinterpret_cast<const double2*>(phases);
  p.Bat = reinterpret_cast<const double2*>(B_atomic);
  p.out = reinterpret_cast<double2*>(out);
  p.P = P; p.n_nops = n_nops; p.n_basis = n_basis; p.n_omega = n_omega;
  p.n_ls = ceil_div(l_tiles, LT);
  p.n_ksteps = ceil_div(n_basis, 4);
  p.KS = std::min(p.n_ksteps, (32 * 1024) / (LT * 32 * 8));  // <= 32 KB per stage
  DevBuf qs;
  const size_t q_doubles = (size_t)std::max(P - 1, 1) * p.n_ls * p.n_ksteps * LT * 32;
  FFB_TRY(qs.alloc(ctx, q_doubles * sizeof(double)));
  if (P > 1) {
    const size_t total = (size_t)(P - 1) * p.n_ls * p.n_ksteps * LT * 32;
    const unsigned blocks = (unsigned)std::min<size_t>(ceil_div_sz(total, 256), (size_t)ctx->sm_count * 16);
    qstream_kernel<<<blocks, 256, 0, ctx->stream>>>(P - 1, n_basis, p.n_ls, p.n_ksteps, LT, Q,
                                                    qs.as<double>());
    FFB_LAUNCHED(ctx);
  }
  p.qstream = qs.as<double>();
  switch (LT) {
    case 16: return launch<16, 4>(ctx, p, n_rows, correlations);
    case 8: return launch<8, 4>(ctx, p, n_rows, correlations);
    default: return launch<4, 8>(ctx, p, n_rows, correlations);
  }
}
