// Analytic gradient of the first-order infidelity with respect to every control amplitude
// (ff.infidelity_derivative; DESIGN.md section 4.11).
//
// Notation of ffb_control_matrix_from_scratch: H_g = sum_h u_h(g) A_h = V_g diag(E) V_g^+,
// Q_{g-1} = propagators[g], U_g = Q_{g-1}^+ V_g, Bbar_a = V_g^+ N_a V_g, Abar_h = V_g^+ A_h V_g,
// z_mn = (w + E_m - E_n) dt_g and I_mn(w) = int_0^dt e^{i x_mn tau} dtau = dt E2(z_mn) with
// E2(z) = exp[iz, 0] = e^{iz/2} sinc(z/2) (divided differences of exp).  The segment term in the lab frame
//     T_{a,g}(w) = e^{iwt_g} s_a(g) U_g (Bbar_a o I(w)) U_g^+,     B_ak(w) = sum_g tr(T_{a,g} C_k)
// and W_a(w) = sum_k conj(B_ak(w)) C_k give
//     dI_a/du_h(g) = 1/(pi d) sum_w u_w S_a(w) Re[c1 + c2 + c3]
//     c1 = e s sum_ij Abar_h,ij R_ij,    R_ij = sum_n Bbar_jn K1_ijn Wt_ni - sum_m Bbar_mi K2_mij Wt_jm
//     c2 = tr(D_{g,h} [W, Y_{>g}]) = sum_ij (Abar_h o I(0))_ij (-i Xt_ji),   Xt = U^+ [W, Y_{>g}] U
//     c3 = (ds_a(g)/du_h(g)) e tr(U (Bbar o I) U^+ W)
// with Wt = U^+ W U, Y_{>g} = sum_{g'>g} T_{a,g'}, u_w the trapezoid weights and K the divided differences
//     K1_ijn = I[x_jn, x_in],  K2_mij = I[x_mi, x_mj],  I[a, b] = i dt^2 exp[i a dt, i b dt, 0].
// Everything that depends on h is a d^2 dot product against the omega-independent Abar_h and Abar_h o I(0),
// so the h axis costs 16 d^2 flops per control and (segment, frequency).
//
// Kernels (all FP64; templates selected by d alone):
//   grad_prologue_kernel<D>  per segment: U, Bbar of the selected noise operators, Abar and Abar o I(0) of
//                            the selected controls (omega-independent);
//   grad_chunk_kernel<D>     per (frequency, noise operator, chunk c >= 1): sum_{g in chunk} T_{a,g}(w);
//   grad_sweep_kernel<D>     per (frequency tile, noise operator, chunk): W_a(w), then Y starts at the sum
//                            of the later chunks' totals and a reverse sweep over the chunk's segments
//                            forms c1 + c2 + c3; the 128 frequencies of a block are reduced per segment in
//                            shared memory and stored per frequency tile;
//   grad_reduce_kernel       sums the frequency tiles in a fixed order and scales by 1 / (pi d).
// No atomics: two calls give the same bits.  Scratch: the prologue (G (1 + n_sel + 2 n_ctrl) d^2), the
// chunk totals ((S - 1) n_sel n_omega d^2) and the tile partials (n_wt n_sel G n_ctrl); nothing of size
// G n_omega.
#include <algorithm>
#include <cmath>
#include <cstdlib>

#include "ffb_common.cuh"

namespace {

constexpr int GRAD_NT = 128;  // frequencies per sweep block (4 warps)
constexpr int GRAD_MAX_D = 8;

struct GradParams {
  int G, n_sel, n_ctrl, n_nops, n_basis, n_omega;
  int L, S;        // segments per chunk, chunks
  int n_wt, tile;  // frequency tiles of the sweep and their length
  int spectrum_2d;
  const double* E;      // (G, d)
  const double* dt;     // (G)
  const double* t;      // (G + 1)
  const double* omega;  // (n_omega)
  const double* spec;   // (n_omega) or (n_sel, n_omega)
  const double* n_coeffs;  // (n_nops, G)
  const double* deps;      // (n_nops, n_ctrl, G) or null
  const int* sel;          // (n_sel) rows of the noise operators
  const double2* B;        // (n_nops, n_basis, n_omega) control matrix
  const double2* basis;    // (n_basis, d, d)
  const double2* U;        // (G, d, d)
  const double2* Bb;       // (n_sel, G, d, d)
  const double2* Ab;       // (n_ctrl, G, d, d)
  const double2* AI0;      // (n_ctrl, G, d, d)
  double2* tot;            // (S - 1, n_sel, n_omega, d, d)
  double* partial;         // (n_wt, n_sel, G, n_ctrl)
};

__device__ __forceinline__ cplx ld2(const double2* p) {
  const double2 v = *p;
  return {v.x, v.y};
}

// E2(z) = exp[iz, 0] = (e^{iz} - 1) / (iz); *half = e^{iz/2}
__device__ __forceinline__ cplx grad_e2(double z, cplx* half) {
  double s, c;
  const double y = 0.5 * z;
  sincos(y, &s, &c);
  *half = {c, s};
  const double sc = y == 0.0 ? 1.0 : s / y;
  return {c * sc, s * sc};
}

// exp[i z1, i z2, 0], the second divided difference of exp; (h, f) = (e^{iz/2}, E2(z)) of both arguments.
// Far apart: the difference quotient of E2.  Close together but away from 0: the quotient against 0 with
// exp[iz1, iz2] = e^{i(z1+z2)/2} sinc((z1-z2)/2).  All three points within 1: Taylor series about their
// centre c, exp[p,q,r] = e^c sum_n h_n(p-c, q-c, r-c) / (n+2)! (h_n complete homogeneous polynomials).
__device__ __forceinline__ cplx grad_e3(double z1, double z2, cplx h1, cplx h2, cplx f1, cplx f2) {
  const double dz = z1 - z2;
  if (fabs(dz) > 1.0) {
    const double inv = 1.0 / dz;
    return {(f1.im - f2.im) * inv, -(f1.re - f2.re) * inv};
  }
  const double a1 = fabs(z1), a2 = fabs(z2);
  if (fmax(a1, a2) > 1.0) {
    const double y = 0.5 * dz;
    const double sc = y == 0.0 ? 1.0 : sin(y) / y;
    cplx p = cmul(h1, h2);
    p = {p.re * sc, p.im * sc};
    const bool first = a1 >= a2;
    const cplx f = first ? f2 : f1;
    const double inv = 1.0 / (first ? z1 : z2);
    return {(p.im - f.im) * inv, -(p.re - f.re) * inv};
  }
  const double lo = fmin(fmin(z1, z2), 0.0), hi = fmax(fmax(z1, z2), 0.0);
  const double cen = 0.5 * (lo + hi);
  const double u0 = z1 - cen, u1 = z2 - cen, u2 = -cen;
  double p0 = 1.0, H2 = 1.0, H3 = 1.0, inv_fact = 0.5;
  double re = 0.5, im = 0.0;
#pragma unroll
  for (int n = 1; n <= 20; ++n) {
    p0 *= u0;
    H2 = p0 + u1 * H2;
    H3 = H2 + u2 * H3;
    inv_fact /= (double)(n + 2);
    const double term = H3 * inv_fact;
    switch (n & 3) {
      case 0: re += term; break;
      case 1: im += term; break;
      case 2: re -= term; break;
      default: im -= term; break;
    }
  }
  double sn, cs;
  sincos(cen, &sn, &cs);
  return {cs * re - sn * im, cs * im + sn * re};
}

// ---- omega-independent prologue: one thread per (segment, item); item 0: U, 1..n_sel: Bbar, then
// ---- Abar and Abar o I(0) of one control
template <int D>
__global__ void __launch_bounds__(128)
grad_prologue_kernel(int G, int n_sel, int n_ctrl, const double2* __restrict__ V,
                     const double2* __restrict__ Q, const double* __restrict__ E,
                     const double* __restrict__ dt, const double2* __restrict__ n_opers,
                     const int* __restrict__ sel, const double2* __restrict__ c_opers,
                     const int* __restrict__ ctrl, double2* __restrict__ U, double2* __restrict__ Bb,
                     double2* __restrict__ Ab, double2* __restrict__ AI0) {
  const int items = 1 + n_sel + n_ctrl;
  const long long id = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= (long long)G * items) return;
  const int g = (int)(id / items), item = (int)(id % items);
  constexpr int DD = D * D;
  const double2* Vg = V + (size_t)g * DD;
  cplx out[DD];
  if (item == 0) {  // U = Q^+ V
    const double2* Qg = Q + (size_t)g * DD;
    for (int i = 0; i < D; ++i)
      for (int j = 0; j < D; ++j) {
        cplx acc = {0.0, 0.0};
        for (int k = 0; k < D; ++k) acc = cadd(acc, cmul(cconj(ld2(Qg + k * D + i)), ld2(Vg + k * D + j)));
        out[i * D + j] = acc;
      }
    for (int e = 0; e < DD; ++e) U[(size_t)g * DD + e] = make_double2(out[e].re, out[e].im);
    return;
  }
  const double2* A = item <= n_sel ? n_opers + (size_t)sel[item - 1] * DD
                                   : c_opers + (size_t)ctrl[item - 1 - n_sel] * DD;
  cplx AV[DD];
  for (int i = 0; i < D; ++i)
    for (int j = 0; j < D; ++j) {
      cplx acc = {0.0, 0.0};
      for (int k = 0; k < D; ++k) acc = cadd(acc, cmul(ld2(A + i * D + k), ld2(Vg + k * D + j)));
      AV[i * D + j] = acc;
    }
  for (int i = 0; i < D; ++i)
    for (int j = 0; j < D; ++j) {
      cplx acc = {0.0, 0.0};
      for (int k = 0; k < D; ++k) acc = cadd(acc, cmul(cconj(ld2(Vg + k * D + i)), AV[k * D + j]));
      out[i * D + j] = acc;
    }
  if (item <= n_sel) {
    double2* dst = Bb + ((size_t)(item - 1) * G + g) * DD;
    for (int e = 0; e < DD; ++e) dst[e] = make_double2(out[e].re, out[e].im);
    return;
  }
  const int h = item - 1 - n_sel;
  double2* dA = Ab + ((size_t)h * G + g) * DD;
  double2* dI = AI0 + ((size_t)h * G + g) * DD;
  const double dtg = dt[g];
  for (int m = 0; m < D; ++m)
    for (int n = 0; n < D; ++n) {
      cplx half;
      const cplx f = grad_e2((E[(size_t)g * D + m] - E[(size_t)g * D + n]) * dtg, &half);
      const cplx a = out[m * D + n];
      const cplx ai = cmul(a, {dtg * f.re, dtg * f.im});
      dA[m * D + n] = make_double2(a.re, a.im);
      dI[m * D + n] = make_double2(ai.re, ai.im);
    }
}

// Bbar o I(w) for segment g (per thread); also the z, e^{iz/2} and E2(z) the divided differences need
template <int D>
__device__ __forceinline__ void grad_segment_integral(const GradParams& p, int a, int g, double w,
                                                      cplx* BI, double* z, cplx* hf, cplx* f) {
  const double dtg = p.dt[g];
  const double* Eg = p.E + (size_t)g * D;
  const double2* Bb = p.Bb + ((size_t)a * p.G + g) * D * D;
  for (int m = 0; m < D; ++m) {
    const double wm = w + Eg[m];
    for (int n = 0; n < D; ++n) {
      const double zz = (wm - Eg[n]) * dtg;
      cplx half;
      const cplx ff = grad_e2(zz, &half);
      z[m * D + n] = zz;
      hf[m * D + n] = half;
      f[m * D + n] = ff;
      BI[m * D + n] = cmul(ld2(Bb + m * D + n), {dtg * ff.re, dtg * ff.im});
    }
  }
}

// out = U X U^+ (lab frame) or U^+ X U
template <int D, bool DAGGER_LEFT>
__device__ __forceinline__ void grad_transform(const double2* Ug, const cplx* X, cplx* out) {
  cplx tmp[D * D];
  for (int i = 0; i < D; ++i)
    for (int j = 0; j < D; ++j) {  // tmp = X U^+ or X U
      cplx acc = {0.0, 0.0};
      for (int k = 0; k < D; ++k) {
        const cplx u = DAGGER_LEFT ? ld2(Ug + k * D + j) : cconj(ld2(Ug + j * D + k));
        acc = cadd(acc, cmul(X[i * D + k], u));
      }
      tmp[i * D + j] = acc;
    }
  for (int i = 0; i < D; ++i)
    for (int j = 0; j < D; ++j) {
      cplx acc = {0.0, 0.0};
      for (int k = 0; k < D; ++k) {
        const cplx u = DAGGER_LEFT ? cconj(ld2(Ug + k * D + i)) : ld2(Ug + i * D + k);
        acc = cadd(acc, cmul(u, tmp[k * D + j]));
      }
      out[i * D + j] = acc;
    }
}

// ---- chunk totals: tot[c - 1][a][w] = sum_{g in chunk c} T_{a,g}(w), c = 1 .. S-1 (chunk 0's is never
// ---- needed: Y of chunk c starts at the sum of the chunks after it)
template <int D>
__global__ void __launch_bounds__(128) grad_chunk_kernel(GradParams p) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  const int a = blockIdx.y, c = blockIdx.z + 1;
  if (w >= p.n_omega) return;
  constexpr int DD = D * D;
  const double wo = p.omega[w];
  const int row = p.sel[a];
  cplx acc[DD];
  for (int e = 0; e < DD; ++e) acc[e] = {0.0, 0.0};
  const int g0 = c * p.L, g1 = min(p.G, g0 + p.L);
  for (int g = g0; g < g1; ++g) {
    cplx BI[DD], hf[DD], f[DD], T[DD];
    double z[DD];
    grad_segment_integral<D>(p, a, g, wo, BI, z, hf, f);
    grad_transform<D, false>(p.U + (size_t)g * DD, BI, T);
    double sn, cs;
    sincos(wo * p.t[g], &sn, &cs);
    const double s = p.n_coeffs[(size_t)row * p.G + g];
    const cplx es = {s * cs, s * sn};
    for (int e = 0; e < DD; ++e) acc[e] = cadd(acc[e], cmul(es, T[e]));
  }
  double2* dst = p.tot + (((size_t)(c - 1) * p.n_sel + a) * p.n_omega + w) * DD;
  for (int e = 0; e < DD; ++e) dst[e] = make_double2(acc[e].re, acc[e].im);
}

__device__ __forceinline__ double grad_warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---- reverse sweep: block (tile, a, chunk), GRAD_NT threads along the frequencies of the tile
template <int D>
__global__ void __launch_bounds__(GRAD_NT) grad_sweep_kernel(GradParams p) {
  extern __shared__ double red[];  // [2][GRAD_NT / 32][n_ctrl]
  constexpr int DD = D * D;
  constexpr int NW = GRAD_NT / 32;
  const int wt = blockIdx.x, a = blockIdx.y, c = blockIdx.z;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int row = p.sel[a];
  const int g0 = c * p.L, g1 = min(p.G, g0 + p.L);
  const int w_lo = wt * p.tile, w_hi = min(p.n_omega, w_lo + p.tile);
  const int n_batch = (w_hi - w_lo + GRAD_NT - 1) / GRAD_NT;
  int buf = 0;
  for (int j = 0; j < n_batch; ++j) {
    const int w = w_lo + j * GRAD_NT + tid;
    const bool active = w < w_hi;
    const double wo = active ? p.omega[w] : 0.0;
    double us = 0.0;  // trapezoid weight times spectrum
    cplx W[DD], Y[DD];
    for (int e = 0; e < DD; ++e) W[e] = Y[e] = {0.0, 0.0};
    if (active) {
      if (p.n_omega > 1) {
        const double left = w > 0 ? wo - p.omega[w - 1] : 0.0;
        const double right = w + 1 < p.n_omega ? p.omega[w + 1] - wo : 0.0;
        us = 0.5 * (left + right);
      }
      us *= p.spec[(p.spectrum_2d ? (size_t)a * p.n_omega : 0) + w];
      for (int k = 0; k < p.n_basis; ++k) {
        const cplx b = cconj(ld2(p.B + ((size_t)row * p.n_basis + k) * p.n_omega + w));
        const double2* Ck = p.basis + (size_t)k * DD;
        for (int e = 0; e < DD; ++e) W[e] = cadd(W[e], cmul(b, ld2(Ck + e)));
      }
      for (int cc = c + 1; cc < p.S; ++cc) {
        const double2* src = p.tot + (((size_t)(cc - 1) * p.n_sel + a) * p.n_omega + w) * DD;
        for (int e = 0; e < DD; ++e) Y[e] = cadd(Y[e], ld2(src + e));
      }
    }
    for (int g = g1 - 1; g >= g0; --g) {
      const double2* Ug = p.U + (size_t)g * DD;
      cplx C1[DD], X2[DD];  // coefficients of Abar_h and of Abar_h o I(0)
      cplx tau = {0.0, 0.0};
      if (active) {
        cplx BI[DD], hf[DD], f[DD], T[DD], Wt[DD];
        double z[DD];
        grad_segment_integral<D>(p, a, g, wo, BI, z, hf, f);
        grad_transform<D, true>(Ug, W, Wt);
        // X2_ij = -i Xt_ji,  Xt = U^+ (W Y - Y W) U
        cplx Cm[DD];
        for (int i = 0; i < D; ++i)
          for (int k = 0; k < D; ++k) {
            cplx acc = {0.0, 0.0};
            for (int l = 0; l < D; ++l) {
              acc = cadd(acc, cmul(W[i * D + l], Y[l * D + k]));
              const cplx yw = cmul(Y[i * D + l], W[l * D + k]);
              acc = {acc.re - yw.re, acc.im - yw.im};
            }
            Cm[i * D + k] = acc;
          }
        grad_transform<D, true>(Ug, Cm, T);
        for (int i = 0; i < D; ++i)
          for (int k = 0; k < D; ++k) X2[i * D + k] = {T[k * D + i].im, -T[k * D + i].re};
        // tau = tr((Bbar o I) Wt)
        for (int m = 0; m < D; ++m)
          for (int n = 0; n < D; ++n) tau = cadd(tau, cmul(BI[m * D + n], Wt[n * D + m]));
        // R_ij = i dt^2 [sum_n Bbar_jn E3(z_jn, z_in) Wt_ni - sum_m Bbar_mi E3(z_mi, z_mj) Wt_jm]
        const double2* Bb = p.Bb + ((size_t)a * p.G + g) * DD;
        const double dtg = p.dt[g];
        double sn, cs;
        sincos(wo * p.t[g], &sn, &cs);
        const double s = p.n_coeffs[(size_t)row * p.G + g];
        const double f2 = dtg * dtg;
        const cplx pre = {-f2 * s * sn, f2 * s * cs};  // i dt^2 s e^{iwt}
        for (int i = 0; i < D; ++i)
          for (int jj = 0; jj < D; ++jj) {
            cplx acc = {0.0, 0.0};
            for (int n = 0; n < D; ++n) {
              const cplx k1 = grad_e3(z[jj * D + n], z[i * D + n], hf[jj * D + n], hf[i * D + n],
                                      f[jj * D + n], f[i * D + n]);
              acc = cadd(acc, cmul(cmul(ld2(Bb + jj * D + n), k1), Wt[n * D + i]));
            }
            for (int m = 0; m < D; ++m) {
              const cplx k2 = grad_e3(z[m * D + i], z[m * D + jj], hf[m * D + i], hf[m * D + jj],
                                      f[m * D + i], f[m * D + jj]);
              const cplx v = cmul(cmul(ld2(Bb + m * D + i), k2), Wt[jj * D + m]);
              acc = {acc.re - v.re, acc.im - v.im};
            }
            C1[i * D + jj] = cmul(pre, acc);
          }
        tau = cmul({cs, sn}, tau);  // e tr(...): c3 per unit ds/du
        // Y += s e T
        grad_transform<D, false>(Ug, BI, T);
        const cplx es = {s * cs, s * sn};
        for (int e = 0; e < DD; ++e) Y[e] = cadd(Y[e], cmul(es, T[e]));
      } else {
        for (int e = 0; e < DD; ++e) C1[e] = X2[e] = {0.0, 0.0};
      }
      double* rb = red + (size_t)buf * NW * p.n_ctrl;
      for (int h = 0; h < p.n_ctrl; ++h) {
        double v = 0.0;
        if (active) {
          const double2* Ah = p.Ab + ((size_t)h * p.G + g) * DD;
          const double2* Ih = p.AI0 + ((size_t)h * p.G + g) * DD;
          for (int e = 0; e < DD; ++e) {
            const cplx x = ld2(Ah + e), y = ld2(Ih + e);
            v += x.re * C1[e].re - x.im * C1[e].im + y.re * X2[e].re - y.im * X2[e].im;
          }
          if (p.deps) v += p.deps[((size_t)row * p.n_ctrl + h) * p.G + g] * tau.re;
          v *= us;
        }
        v = grad_warp_sum(v);
        if (lane == 0) rb[warp * p.n_ctrl + h] = v;
      }
      __syncthreads();
      for (int h = tid; h < p.n_ctrl; h += GRAD_NT) {
        double v = rb[h];
        for (int k = 1; k < NW; ++k) v += rb[k * p.n_ctrl + h];
        double* dst = p.partial + (((size_t)wt * p.n_sel + a) * p.G + g) * p.n_ctrl + h;
        *dst = j == 0 ? v : *dst + v;
      }
      buf ^= 1;
    }
  }
}

__global__ void __launch_bounds__(256)
grad_reduce_kernel(int n_wt, size_t n_out, double scale, const double* __restrict__ partial,
                   double* __restrict__ out) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_out) return;
  double v = 0.0;
  for (int k = 0; k < n_wt; ++k) v += partial[(size_t)k * n_out + i];
  out[i] = scale * v;
}

template <int D>
int grad_launch(ffb_ctx* ctx, GradParams p, const double* eigvecs, const double* propagators,
                const double* n_opers, const double* c_opers, const int* ctrl) {
  const int items = 1 + p.n_sel + p.n_ctrl;
  const long long n_pro = (long long)p.G * items;
  grad_prologue_kernel<D><<<(unsigned)((n_pro + 127) / 128), 128, 0, ctx->stream>>>(
      p.G, p.n_sel, p.n_ctrl, reinterpret_cast<const double2*>(eigvecs),
      reinterpret_cast<const double2*>(propagators), p.E, p.dt, reinterpret_cast<const double2*>(n_opers),
      p.sel, reinterpret_cast<const double2*>(c_opers), ctrl, const_cast<double2*>(p.U),
      const_cast<double2*>(p.Bb), const_cast<double2*>(p.Ab), const_cast<double2*>(p.AI0));
  FFB_LAUNCHED(ctx);
  if (p.S > 1) {
    grad_chunk_kernel<D><<<dim3(ceil_div(p.n_omega, 128), p.n_sel, p.S - 1), 128, 0, ctx->stream>>>(p);
    FFB_LAUNCHED(ctx);
  }
  const size_t smem = (size_t)2 * (GRAD_NT / 32) * p.n_ctrl * sizeof(double);
  FFB_TRY(ffb_func_smem(ctx, grad_sweep_kernel<D>, smem));
  grad_sweep_kernel<D><<<dim3(p.n_wt, p.n_sel, p.S), GRAD_NT, smem, ctx->stream>>>(p);
  FFB_LAUNCHED(ctx);
  return FFB_OK;
}

}  // namespace

// Device-pointer stage of ffb_infidelity_derivative (ffb_api.cu): every pointer is a device pointer;
// control_matrix holds all n_nops rows; out (n_sel, G, n_ctrl).
int ffbi_infidelity_derivative(ffb_ctx* ctx, int G, int d, int n_nops, int n_basis, int n_omega,
                               const double* eigvals, const double* eigvecs,
                               const double* propagators, const double* omega, const double* basis,
                               const double* n_opers, const double* n_coeffs, const double* dt,
                               const double* t, const double* c_opers, const double* control_matrix,
                               int n_ctrl, const int* ctrl_idx, int n_sel, const int* sel_idx,
                               const double* spectrum, int spectrum_ndim,
                               const double* n_coeffs_deps, int norm_d, double* out) {
  FFB_REQUIRE(ctx, d >= 1 && d <= GRAD_MAX_D,
              "infidelity derivative: Hilbert-space dimension d = %d exceeds the supported maximum of %d "
              "(README: limits)", d, GRAD_MAX_D);
  FFB_REQUIRE(ctx, G >= 1 && n_nops >= 1 && n_basis >= 1 && n_omega >= 1 && n_ctrl >= 1 && n_sel >= 1 &&
                       (spectrum_ndim == 1 || spectrum_ndim == 2) && norm_d >= 1,
              "infidelity derivative: bad shape");
  const size_t dd = (size_t)d * d;
  GradParams p{};
  p.G = G;
  p.n_sel = n_sel;
  p.n_ctrl = n_ctrl;
  p.n_nops = n_nops;
  p.n_basis = n_basis;
  p.n_omega = n_omega;
  p.spectrum_2d = spectrum_ndim == 2;
  // split of the segment axis: enough (frequency, operator, chunk) sweeps to fill the device
  const long long sweeps = (long long)n_omega * n_sel;
  const long long want = (long long)ctx->sm_count * 1024;
  int S = (int)std::min<long long>(std::max<long long>(1, (want + sweeps - 1) / sweeps), 32);
  S = std::min(S, G);
  p.L = (G + S - 1) / S;
  if (const char* e = getenv("FFB_GRAD_SEGS_PER_CHUNK")) p.L = std::max(1, std::min(G, atoi(e)));
  p.S = (G + p.L - 1) / p.L;
  // frequency tiles: enough blocks for 4 per SM, partials capped at 64 MiB
  const size_t per_tile = (size_t)n_sel * G * n_ctrl * 8;
  int n_wt = ceil_div(n_omega, GRAD_NT);
  n_wt = std::min(n_wt, std::max(1, ceil_div(4 * ctx->sm_count, n_sel * p.S)));
  n_wt = (int)std::min<size_t>(n_wt, std::max<size_t>(1, ((size_t)64 << 20) / per_tile));
  p.tile = ceil_div(ceil_div(n_omega, n_wt), GRAD_NT) * GRAD_NT;
  p.n_wt = ceil_div(n_omega, p.tile);
  DevBuf U, Bb, Ab, AI0, tot, part;
  FFB_TRY(U.alloc(ctx, (size_t)G * dd * 16));
  FFB_TRY(Bb.alloc(ctx, (size_t)n_sel * G * dd * 16));
  FFB_TRY(Ab.alloc(ctx, (size_t)n_ctrl * G * dd * 16));
  FFB_TRY(AI0.alloc(ctx, (size_t)n_ctrl * G * dd * 16));
  FFB_TRY(tot.alloc(ctx, (size_t)(p.S - 1) * n_sel * n_omega * dd * 16));
  FFB_TRY(part.alloc(ctx, (size_t)p.n_wt * per_tile));
  p.E = eigvals;
  p.dt = dt;
  p.t = t;
  p.omega = omega;
  p.spec = spectrum;
  p.n_coeffs = n_coeffs;
  p.deps = n_coeffs_deps;
  p.sel = sel_idx;
  p.B = reinterpret_cast<const double2*>(control_matrix);
  p.basis = reinterpret_cast<const double2*>(basis);
  p.U = U.as<double2>();
  p.Bb = Bb.as<double2>();
  p.Ab = Ab.as<double2>();
  p.AI0 = AI0.as<double2>();
  p.tot = tot.as<double2>();
  p.partial = part.as<double>();
  int rc = FFB_EINVAL;
  switch (d) {
    case 1: rc = grad_launch<1>(ctx, p, eigvecs, propagators, n_opers, c_opers, ctrl_idx); break;
    case 2: rc = grad_launch<2>(ctx, p, eigvecs, propagators, n_opers, c_opers, ctrl_idx); break;
    case 3: rc = grad_launch<3>(ctx, p, eigvecs, propagators, n_opers, c_opers, ctrl_idx); break;
    case 4: rc = grad_launch<4>(ctx, p, eigvecs, propagators, n_opers, c_opers, ctrl_idx); break;
    case 5: rc = grad_launch<5>(ctx, p, eigvecs, propagators, n_opers, c_opers, ctrl_idx); break;
    case 6: rc = grad_launch<6>(ctx, p, eigvecs, propagators, n_opers, c_opers, ctrl_idx); break;
    case 7: rc = grad_launch<7>(ctx, p, eigvecs, propagators, n_opers, c_opers, ctrl_idx); break;
    default: rc = grad_launch<8>(ctx, p, eigvecs, propagators, n_opers, c_opers, ctrl_idx); break;
  }
  FFB_TRY(rc);
  const size_t n_out = (size_t)n_sel * G * n_ctrl;
  grad_reduce_kernel<<<(unsigned)ceil_div_sz(n_out, 256), 256, 0, ctx->stream>>>(
      p.n_wt, n_out, 1.0 / (M_PI * norm_d), p.partial, out);
  FFB_LAUNCHED(ctx);
  return FFB_OK;
}
