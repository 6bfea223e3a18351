// K1 -- batched Hermitian eigendecomposition, piecewise propagators and their running product.
//
// Replaces PulseSequence.diagonalize (pulse_sequence.py:577-586) and numeric.diagonalize
// (numeric.py:1886-1935) of the reference:
//     H_g = sum_i a_i(t_g) A_i                                    (einsum 'ijk,il->ljk')
//     H_g = V_g D_g V_g^dagger, eigenvalues ascending             (numpy.linalg.eigh)
//     P_g = V_g exp(-i D_g dt_g) V_g^dagger
//     Q   = [1, P_0, P_1 P_0, ...]                                (util.adot, util.py:868-877)
//
// B200 mapping: one warp per segment runs a cyclic complex Jacobi iteration with the d x d matrix
// and the accumulating eigenvector matrix in shared memory (lanes own rows / columns); the
// running product, which the reference forms with G sequential matmuls, is a three-phase parallel
// scan over the (associative, non-commutative) matrix product.
#include "ffb_common.cuh"

namespace {

constexpr int DIAG_WARPS = 4;
constexpr int MAX_D = 32;  // one lane per row/column
constexpr int MAX_SWEEPS = 40;

__device__ __forceinline__ cplx lds_c(const double* m, int i) { return {m[2 * i], m[2 * i + 1]}; }
__device__ __forceinline__ void sts_c(double* m, int i, cplx v) {
  m[2 * i] = v.re;
  m[2 * i + 1] = v.im;
}

// One warp per segment. Shared memory per warp: H (d*d c128), V (d*d c128), ev (d), perm (d ints).
__global__ void __launch_bounds__(DIAG_WARPS * 32)
diag_kernel(int G, int d, int n_cops, const double* __restrict__ c_opers,
            const double* __restrict__ c_coeffs, const double* __restrict__ dt,
            double* __restrict__ eigvals, double* __restrict__ eigvecs,
            double* __restrict__ piecewise, int* __restrict__ not_converged) {
  extern __shared__ double smem[];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int g = blockIdx.x * DIAG_WARPS + warp;
  if (g >= G) return;
  const int dd = d * d;
  const int per_warp = 4 * dd + 2 * d;  // doubles
  double* H = smem + (size_t)warp * per_warp;
  double* V = H + 2 * dd;
  double* ev = V + 2 * dd;
  int* perm = reinterpret_cast<int*>(ev + d);

  // ---- build H_g (lower triangle is authoritative, as LAPACK's UPLO='L' in numpy.linalg.eigh)
  for (int e = lane; e < dd; e += 32) {
    cplx h = {0.0, 0.0};
    if (c_coeffs != nullptr) {
      for (int i = 0; i < n_cops; ++i) {
        const double a = c_coeffs[(size_t)i * G + g];
        // rounded product, rounded sum, operators in order: the bits of np.einsum('ijk,il->ljk') in
        // PulseSequence.diagonalize (pulse_sequence.py:582), so that H -- and everything derived from it --
        // is the same whether the pulse or the caller formed the Hamiltonian
        h.re = __dadd_rn(h.re, __dmul_rn(a, c_opers[2 * ((size_t)i * dd + e)]));
        h.im = __dadd_rn(h.im, __dmul_rn(a, c_opers[2 * ((size_t)i * dd + e) + 1]));
      }
    } else {
      h.re = c_opers[2 * ((size_t)g * dd + e)];
      h.im = c_opers[2 * ((size_t)g * dd + e) + 1];
    }
    sts_c(H, e, h);
    const int r = e / d, c = e % d;
    sts_c(V, e, cplx{r == c ? 1.0 : 0.0, 0.0});
  }
  __syncwarp();
  for (int e = lane; e < dd; e += 32) {
    const int r = e / d, c = e % d;
    if (r < c) sts_c(H, e, cconj(lds_c(H, c * d + r)));
    if (r == c) H[2 * e + 1] = 0.0;
  }
  __syncwarp();

  // H <- 2^-e H with e the exponent of its largest entry. The iteration is equivariant under powers of two
  // except for the squares in its convergence test, which underflow for max|H| below ~1e-160 (0 sweeps,
  // the diagonal returned as the eigenvalues) and overflow above ~1e154 (reported as not converged).
  // Scaling by a power of two is exact, so no bit changes for H in between; NaN / Inf stay unscaled.
  double hmax = 0.0;
  for (int e = lane; e < dd; e += 32) hmax = fmax(hmax, fmax(fabs(H[2 * e]), fabs(H[2 * e + 1])));
  for (int o = 16; o > 0; o >>= 1) hmax = fmax(hmax, __shfl_xor_sync(0xffffffffu, hmax, o));
  int scale_exp = 0;
  if (hmax > 0.0 && isfinite(hmax)) {
    frexp(hmax, &scale_exp);
    for (int e = lane; e < 2 * dd; e += 32) H[e] = ldexp(H[e], -scale_exp);
  }
  __syncwarp();

  double norm2 = 0.0;
  for (int e = lane; e < dd; e += 32) {
    const cplx h = lds_c(H, e);
    norm2 += h.re * h.re + h.im * h.im;
  }
  for (int o = 16; o > 0; o >>= 1) norm2 += __shfl_xor_sync(0xffffffffu, norm2, o);

  // ---- cyclic Jacobi sweeps
  bool converged = (d == 1);
  for (int sweep = 0; sweep < MAX_SWEEPS && !converged; ++sweep) {
    double off = 0.0;
    for (int e = lane; e < dd; e += 32) {
      const int r = e / d, c = e % d;
      if (r < c) {
        const cplx h = lds_c(H, e);
        off += h.re * h.re + h.im * h.im;
      }
    }
    for (int o = 16; o > 0; o >>= 1) off += __shfl_xor_sync(0xffffffffu, off, o);
    if (off <= 1e-34 * norm2 || off == 0.0) {
      converged = true;
      break;
    }
    for (int p = 0; p < d - 1; ++p) {
      for (int q = p + 1; q < d; ++q) {
        const cplx h = lds_c(H, p * d + q);
        const double beta = hypot(h.re, h.im);
        if (beta == 0.0) continue;  // warp-uniform (all lanes read the same element)
        const cplx w = {h.re / beta, h.im / beta};
        const double a = H[2 * (p * d + p)], b = H[2 * (q * d + q)];
        const double tau = (b - a) / (2.0 * beta);
        const double t = (tau >= 0.0 ? 1.0 : -1.0) / (fabs(tau) + sqrt(1.0 + tau * tau));
        const double c = 1.0 / sqrt(1.0 + t * t);
        const double s = t * c;
        const cplx swc = {s * w.re, -s * w.im};  // s * conj(w)
        const cplx cwc = {c * w.re, -c * w.im};  // c * conj(w)
        __syncwarp();
        // columns p, q of H and V:  X[:,p] <- c X[:,p] - s conj(w) X[:,q];  X[:,q] <- s X[:,p] + c conj(w) X[:,q]
        if (lane < d) {
          const int k = lane;
          cplx xp = lds_c(H, k * d + p), xq = lds_c(H, k * d + q);
          cplx a1 = cmul(swc, xq), a2 = cmul(cwc, xq);
          sts_c(H, k * d + p, cplx{c * xp.re - a1.re, c * xp.im - a1.im});
          sts_c(H, k * d + q, cplx{s * xp.re + a2.re, s * xp.im + a2.im});
          xp = lds_c(V, k * d + p);
          xq = lds_c(V, k * d + q);
          a1 = cmul(swc, xq);
          a2 = cmul(cwc, xq);
          sts_c(V, k * d + p, cplx{c * xp.re - a1.re, c * xp.im - a1.im});
          sts_c(V, k * d + q, cplx{s * xp.re + a2.re, s * xp.im + a2.im});
        }
        __syncwarp();
        // rows p, q of H:  H[p,:] <- c H[p,:] - s w H[q,:];  H[q,:] <- s H[p,:] + c w H[q,:]
        if (lane < d) {
          const int k = lane;
          const cplx yp = lds_c(H, p * d + k), yq = lds_c(H, q * d + k);
          const cplx sw = {s * w.re, s * w.im}, cw = {c * w.re, c * w.im};
          const cplx a1 = cmul(sw, yq), a2 = cmul(cw, yq);
          sts_c(H, p * d + k, cplx{c * yp.re - a1.re, c * yp.im - a1.im});
          sts_c(H, q * d + k, cplx{s * yp.re + a2.re, s * yp.im + a2.im});
        }
        __syncwarp();
        if (lane == 0) {
          sts_c(H, p * d + q, cplx{0.0, 0.0});
          sts_c(H, q * d + p, cplx{0.0, 0.0});
          // classical diagonal update (one rounding each), see diag_small_one
          sts_c(H, p * d + p, cplx{fma(-t, beta, a), 0.0});
          sts_c(H, q * d + q, cplx{fma(t, beta, b), 0.0});
        }
        __syncwarp();
      }
    }
  }
  // unit columns (see diag_small_one)
  if (lane < d) {
    double n2 = 0.0;
    for (int r = 0; r < d; ++r) {
      const cplx v = lds_c(V, r * d + lane);
      n2 += v.re * v.re + v.im * v.im;
    }
    const double f = fma(-0.5, n2, 1.5);
    for (int r = 0; r < d; ++r) {
      const cplx v = lds_c(V, r * d + lane);
      sts_c(V, r * d + lane, cplx{v.re * f, v.im * f});
    }
  }
  __syncwarp();
  // (a NaN / Inf entry can "converge" because a rotation sets its pivot to exactly zero)
  if ((!converged || !isfinite(norm2)) && lane == 0) atomicAdd(not_converged, 1);

  // ---- ascending order (stable), as numpy.linalg.eigh returns them
  if (lane < d) {
    ev[lane] = ldexp(H[2 * (lane * d + lane)], scale_exp);
    perm[lane] = lane;  // stays a valid permutation entry even if NaN eigenvalues make ranks collide
  }
  __syncwarp();
  if (lane < d) {
    const double mine = ev[lane];
    int rank = 0;
    for (int j = 0; j < d; ++j) {
      const double other = ev[j];
      // total order (NaN last, ties by index): the ranks are a permutation for ANY input, so no two
      // lanes ever write the same entry (compute-sanitizer racecheck, NaN Hamiltonians)
      const bool mine_nan = mine != mine, other_nan = other != other;
      rank += mine_nan ? (!other_nan || j < lane)
                       : (!other_nan && ((other < mine) || (other == mine && j < lane)));
    }
    perm[rank] = lane;
  }
  __syncwarp();
  if (lane < d) eigvals[(size_t)g * d + lane] = ev[perm[lane]];
  for (int e = lane; e < dd; e += 32) {
    const int r = e / d, c = e % d;
    const cplx v = lds_c(V, r * d + perm[c]);
    eigvecs[2 * ((size_t)g * dd + e)] = v.re;
    eigvecs[2 * ((size_t)g * dd + e) + 1] = v.im;
  }

  // ---- P_g = V exp(-i D dt) V^dagger  (order of eigenpairs is irrelevant here)
  const double dtg = dt[g];
  for (int e = lane; e < dd; e += 32) {
    const int r = e / d, c = e % d;
    cplx acc = {0.0, 0.0};
    for (int j = 0; j < d; ++j) {
      double sn, cs;
      sincos(-dtg * ev[j], &sn, &cs);
      const cplx vv = cmulc(lds_c(V, r * d + j), lds_c(V, c * d + j));
      acc.re += vv.re * cs - vv.im * sn;
      acc.im += vv.re * sn + vv.im * cs;
    }
    piecewise[2 * ((size_t)g * dd + e)] = acc.re;
    piecewise[2 * ((size_t)g * dd + e) + 1] = acc.im;
  }
}

// ---- small matrices (d <= 4): one THREAD per segment, H and V in registers -------------------------
// The warp-per-segment kernel above spends its time in warp synchronisation and in scalar work that
// all 32 lanes repeat (hypot, three divisions and two square roots per rotation): 17.5 us for the 1e4
// 2 x 2 matrices of config 2.  For d <= 4 the whole cyclic Jacobi iteration fits the registers of one
// thread (fully unrolled, same rotation formulas, same convergence test, same stable ascending
// order), so a segment costs one thread instead of one warp.
// eigendecomposition of segment g (written to eigvals / eigvecs) and its propagator P (registers)
template <int D>
__device__ __forceinline__ void diag_small_one(int G, int g, int n_cops,
                                               const double* __restrict__ c_opers,
                                               const double* __restrict__ c_coeffs,
                                               const double* __restrict__ dt,
                                               double* __restrict__ eigvals,
                                               double* __restrict__ eigvecs,
                                               int* __restrict__ not_converged, double2 (&P)[D * D]) {
  constexpr int DD = D * D;
  cplx H[D][D], V[D][D];
  // ---- H_g (lower triangle is authoritative, as LAPACK's UPLO='L' in numpy.linalg.eigh)
#pragma unroll
  for (int r = 0; r < D; ++r) {
#pragma unroll
    for (int c = 0; c < D; ++c) {
      cplx h = {0.0, 0.0};
      if (c_coeffs != nullptr) {
        for (int i = 0; i < n_cops; ++i) {
          const double a = c_coeffs[(size_t)i * G + g];
          // same bits as np.einsum('ijk,il->ljk') (see diag_kernel)
          h.re = __dadd_rn(h.re, __dmul_rn(a, c_opers[2 * ((size_t)i * DD + r * D + c)]));
          h.im = __dadd_rn(h.im, __dmul_rn(a, c_opers[2 * ((size_t)i * DD + r * D + c) + 1]));
        }
      } else {
        h.re = c_opers[2 * ((size_t)g * DD + r * D + c)];
        h.im = c_opers[2 * ((size_t)g * DD + r * D + c) + 1];
      }
      H[r][c] = h;
      V[r][c] = cplx{r == c ? 1.0 : 0.0, 0.0};
    }
  }
#pragma unroll
  for (int r = 0; r < D; ++r) {
    H[r][r].im = 0.0;
#pragma unroll
    for (int c = r + 1; c < D; ++c) H[r][c] = cconj(H[c][r]);
  }
  // H <- 2^-e H, e the exponent of its largest entry (exact; see diag_kernel)
  double hmax = 0.0;
#pragma unroll
  for (int r = 0; r < D; ++r)
#pragma unroll
    for (int c = 0; c < D; ++c) hmax = fmax(hmax, fmax(fabs(H[r][c].re), fabs(H[r][c].im)));
  int scale_exp = 0;
  if (hmax > 0.0 && isfinite(hmax)) {
    frexp(hmax, &scale_exp);
#pragma unroll
    for (int r = 0; r < D; ++r)
#pragma unroll
      for (int c = 0; c < D; ++c)
        H[r][c] = cplx{ldexp(H[r][c].re, -scale_exp), ldexp(H[r][c].im, -scale_exp)};
  }
  double norm2 = 0.0;
#pragma unroll
  for (int r = 0; r < D; ++r)
#pragma unroll
    for (int c = 0; c < D; ++c) norm2 += H[r][c].re * H[r][c].re + H[r][c].im * H[r][c].im;

  // ---- cyclic Jacobi sweeps
  bool converged = (D == 1);
  for (int sweep = 0; sweep < MAX_SWEEPS && !converged; ++sweep) {
    double off = 0.0;
#pragma unroll
    for (int r = 0; r < D; ++r)
#pragma unroll
      for (int c = r + 1; c < D; ++c) off += H[r][c].re * H[r][c].re + H[r][c].im * H[r][c].im;
    if (off <= 1e-34 * norm2 || off == 0.0) {
      converged = true;
      break;
    }
#pragma unroll
    for (int p = 0; p < D - 1; ++p) {
#pragma unroll
      for (int q = p + 1; q < D; ++q) {
        const cplx h = H[p][q];
        const double beta = hypot(h.re, h.im);
        if (beta != 0.0) {
          const cplx w = {h.re / beta, h.im / beta};
          const double a = H[p][p].re, b = H[q][q].re;
          const double tau = (b - a) / (2.0 * beta);
          const double t = (tau >= 0.0 ? 1.0 : -1.0) / (fabs(tau) + sqrt(1.0 + tau * tau));
          const double c = 1.0 / sqrt(1.0 + t * t);
          const double s = t * c;
          const cplx swc = {s * w.re, -s * w.im};  // s * conj(w)
          const cplx cwc = {c * w.re, -c * w.im};  // c * conj(w)
          // columns p, q of H and V
#pragma unroll
          for (int k = 0; k < D; ++k) {
            cplx xp = H[k][p], xq = H[k][q];
            cplx a1 = cmul(swc, xq), a2 = cmul(cwc, xq);
            H[k][p] = cplx{c * xp.re - a1.re, c * xp.im - a1.im};
            H[k][q] = cplx{s * xp.re + a2.re, s * xp.im + a2.im};
            xp = V[k][p];
            xq = V[k][q];
            a1 = cmul(swc, xq);
            a2 = cmul(cwc, xq);
            V[k][p] = cplx{c * xp.re - a1.re, c * xp.im - a1.im};
            V[k][q] = cplx{s * xp.re + a2.re, s * xp.im + a2.im};
          }
          // rows p, q of H
          const cplx sw = {s * w.re, s * w.im}, cw = {c * w.re, c * w.im};
#pragma unroll
          for (int k = 0; k < D; ++k) {
            const cplx yp = H[p][k], yq = H[q][k];
            const cplx a1 = cmul(sw, yq), a2 = cmul(cw, yq);
            H[p][k] = cplx{c * yp.re - a1.re, c * yp.im - a1.im};
            H[q][k] = cplx{s * yp.re + a2.re, s * yp.im + a2.im};
          }
          H[p][q] = cplx{0.0, 0.0};
          H[q][p] = cplx{0.0, 0.0};
          // the rotated diagonal from the classical update a - t |h|, b + t |h| (one rounding each) instead
          // of the two-sided products above (six): the eigenvalue noise of a segment, ~eps ||H||, is what
          // the propagator chain accumulates over the pulse (DESIGN 4.3)
          H[p][p] = cplx{fma(-t, beta, a), 0.0};
          H[q][q] = cplx{fma(t, beta, b), 0.0};
        }
      }
    }
  }
  // unit columns: the products of ~30 rotations leave |v_j|^2 = 1 + O(1e-15) with a slight BIAS, and a
  // biased norm of P_g = V exp(-i D dt) V^+ grows linearly along the propagator chain
#pragma unroll
  for (int j = 0; j < D; ++j) {
    double n2 = 0.0;
#pragma unroll
    for (int r = 0; r < D; ++r) n2 += V[r][j].re * V[r][j].re + V[r][j].im * V[r][j].im;
    const double f = fma(-0.5, n2, 1.5);   // 1 / sqrt(n2) to second order in (n2 - 1)
#pragma unroll
    for (int r = 0; r < D; ++r) V[r][j] = cplx{V[r][j].re * f, V[r][j].im * f};
  }
  // (a NaN / Inf entry can "converge" because a rotation sets its pivot to exactly zero)
  if (!converged || !isfinite(norm2)) atomicAdd(not_converged, 1);

  // ---- ascending order (stable), as numpy.linalg.eigh returns them: rank of every eigenvalue
  double ev[D];
  int rank[D];
#pragma unroll
  for (int j = 0; j < D; ++j) ev[j] = ldexp(H[j][j].re, scale_exp);
#pragma unroll
  for (int j = 0; j < D; ++j) {
    int rk = 0;
#pragma unroll
    for (int i = 0; i < D; ++i) rk += (ev[i] < ev[j]) || (ev[i] == ev[j] && i < j);
    rank[j] = rk;
  }
#pragma unroll
  for (int j = 0; j < D; ++j) {  // column j of V goes to position rank[j] (compile-time register indices)
    eigvals[(size_t)g * D + rank[j]] = ev[j];
#pragma unroll
    for (int r = 0; r < D; ++r) {
      eigvecs[2 * ((size_t)g * DD + r * D + rank[j])] = V[r][j].re;
      eigvecs[2 * ((size_t)g * DD + r * D + rank[j]) + 1] = V[r][j].im;
    }
  }

  // ---- P_g = V exp(-i D dt) V^dagger  (order of eigenpairs is irrelevant here)
  const double dtg = dt[g];
  double cs[D], sn[D];
#pragma unroll
  for (int j = 0; j < D; ++j) sincos(-dtg * ev[j], &sn[j], &cs[j]);
#pragma unroll
  for (int r = 0; r < D; ++r) {
#pragma unroll
    for (int c = 0; c < D; ++c) {
      cplx acc = {0.0, 0.0};
#pragma unroll
      for (int j = 0; j < D; ++j) {
        const cplx vv = cmulc(V[r][j], V[c][j]);
        acc.re += vv.re * cs[j] - vv.im * sn[j];
        acc.im += vv.re * sn[j] + vv.im * cs[j];
      }
      P[r * D + c] = make_double2(acc.re, acc.im);
    }
  }
}

template <int D>
__global__ void __launch_bounds__(128)
diag_small_kernel(int G, int n_cops, const double* __restrict__ c_opers,
                  const double* __restrict__ c_coeffs, const double* __restrict__ dt,
                  double* __restrict__ eigvals, double* __restrict__ eigvecs,
                  double* __restrict__ piecewise, int* __restrict__ not_converged) {
  constexpr int DD = D * D;
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= G) return;
  double2 P[DD];
  diag_small_one<D>(G, g, n_cops, c_opers, c_coeffs, dt, eigvals, eigvecs, not_converged, P);
#pragma unroll
  for (int e = 0; e < DD; ++e) reinterpret_cast<double2*>(piecewise)[(size_t)g * DD + e] = P[e];
}

// ---- parallel scan of Q_{g+1} = P_g Q_g -----------------------------------------------------------
// phase A: warp c forms the running products inside chunk c: local[g+1] = P_g ... P_{c*L}, written to
//          propagators[g+1]; the chunk total goes to totals[c].
__global__ void __launch_bounds__(DIAG_WARPS * 32)
scan_local_kernel(int G, int d, int L, const double* __restrict__ piecewise,
                  double* __restrict__ propagators, double* __restrict__ totals) {
  extern __shared__ double smem[];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int c = blockIdx.x * DIAG_WARPS + warp;
  const int g0 = c * L;
  if (g0 >= G) return;
  const int g1 = min(G, g0 + L);
  const int dd = d * d;
  double* R0 = smem + (size_t)warp * 4 * dd;
  double* R1 = R0 + 2 * dd;
  for (int e = lane; e < dd; e += 32) {
    sts_c(R0, e, cplx{piecewise[2 * ((size_t)g0 * dd + e)], piecewise[2 * ((size_t)g0 * dd + e) + 1]});
  }
  __syncwarp();
  for (int e = lane; e < 2 * dd; e += 32) propagators[(size_t)(g0 + 1) * 2 * dd + e] = R0[e];
  double* cur = R0;
  double* nxt = R1;
  for (int g = g0 + 1; g < g1; ++g) {
    const double* Pg = piecewise + (size_t)g * 2 * dd;
    for (int e = lane; e < dd; e += 32) {
      const int r = e / d, col = e % d;
      cplx acc = {0.0, 0.0};
      for (int j = 0; j < d; ++j) {
        const cplx a = {Pg[2 * (r * d + j)], Pg[2 * (r * d + j) + 1]};
        const cplx b = lds_c(cur, j * d + col);
        acc.re += a.re * b.re - a.im * b.im;
        acc.im += a.re * b.im + a.im * b.re;
      }
      sts_c(nxt, e, acc);
      propagators[2 * ((size_t)(g + 1) * dd + e)] = acc.re;
      propagators[2 * ((size_t)(g + 1) * dd + e) + 1] = acc.im;
    }
    __syncwarp();
    double* tmp = cur;
    cur = nxt;
    nxt = tmp;
  }
  for (int e = lane; e < 2 * dd; e += 32) totals[(size_t)c * 2 * dd + e] = cur[e];
}

// phase B: one warp, exclusive prefix over the chunk totals: prefix[c] = totals[c-1] ... totals[0]
__global__ void __launch_bounds__(32)
scan_totals_kernel(int n_chunks, int d, const double* __restrict__ totals,
                   double* __restrict__ prefix) {
  extern __shared__ double smem[];
  const int lane = threadIdx.x;
  const int dd = d * d;
  double* cur = smem;
  double* nxt = smem + 2 * dd;
  for (int e = lane; e < dd; e += 32) {
    const int r = e / d, col = e % d;
    sts_c(cur, e, cplx{r == col ? 1.0 : 0.0, 0.0});
  }
  __syncwarp();
  for (int c = 0; c < n_chunks; ++c) {
    for (int e = lane; e < 2 * dd; e += 32) prefix[(size_t)c * 2 * dd + e] = cur[e];
    if (c + 1 == n_chunks) break;
    const double* T = totals + (size_t)c * 2 * dd;
    for (int e = lane; e < dd; e += 32) {
      const int r = e / d, col = e % d;
      cplx acc = {0.0, 0.0};
      for (int j = 0; j < d; ++j) {
        const cplx a = {T[2 * (r * d + j)], T[2 * (r * d + j) + 1]};
        const cplx b = lds_c(cur, j * d + col);
        acc.re += a.re * b.re - a.im * b.im;
        acc.im += a.re * b.im + a.im * b.re;
      }
      sts_c(nxt, e, acc);
    }
    __syncwarp();
    double* tmp = cur;
    cur = nxt;
    nxt = tmp;
  }
}

// phase C: propagators[g+1] = local[g+1] * prefix[chunk(g)]; propagators[0] = 1. One thread per matrix
// element; the local products live in a scratch buffer so nothing is updated in place.
__global__ void scan_apply_from_kernel(int G, int d, int L, const double* __restrict__ local,
                                       const double* __restrict__ prefix,
                                       double* __restrict__ propagators) {
  const int dd = d * d;
  const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (tid >= (size_t)(G + 1) * dd) return;
  const int gi = (int)(tid / dd);
  const int e = (int)(tid % dd);
  const int r = e / d, col = e % d;
  if (gi == 0) {
    propagators[2 * tid] = (r == col) ? 1.0 : 0.0;
    propagators[2 * tid + 1] = 0.0;
    return;
  }
  const int c = (gi - 1) / L;
  const double* Lm = local + (size_t)gi * 2 * dd;
  if (c == 0) {
    propagators[2 * tid] = Lm[2 * e];
    propagators[2 * tid + 1] = Lm[2 * e + 1];
    return;
  }
  const double* T = prefix + (size_t)c * 2 * dd;
  cplx acc = {0.0, 0.0};
  for (int j = 0; j < d; ++j) {
    const cplx a = {Lm[2 * (r * d + j)], Lm[2 * (r * d + j) + 1]};
    const cplx b = {T[2 * (j * d + col)], T[2 * (j * d + col) + 1]};
    acc.re += a.re * b.re - a.im * b.im;
    acc.im += a.re * b.im + a.im * b.re;
  }
  propagators[2 * tid] = acc.re;
  propagators[2 * tid + 1] = acc.im;
}
}  // namespace

// ---- small matrices (d <= 4): one thread per matrix, Hillis-Steele scan through shared memory -------
// R_i = P_i P_{i-1} ... P_{block start}; log2(NT) steps of one register-resident matmul each instead of
// NT dependent steps that each wait on a global load (first version: 77 + 53 us for G = 1e4, d = 2).
namespace {

template <int D>
__device__ __forceinline__ void matmul_reg(const double2 (&a)[D * D], const double2 (&b)[D * D],
                                           double2 (&c)[D * D]) {
#pragma unroll
  for (int r = 0; r < D; ++r) {
#pragma unroll
    for (int col = 0; col < D; ++col) {
      double re = 0.0, im = 0.0;
#pragma unroll
      for (int j = 0; j < D; ++j) {
        const double2 x = a[r * D + j], y = b[j * D + col];
        re += x.x * y.x - x.y * y.y;
        im += x.x * y.y + x.y * y.x;
      }
      c[r * D + col] = make_double2(re, im);
    }
  }
}

// arguments of the fused diagonalisation (in == nullptr: thread g first diagonalises segment g and
// scans its propagator straight out of registers -- no diag launch, no piecewise array)
struct DiagArgs {
  int n_cops;
  const double* c_opers;
  const double* c_coeffs;
  const double* dt;
  double* eigvals;
  double* eigvecs;
  int* not_converged;
};

template <int D, int NT>
__global__ void __launch_bounds__(NT)
scan_block_kernel(int n, const double2* __restrict__ in, double2* __restrict__ local,
                  double2* __restrict__ totals, const DiagArgs da) {
  extern __shared__ double2 sbuf[];  // [2][D*D][NT], element-major so that lanes hit distinct banks
  constexpr int DD = D * D;
  const int i = threadIdx.x;
  const int g = blockIdx.x * NT + i;
  double2 m[DD];
  if (g < n) {
    if (in != nullptr) {
#pragma unroll
      for (int e = 0; e < DD; ++e) m[e] = in[(size_t)g * DD + e];
    } else {
      diag_small_one<D>(n, g, da.n_cops, da.c_opers, da.c_coeffs, da.dt, da.eigvals, da.eigvecs,
                        da.not_converged, m);
    }
  } else {  // identity padding
#pragma unroll
    for (int e = 0; e < DD; ++e) m[e] = make_double2((e / D == e % D) ? 1.0 : 0.0, 0.0);
  }
  int cur = 0;
  for (int o = 1; o < NT; o <<= 1) {
    double2* buf = sbuf + (size_t)cur * DD * NT;
#pragma unroll
    for (int e = 0; e < DD; ++e) buf[e * NT + i] = m[e];
    __syncthreads();
    if (i >= o) {
      double2 other[DD], prod[DD];
#pragma unroll
      for (int e = 0; e < DD; ++e) other[e] = buf[e * NT + i - o];
      matmul_reg<D>(m, other, prod);
#pragma unroll
      for (int e = 0; e < DD; ++e) m[e] = prod[e];
    }
    cur ^= 1;
  }
  if (g < n) {
#pragma unroll
    for (int e = 0; e < DD; ++e) local[(size_t)g * DD + e] = m[e];
  }
  if (i == NT - 1) {
#pragma unroll
    for (int e = 0; e < DD; ++e) totals[(size_t)blockIdx.x * DD + e] = m[e];
  }
}

// out[i + shift] = local[i] * incl_totals[block(i) - 1]  (identity for block 0); with shift = 1 the
// kernel also writes the identity to out[0] (the propagators array starts with Q_0 = 1).
// Same, but the inclusive product of the block totals is formed HERE (every block multiplies up the
// totals of the source blocks before it, at most SCAN_PREFIX_MAX of them) instead of two more launches
// for a scan over a few dozen matrices.  blockDim.x == NT >= SCAN_PREFIX_MAX / 2.
constexpr int SCAN_PREFIX_MAX = 96;
template <int D, int NT>
__global__ void __launch_bounds__(NT)
scan_apply_prefix_kernel(int n, int shift, const double2* __restrict__ local,
                         const double2* __restrict__ totals, double2* __restrict__ out) {
  constexpr int DD = D * D;
  __shared__ double2 prefix[DD];
  __shared__ double2 tot[SCAN_PREFIX_MAX * DD];
  const int blk = blockIdx.x;
  const int g = blk * NT + threadIdx.x;
  // the totals before this block come in with one coalesced load (a chain of dependent global loads
  // would cost an L2 round trip per matrix), then an ORDERED tree product in shared memory: after the
  // level with stride s, tot[i] (i a multiple of 2 s) holds T_{i+2s-1} ... T_i -- log2(blk) levels of
  // one register matmul each instead of a chain of blk - 1 (60 us for 79 4 x 4 totals).
  for (int e = threadIdx.x; e < blk * DD; e += NT) tot[e] = totals[e];
  __syncthreads();
  for (int stride = 1; stride < blk; stride <<= 1) {
    const int i = threadIdx.x * 2 * stride;
    const bool act = i + stride < blk;
    double2 prod[DD];
    if (act) {
      double2 later[DD], earlier[DD];
#pragma unroll
      for (int e = 0; e < DD; ++e) {
        later[e] = tot[(i + stride) * DD + e];
        earlier[e] = tot[i * DD + e];
      }
      matmul_reg<D>(later, earlier, prod);
    }
    __syncthreads();
    if (act) {
#pragma unroll
      for (int e = 0; e < DD; ++e) tot[i * DD + e] = prod[e];
    }
    __syncthreads();
  }
  if (threadIdx.x < DD && blk > 0) prefix[threadIdx.x] = tot[threadIdx.x];
  if (g == 0 && shift) {
#pragma unroll
    for (int e = 0; e < DD; ++e) out[e] = make_double2((e / D == e % D) ? 1.0 : 0.0, 0.0);
  }
  __syncthreads();
  if (g >= n) return;
  double2 a[DD], r[DD];
#pragma unroll
  for (int e = 0; e < DD; ++e) a[e] = local[(size_t)g * DD + e];
  if (blk == 0) {
#pragma unroll
    for (int e = 0; e < DD; ++e) r[e] = a[e];
  } else {
    double2 b[DD];
#pragma unroll
    for (int e = 0; e < DD; ++e) b[e] = prefix[e];
    matmul_reg<D>(a, b, r);
  }
#pragma unroll
  for (int e = 0; e < DD; ++e) out[(size_t)(g + shift) * DD + e] = r[e];
}

template <int D, int NT>
__global__ void __launch_bounds__(256)
scan_apply_small_kernel(int n, int shift, const double2* __restrict__ local,
                        const double2* __restrict__ incl_totals, double2* __restrict__ out) {
  constexpr int DD = D * D;
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g == 0 && shift) {
#pragma unroll
    for (int e = 0; e < DD; ++e) out[e] = make_double2((e / D == e % D) ? 1.0 : 0.0, 0.0);
  }
  if (g >= n) return;
  double2 a[DD], r[DD];
#pragma unroll
  for (int e = 0; e < DD; ++e) a[e] = local[(size_t)g * DD + e];
  const int blk = g / NT;
  if (blk == 0) {
#pragma unroll
    for (int e = 0; e < DD; ++e) r[e] = a[e];
  } else {
    double2 b[DD];
#pragma unroll
    for (int e = 0; e < DD; ++e) b[e] = incl_totals[(size_t)(blk - 1) * DD + e];
    matmul_reg<D>(a, b, r);
  }
#pragma unroll
  for (int e = 0; e < DD; ++e) out[(size_t)(g + shift) * DD + e] = r[e];
}

// the scan kernel instances a diagonalisation launched, each named once in order of first launch, and
// the number of scan levels (the dispatch record's prologue and S)
struct ScanTrace {
  std::string kernels;
  int levels = 0;
  void add(const char* name) {
    if (kernels.find(name) != std::string::npos) return;
    if (!kernels.empty()) kernels += '+';
    kernels += name;
  }
  template <int D, int NT>
  void add(const char* kernel) {
    char name[64];
    snprintf(name, sizeof name, "%s<%d, %d>", kernel, D, NT);
    add(name);
  }
};

// inclusive scan of n matrices `in` -> out[i + shift]; recursive over the block totals
template <int D, int NT>
int scan_small(ffb_ctx* ctx, ScanTrace& trace, int n, const double2* in, double2* out, int shift,
               const DiagArgs& da = DiagArgs{}) {
  constexpr int DD = D * D;
  const int nb = ceil_div(n, NT);
  trace.levels++;
  trace.add<D, NT>("scan_block_kernel");
  DevBuf local, totals, totals_incl;
  FFB_TRY(local.alloc(ctx, (size_t)n * DD * 16));
  FFB_TRY(totals.alloc(ctx, (size_t)nb * DD * 16));
  const size_t smem = (size_t)2 * DD * NT * sizeof(double2);
  auto kern = scan_block_kernel<D, NT>;
  FFB_TRY(ffb_func_smem(ctx, kern, smem));
  kern<<<nb, NT, smem, ctx->stream>>>(n, in, local.as<double2>(), totals.as<double2>(), da);
  FFB_LAUNCHED(ctx);
  if (nb <= SCAN_PREFIX_MAX) {  // few blocks: their totals are combined inside the apply kernel
    trace.add<D, NT>("scan_apply_prefix_kernel");
    scan_apply_prefix_kernel<D, NT><<<nb, NT, 0, ctx->stream>>>(
        n, shift, local.as<double2>(), totals.as<double2>(), out);
    FFB_LAUNCHED(ctx);
    return FFB_OK;
  }
  if (nb > 1) {
    FFB_TRY(totals_incl.alloc(ctx, (size_t)nb * DD * 16));
    FFB_TRY((scan_small<D, NT>(ctx, trace, nb, totals.as<double2>(), totals_incl.as<double2>(), 0)));
  }
  trace.add<D, NT>("scan_apply_small_kernel");
  scan_apply_small_kernel<D, NT><<<ceil_div(n + 1, 256), 256, 0, ctx->stream>>>(
      n, shift, local.as<double2>(), nb > 1 ? totals_incl.as<double2>() : nullptr, out);
  FFB_LAUNCHED(ctx);
  return FFB_OK;
}

}  // namespace

int ffbi_diagonalize(ffb_ctx* ctx, int G, int d, int n_cops, const double* c_opers,
                     const double* c_coeffs, const double* dt, double* eigvals, double* eigvecs,
                     double* propagators) {
  FFB_REQUIRE(ctx, G >= 1, "diagonalize: need at least one segment (G=%d)", G);
  FFB_REQUIRE(ctx, d >= 1 && d <= MAX_D, "diagonalize: dimension d=%d outside [1, %d]", d, MAX_D);
  FFB_REQUIRE(ctx, c_coeffs == nullptr || n_cops >= 1, "diagonalize: n_cops=%d", n_cops);
  const int dd = d * d;
  int L = 8;
  while ((long long)L * L < G && L < 256) L *= 2;
  const int n_chunks = ceil_div(G, L);

  int* conv = nullptr;  // counter of matrices whose Jacobi iteration did not converge (per context)
  FFB_TRY(ffb_conv_counter(ctx, &conv));
  static const bool small_ok = !(getenv("FFB_DIAG_SMALL") && atoi(getenv("FFB_DIAG_SMALL")) == 0);
  static const bool fuse_ok = !(getenv("FFB_DIAG_FUSED") && atoi(getenv("FFB_DIAG_FUSED")) == 0);
  ffb_dispatch_record disp = {};
  disp.n_pass = G;
  ScanTrace trace;
  auto logged = [&](int rc, int per_chunk) -> int {
    if (rc != FFB_OK) return rc;
    snprintf(disp.prologue, sizeof disp.prologue, "%s", trace.kernels.c_str());
    disp.S = trace.levels;
    disp.passes_per_chunk = per_chunk;
    if (ctx->diag_dispatch_log.size() >= FFB_DISPATCH_LOG_MAX) ctx->diag_dispatch_log.pop_front();
    ctx->diag_dispatch_log.push_back(disp);
    return FFB_OK;
  };
  if (d >= 2 && d <= 4 && small_ok && fuse_ok) {
    // diagonalisation fused into the block scan: thread per segment, propagator scanned from registers
    const DiagArgs da{n_cops, c_opers, c_coeffs, dt, eigvals, eigvecs, conv};
    if (d == 2) {
      snprintf(disp.kernel, sizeof disp.kernel, "scan_block_kernel<2, 256>");
      return logged(scan_small<2, 256>(ctx, trace, G, nullptr, (double2*)propagators, 1, da), 256);
    }
    snprintf(disp.kernel, sizeof disp.kernel, "scan_block_kernel<%d, 128>", d);
    if (d == 3) return logged(scan_small<3, 128>(ctx, trace, G, nullptr, (double2*)propagators, 1, da), 128);
    return logged(scan_small<4, 128>(ctx, trace, G, nullptr, (double2*)propagators, 1, da), 128);
  }
  DevBuf piecewise, local, totals, prefix;
  FFB_TRY(piecewise.alloc(ctx, (size_t)G * dd * 16));
  FFB_TRY(local.alloc(ctx, (size_t)(G + 1) * dd * 16));
  FFB_TRY(totals.alloc(ctx, (size_t)n_chunks * dd * 16));
  FFB_TRY(prefix.alloc(ctx, (size_t)n_chunks * dd * 16));
  if (d >= 2 && d <= 4 && small_ok) {
    snprintf(disp.kernel, sizeof disp.kernel, "diag_small_kernel<%d>", d);
    const unsigned nb = (unsigned)ceil_div(G, 128);
    if (d == 2)
      diag_small_kernel<2><<<nb, 128, 0, ctx->stream>>>(G, n_cops, c_opers, c_coeffs, dt, eigvals, eigvecs,
                                                        piecewise.as<double>(), conv);
    else if (d == 3)
      diag_small_kernel<3><<<nb, 128, 0, ctx->stream>>>(G, n_cops, c_opers, c_coeffs, dt, eigvals, eigvecs,
                                                        piecewise.as<double>(), conv);
    else
      diag_small_kernel<4><<<nb, 128, 0, ctx->stream>>>(G, n_cops, c_opers, c_coeffs, dt, eigvals, eigvecs,
                                                        piecewise.as<double>(), conv);
    FFB_LAUNCHED(ctx);
  } else {
    snprintf(disp.kernel, sizeof disp.kernel, "diag_kernel");
    const size_t smem = (size_t)DIAG_WARPS * (4 * dd + 2 * d) * sizeof(double);
    FFB_CUDA(ctx, cudaFuncSetAttribute(diag_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)smem));
    diag_kernel<<<ceil_div(G, DIAG_WARPS), DIAG_WARPS * 32, smem, ctx->stream>>>(
        G, d, n_cops, c_opers, c_coeffs, dt, eigvals, eigvecs, piecewise.as<double>(),
        conv);
    FFB_LAUNCHED(ctx);
  }
  // running product Q_{g+1} = P_g ... P_0
  const double2* P = piecewise.as<double2>();
  if (d == 2) return logged(scan_small<2, 256>(ctx, trace, G, P, (double2*)propagators, 1), 256);
  if (d == 3) return logged(scan_small<3, 128>(ctx, trace, G, P, (double2*)propagators, 1), 128);
  if (d == 4) return logged(scan_small<4, 128>(ctx, trace, G, P, (double2*)propagators, 1), 128);
  {
    const size_t smem = (size_t)DIAG_WARPS * 4 * dd * sizeof(double);
    FFB_CUDA(ctx, cudaFuncSetAttribute(scan_local_kernel,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    scan_local_kernel<<<ceil_div(n_chunks, DIAG_WARPS), DIAG_WARPS * 32, smem, ctx->stream>>>(
        G, d, L, piecewise.as<double>(), local.as<double>(), totals.as<double>());
    FFB_LAUNCHED(ctx);
  }
  {
    const size_t smem = (size_t)4 * dd * sizeof(double);
    scan_totals_kernel<<<1, 32, smem, ctx->stream>>>(n_chunks, d, totals.as<double>(),
                                                     prefix.as<double>());
    FFB_LAUNCHED(ctx);
  }
  {
    const size_t n = (size_t)(G + 1) * dd;
    scan_apply_from_kernel<<<(unsigned)ceil_div_sz(n, 256), 256, 0, ctx->stream>>>(
        G, d, L, local.as<double>(), prefix.as<double>(), propagators);
    FFB_LAUNCHED(ctx);
  }
  trace.levels = 1;
  trace.kernels = "scan_local_kernel+scan_totals_kernel+scan_apply_from_kernel";
  return logged(FFB_OK, L);
}
