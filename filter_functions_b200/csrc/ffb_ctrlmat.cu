// K2 -- first-order control matrix from scratch (numeric.calculate_control_matrix_from_scratch,
// numeric.py:707-881 of the reference).
//
// Reference algorithm (numeric.py:846-869), per segment g and frequency w:
//     step[j,k,w] = e^{i w t_g} sum_{mn} Bbar^{(g)}_j[m,n] I^{(g)}_{mn}(w) Cbar^{(g)}_k[n,m]
//     I_mn(w) = (e^{i (w + E_m - E_n) dt} - 1) / (i (w + E_m - E_n)),  = dt if the denominator is 0
// with Bbar = s_j V^+ B_j V (numeric.py:98-123) and Cbar = (Q^+ V)^+ C_k (Q^+ V) (numeric.py:93-95,
// :126-141).  NumPy materialises (n_omega, d, d) temporaries per segment and contracts them with
// opt_einsum ('o,jmn,omn,knm->jko', numeric.py:843).
//
// B200 formulation.  The sum over (g, m, n) is a GEMM whose right operand is generated on the fly:
//     B[(j,k), w] = sum_{(g,kappa)} A[(j,k), (g,kappa)] * P[(g,kappa), w]
// For Hermitian noise operators and basis elements Bbar and Cbar are Hermitian, so the (m,n) and
// (n,m) terms are complex conjugates in their w-independent factor M_mn = Bbar_j[m,n] Cbar_k[n,m]:
//     M_mn I_mn + conj(M_mn) I_nm = Re(M_mn) (I_mn + I_nm) + Im(M_mn) i (I_mn - I_nm)
// and all diagonal terms share I_mm = I(w).  The left operand therefore becomes a REAL matrix with
// Kh = 1 + d(d-1) columns per segment (instead of d^2 complex ones) and the right operand the complex
// functions {I_0, S_p = I_mn + I_nm, D_p = i (I_mn - I_nm)} times the phase e^{i w t_g}: 2 + 2 d (d-1)
// real multiply-adds per (j,k) and segment-frequency pair instead of 4 d^2.  Non-Hermitian operators
// are split into Hermitian and anti-Hermitian parts (the control matrix is linear in B_j and C_k), which
// multiplies the row count by 2 (or 4) and is undone in the finalize kernel.
//
// The real GEMM runs on the FP64 tensor path (DMMA.8x8x4): M = 8 rows, N = 8 frequencies (two
// accumulator tiles per row tile: real and imaginary part of P), K = 4 consecutive segments.  Lane
// (q = lane % 4, w = lane / 4) owns frequency w of the warp's 8 and segment q of the pass's 4: it
// generates exactly the B-fragment element the instruction expects, so P never leaves registers and
// nothing of size (G, n_omega, d, d) is ever materialised.
//
// Transcendentals.  With x = w + Omega, I(x) = e^{i x dt / 2} * 2 sin(x dt / 2) / x, and the half-angle
// exponential factorises, e^{i (w + Omega) dt / 2} = e^{i w dt / 2} e^{i Omega dt / 2}: the second factor
// is precomputed per segment, the first is recomputed only when dt changes, and sin(x dt / 2) is the
// imaginary part of the product.  That leaves ONE sincos per (segment, frequency) -- the phase
// e^{i w t_g} -- instead of the 2 d^2 + 2 of the reference.  The product form cancels when
// |sin(x dt / 2)| is small (near the removable singularity x = 0, which includes the exact-zero rule of
// numeric.py:162-165); lanes below 2^-10 are re-evaluated directly with the reference's own rounding
// sequence (x = w + Omega, y = x dt) in a rarely taken warp-uniform fix-up.
//
// Software pipelining.  The operands of unit u+1 (a unit = one A column pair plus its constants) are
// generated in the same basic block as the DMMAs of unit u, so the FP64 pipe always has independent
// work: first version without it measured 71 % DMMA-pipe activity for d = 4 (profiles/).
//
// Measured on B200 (tools/microbench/fp64_peaks.cu, profiles/fp64_peaks_r01.jsonl): DFMA peak 36.95
// TFLOP/s, DMMA peak 37.14 TFLOP/s, and the two do NOT overlap (one FP64 pipe, 64 lanes/clk/SM); DMMA
// is used because it needs 1/8 of the issue slots and shares the operands through the fragment layout.
#include <cstdlib>

#include "ffb_common.cuh"
#include "ffb_device.cuh"
#include "ffb_phase.cuh"


namespace {

// ------------------------------------------------------------------------------------------------
// math helpers
// ------------------------------------------------------------------------------------------------
// Table-driven variant for the thread-per-frequency kernel: x = k pi/128 + r, |r| <= pi/256, so sin r
// and cos r need three terms each (remainders r^7/5040 < 1e-17, r^8/40320 < 1e-20) and the quadrant
// logic disappears into the 256-entry table (sin, cos)(k pi/128) held in shared memory:
// 15 FP64 operations and one LDS.128 instead of 22 and ~12 integer/select instructions.  On sm_100 an
// FP64 instruction holds the scheduler's dispatch port for 2 cycles and nothing else issues meanwhile
// (measured: time = 2 N_fp64 + 16 N_dmma + N_other on every variant of these kernels), so both counts
// matter.  Same absolute accuracy as sincos_cw (table entries and the reduction are exact to 1 ulp).
constexpr int TRIG_TABLE_SIZE = 256;
// (the constants of the reduction and the two polynomials are in TrigConsts, passed as kernel parameters)

__global__ void trig_table_kernel(double2* __restrict__ table) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= TRIG_TABLE_SIZE) return;
  double sn, cs;
  sincospi((double)k / 128.0, &sn, &cs);
  table[k] = make_double2(sn, cs);
}

constexpr double TINY_OMEGA = 1e-290;               // |w| below this is treated as the exact zero

__device__ __forceinline__ void pair_from_index(int p, int d, int& m, int& n) {
  m = 0;
  while (p >= d - 1 - m) {
    p -= d - 1 - m;
    ++m;
  }
  n = m + 1 + p;
}

// ------------------------------------------------------------------------------------------------
// prologue 1: eigenbasis transforms (omega independent, O(G (n_nops + n_basis) d^3))
//   Bbar[g, jr] = s_j^{(g)} herm-part(V^+ B_j V),   Cbar[g, kr] = herm-part(U^+ C_k U),  U = Q_g^+ V_g
// one block per (segment, operator slice): blockIdx.y strides over the operators, so that short pulses
// with many operators (a one-segment gate with 270 16x16 operators took 1.7 ms in a single block) still
// fill the machine; operators of a slice are transformed one after the other through shared memory.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
transform_kernel(int G, int d, int n_nops, int n_basis, int parts_j, int parts_k,
                 const double* __restrict__ eigvecs, const double* __restrict__ propagators,
                 const double* __restrict__ n_opers, const double* __restrict__ n_coeffs,
                 const double* __restrict__ basis, double* __restrict__ Bbar,
                 double* __restrict__ Cbar) {
  extern __shared__ double sm[];
  const int g = blockIdx.x;
  const int dd = d * d;
  double* V = sm;            // d*d complex
  double* U = V + 2 * dd;    // d*d complex
  double* T = U + 2 * dd;    // scratch
  double* X = T + 2 * dd;    // transformed operator
  const double* Vg = eigvecs + (size_t)g * 2 * dd;
  const double* Qg = propagators + (size_t)g * 2 * dd;
  for (int e = threadIdx.x; e < 2 * dd; e += blockDim.x) V[e] = Vg[e];
  __syncthreads();
  for (int e = threadIdx.x; e < dd; e += blockDim.x) {
    const int a = e / d, b = e % d;
    cplx acc = {0.0, 0.0};
    for (int c = 0; c < d; ++c) {  // U[a][b] = sum_c conj(Q[c][a]) V[c][b]
      const cplx qv = {Qg[2 * (c * d + a)], -Qg[2 * (c * d + a) + 1]};
      const cplx vv = {V[2 * (c * d + b)], V[2 * (c * d + b) + 1]};
      acc = cadd(acc, cmul(qv, vv));
    }
    U[2 * e] = acc.re;
    U[2 * e + 1] = acc.im;
  }
  __syncthreads();
  const int n_ops = n_nops + n_basis;
  for (int op = blockIdx.y; op < n_ops; op += gridDim.y) {
    const bool is_noise = op < n_nops;
    const double* O = is_noise ? n_opers + (size_t)op * 2 * dd : basis + (size_t)(op - n_nops) * 2 * dd;
    const double* W = is_noise ? V : U;
    for (int e = threadIdx.x; e < dd; e += blockDim.x) {  // T = O W
      const int a = e / d, b = e % d;
      cplx acc = {0.0, 0.0};
      for (int c = 0; c < d; ++c) {
        const cplx o = {O[2 * (a * d + c)], O[2 * (a * d + c) + 1]};
        const cplx w = {W[2 * (c * d + b)], W[2 * (c * d + b) + 1]};
        acc = cadd(acc, cmul(o, w));
      }
      T[2 * e] = acc.re;
      T[2 * e + 1] = acc.im;
    }
    __syncthreads();
    for (int e = threadIdx.x; e < dd; e += blockDim.x) {  // X = W^+ T
      const int a = e / d, b = e % d;
      cplx acc = {0.0, 0.0};
      for (int c = 0; c < d; ++c) {
        const cplx w = {W[2 * (c * d + a)], -W[2 * (c * d + a) + 1]};
        const cplx t = {T[2 * (c * d + b)], T[2 * (c * d + b) + 1]};
        acc = cadd(acc, cmul(w, t));
      }
      X[2 * e] = acc.re;
      X[2 * e + 1] = acc.im;
    }
    __syncthreads();
    const int parts = is_noise ? parts_j : parts_k;
    const double scale = is_noise ? n_coeffs[(size_t)op * G + g] : 1.0;
    double* dst = is_noise ? Bbar + ((size_t)g * n_nops * parts_j + (size_t)op * parts_j) * 2 * dd
                           : Cbar + ((size_t)g * n_basis * parts_k + (size_t)(op - n_nops) * parts_k) * 2 * dd;
    for (int e = threadIdx.x; e < dd; e += blockDim.x) {
      const int a = e / d, b = e % d;
      const cplx x = {X[2 * e], X[2 * e + 1]};
      const cplx xt = {X[2 * (b * d + a)], -X[2 * (b * d + a) + 1]};  // conj(X[b][a])
      // Hermitian part (X + X^+)/2 and, if requested, (X - X^+)/(2i)
      dst[2 * e] = scale * 0.5 * (x.re + xt.re);
      dst[2 * e + 1] = scale * 0.5 * (x.im + xt.im);
      if (parts == 2) {
        dst[2 * dd + 2 * e] = scale * 0.5 * (x.im - xt.im);
        dst[2 * dd + 2 * e + 1] = -scale * 0.5 * (x.re - xt.re);
      }
    }
    __syncthreads();
  }
}

// Small Hilbert spaces (d <= 4): one THREAD per (segment, operator), everything in registers.  The
// block-per-segment kernel above spends its time in __syncthreads for 2x2 matrices (66 us for
// G = 1e4, d = 2 in the first version).
// transform of ONE operator of ONE segment: op < n_nops -> s_op V^+ B_op V, else U^+ C_{op - n_nops} U with
// U = Q_g^+ V_g; the Hermitian part (and, if parts == 2, the anti-Hermitian part / i) go to dst
template <int D>
__device__ __forceinline__ void transform_small_one(int G, int g, int op, int n_nops, int parts,
                                                    const double2* __restrict__ eigvecs,
                                                    const double2* __restrict__ propagators,
                                                    const double2* __restrict__ n_opers,
                                                    const double* __restrict__ n_coeffs,
                                                    const double2* __restrict__ basis, double2* dst) {
  constexpr int DD = D * D;
  const bool is_noise = op < n_nops;
  double2 W[DD];
  {
    double2 V[DD];
#pragma unroll
    for (int e = 0; e < DD; ++e) V[e] = eigvecs[(size_t)g * DD + e];
    if (is_noise) {
#pragma unroll
      for (int e = 0; e < DD; ++e) W[e] = V[e];
    } else {  // W = Q_g^+ V_g
      double2 Q[DD];
#pragma unroll
      for (int e = 0; e < DD; ++e) Q[e] = propagators[(size_t)g * DD + e];
#pragma unroll
      for (int a = 0; a < D; ++a) {
#pragma unroll
        for (int b = 0; b < D; ++b) {
          double re = 0.0, im = 0.0;
#pragma unroll
          for (int c = 0; c < D; ++c) {
            const double2 qv = Q[c * D + a], vv = V[c * D + b];  // conj(Q[c][a]) * V[c][b]
            re += qv.x * vv.x + qv.y * vv.y;
            im += qv.x * vv.y - qv.y * vv.x;
          }
          W[a * D + b] = make_double2(re, im);
        }
      }
    }
  }
  const double2* O = is_noise ? n_opers + (size_t)op * DD : basis + (size_t)(op - n_nops) * DD;
  double2 T[DD];
#pragma unroll
  for (int a = 0; a < D; ++a) {
#pragma unroll
    for (int b = 0; b < D; ++b) {  // T = O W
      double re = 0.0, im = 0.0;
#pragma unroll
      for (int c = 0; c < D; ++c) {
        const double2 o = O[a * D + c], w = W[c * D + b];
        re += o.x * w.x - o.y * w.y;
        im += o.x * w.y + o.y * w.x;
      }
      T[a * D + b] = make_double2(re, im);
    }
  }
  double2 X[DD];
#pragma unroll
  for (int a = 0; a < D; ++a) {
#pragma unroll
    for (int b = 0; b < D; ++b) {  // X = W^+ T
      double re = 0.0, im = 0.0;
#pragma unroll
      for (int c = 0; c < D; ++c) {
        const double2 w = W[c * D + a], t = T[c * D + b];
        re += w.x * t.x + w.y * t.y;
        im += w.x * t.y - w.y * t.x;
      }
      X[a * D + b] = make_double2(re, im);
    }
  }
  const double scale = is_noise ? n_coeffs[(size_t)op * G + g] : 1.0;
#pragma unroll
  for (int a = 0; a < D; ++a) {
#pragma unroll
    for (int b = 0; b < D; ++b) {
      const double2 x = X[a * D + b], xt = X[b * D + a];  // xt -> conj below
      dst[a * D + b] = make_double2(scale * 0.5 * (x.x + xt.x), scale * 0.5 * (x.y - xt.y));
      if (parts == 2) {
        dst[DD + a * D + b] = make_double2(scale * 0.5 * (x.y + xt.y), -scale * 0.5 * (x.x - xt.x));
      }
    }
  }
}

template <int D>
__global__ void __launch_bounds__(128)
transform_small_kernel(int G, int n_nops, int n_basis, int parts_j, int parts_k,
                       const double2* __restrict__ eigvecs, const double2* __restrict__ propagators,
                       const double2* __restrict__ n_opers, const double* __restrict__ n_coeffs,
                       const double2* __restrict__ basis, double2* __restrict__ Bbar,
                       double2* __restrict__ Cbar) {
  constexpr int DD = D * D;
  const int n_ops = n_nops + n_basis;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)G * n_ops) return;
  const int g = (int)(idx / n_ops), op = (int)(idx % n_ops);
  const bool is_noise = op < n_nops;
  double2* dst = is_noise ? Bbar + ((size_t)g * n_nops * parts_j + (size_t)op * parts_j) * DD
                          : Cbar + ((size_t)g * n_basis * parts_k + (size_t)(op - n_nops) * parts_k) * DD;
  transform_small_one<D>(G, g, op, n_nops, is_noise ? parts_j : parts_k, eigvecs, propagators, n_opers,
                         n_coeffs, basis, dst);
}

// Centre of chunk c of L segments.  On the banded route (see band_eval_kernel) the stream carries the segment
// start times relative to the centre of their chunk, so that the partial sum of a chunk is a smooth function
// of omega of exponential type T_c / 2; the evaluation kernel puts e^{i w t_c} back with the same t_c.
__device__ __forceinline__ double chunk_centre(const double* __restrict__ t, const double* __restrict__ dt,
                                               int G, int L, int c) {
  const int g0 = c * L, g1 = min(G, g0 + L) - 1;
  return 0.5 * (t[g0] + (t[g1] + dt[g1]));
}

// ------------------------------------------------------------------------------------------------
// prologue 2: the operand stream of the main kernel.
// Per row block rb and pass (4 consecutive segments) the stream holds 1 + n_pairs units:
//   diag unit   : A column [MT][32], t[4], dt[4]
//   pair unit p : A column Re [MT][32], A column Im [MT][32], Omega[4], cos(Omega dt/2)[4], sin(Omega dt/2)[4]
// An A column holds, for lane l = 4*row_in_tile + q, the coefficient of row 8*mt + row_in_tile and
// segment 4*pass + q -- exactly the DMMA A-fragment, so the main kernel loads it with one LDS.64.
// ------------------------------------------------------------------------------------------------
struct StreamGeom {
  int MT;          // row tiles per row block
  int n_rb;        // row blocks
  int n_pass;      // ceil(G / 4); G in transposed mode
  int n_pairs;     // pair UNITS per pass: d (d-1) / 2; ceil(d (d-1) / 8) in transposed mode
  int real_pairs;  // d (d-1) / 2
  int transposed;  // 1: the 4 K-slots of a unit are 4 level pairs of ONE segment (short pulses)
  int diag_unit;   // doubles
  int pair_unit;   // doubles
  size_t pass_doubles;
  size_t rb_doubles;
};

// Regular layout: the K = 4 slots of a DMMA are 4 consecutive segments, so a pulse of G segments costs
// ceil(G / 4) (1 + 2 n_pairs) A columns.  For short pulses (gate pulses of one or two segments, the
// constituents of a concatenation) most of those slots would be padding; the transposed layout puts 4
// level pairs (m, n) of the SAME segment into the K slots instead: G (1 + 2 ceil(n_pairs / 4)) columns.
// The main kernel is the same for both -- a lane's slot constants (Omega, e^{i Omega dt / 2}) are
// per-slot already, and the per-lane segment state (phase, dt) is simply equal across the 4 slots.
__host__ __device__ inline StreamGeom make_geom(int rows, int G, int d, int MT) {
  StreamGeom s;
  s.MT = MT;
  s.n_rb = ((rows + 7) / 8 + MT - 1) / MT;
  s.real_pairs = d * (d - 1) / 2;
  const long long cost_regular = (long long)((G + 3) / 4) * (1 + 2 * s.real_pairs);
  const long long cost_transposed = (long long)G * (1 + 2 * ((s.real_pairs + 3) / 4));
  s.transposed = (s.real_pairs >= 1 && cost_transposed < cost_regular) ? 1 : 0;
  s.n_pass = s.transposed ? G : (G + 3) / 4;
  s.n_pairs = s.transposed ? (s.real_pairs + 3) / 4 : s.real_pairs;
  s.diag_unit = MT * 32 + 8;
  s.pair_unit = 2 * MT * 32 + 12;
  s.pass_doubles = (size_t)s.diag_unit + (size_t)s.n_pairs * s.pair_unit;
  s.rb_doubles = s.pass_doubles * s.n_pass;
  return s;
}

// One block per (row block, pass).  A thread takes one (row, K slot) of the pass and walks its units
// (diagonal term, then the level pairs), so the index arithmetic is done once per 1 + 2 n_pairs values
// instead of once per value (the first version decoded every double of the stream on its own: ~300
// instructions per value, 143 us for the 100 MB stream of d = 4, G = 1e4), and consecutive threads write
// consecutive addresses of every A column.  STAGED: the transformed operators of the pass's segments are
// copied to shared memory first (coalesced); used when they fit, i.e. for small d.
template <bool STAGED>
__global__ void __launch_bounds__(256)
assemble_kernel(StreamGeom geo, int G, int d, int rows, int n_jrows, int n_krows, int split_rf,
                int chunk_segs, const double* __restrict__ Bbar_g, const double* __restrict__ Cbar_g,
                const double* __restrict__ eigvals, const double* __restrict__ dt,
                const double* __restrict__ t, double* __restrict__ stream) {
  extern __shared__ __align__(16) double stage[];
  const int dd = d * d;
  const int rb = blockIdx.x / geo.n_pass, pass = blockIdx.x % geo.n_pass;
  const int segs = geo.transposed ? 1 : 4;
  const int g0 = geo.transposed ? pass : pass * 4;  // first segment of the pass
  const double* Bbar = Bbar_g;
  const double* Cbar = Cbar_g;
  int g_base = 0;  // segment whose operators sit at index 0 of Bbar / Cbar
  if (STAGED) {
    const int n_seg = max(0, min(segs, G - g0));
    const int nb = n_jrows * 2 * dd, nc = n_krows * 2 * dd;
    double* Bs = stage;
    double* Cs = stage + (size_t)segs * nb;
    for (int e = threadIdx.x; e < n_seg * nb; e += blockDim.x) Bs[e] = Bbar_g[(size_t)g0 * nb + e];
    for (int e = threadIdx.x; e < n_seg * nc; e += blockDim.x) Cs[e] = Cbar_g[(size_t)g0 * nc + e];
    __syncthreads();
    Bbar = Bs;
    Cbar = Cs;
    g_base = g0;
  }
  double* const out = stream + (size_t)rb * geo.rb_doubles + (size_t)pass * geo.pass_doubles;
  const int col = geo.MT * 32;  // doubles per A column

  // ---- A columns
  for (int item = threadIdx.x; item < col; item += blockDim.x) {
    const int mt = item >> 5, l = item & 31;
    const int row = (rb * geo.MT + mt) * 8 + (l >> 2);
    const int slot = l & 3;
    const int g = geo.transposed ? pass : g0 + slot;
    const bool live = row < rows && g < G;
    const double* Bm = nullptr;
    const double* Cm = nullptr;
    if (live) {
      // split_rf > 0: rows ordered [(j, k >= 1) ... | (j, 0) ...] (identity basis element last, see
      // ctrlmat_static_kernel<..., SPLIT>); finalize_kernel undoes the order
      int j = row / n_krows, k = row % n_krows;
      if (split_rf > 0) {
        j = row < split_rf ? row / (n_krows - 1) : row - split_rf;
        k = row < split_rf ? 1 + row % (n_krows - 1) : 0;
      }
      Bm = Bbar + ((size_t)(g - g_base) * n_jrows + j) * 2 * dd;
      Cm = Cbar + ((size_t)(g - g_base) * n_krows + k) * 2 * dd;
    }
    // diagonal unit (transposed layout: only K slot 0 carries it)
    double diag = 0.0;
    if (live && !(geo.transposed && slot != 0))
      for (int m = 0; m < d; ++m) diag += Bm[2 * (m * d + m)] * Cm[2 * (m * d + m)];
    out[item] = diag;
    // pair units
    int m = 0, n = 1;  // level pair of unit 1 in the regular layout
    for (int u = 1; u <= geo.n_pairs; ++u) {
      const int pair = geo.transposed ? (u - 1) * 4 + slot : u - 1;
      double re = 0.0, im = 0.0;
      if (live && pair < geo.real_pairs) {
        if (geo.transposed) pair_from_index(pair, d, m, n);
        const cplx bv = {Bm[2 * (m * d + n)], Bm[2 * (m * d + n) + 1]};
        const cplx cv = {Cm[2 * (n * d + m)], Cm[2 * (n * d + m) + 1]};
        const cplx prod = cmul(bv, cv);
        re = prod.re;
        im = prod.im;
      }
      double* unit = out + geo.diag_unit + (size_t)(u - 1) * geo.pair_unit;
      unit[item] = re;
      unit[col + item] = im;
      if (!geo.transposed && ++n == d) {  // next pair (m, n) in row-major order of the upper triangle
        ++m;
        n = m + 1;
      }
    }
  }

  // ---- constants: t[4], dt[4] behind the diagonal column; Omega[4], cos[4], sin[4] behind a pair's columns
  for (int e = threadIdx.x; e < 8 + 12 * geo.n_pairs; e += blockDim.x) {
    double val = 0.0;
    if (e < 8) {
      const int which = e >> 2, slot = e & 3;
      const int g = geo.transposed ? pass : g0 + slot;
      if (g < G) val = which == 0 ? t[g] - (chunk_segs ? chunk_centre(t, dt, G, chunk_segs, g / chunk_segs) : 0.0)
                                  : dt[g];
      out[col + e] = val;
    } else {
      const int u = 1 + (e - 8) / 12, c = (e - 8) % 12;
      const int which = c >> 2, slot = c & 3;
      const int g = geo.transposed ? pass : g0 + slot;
      // padding slots (A coefficients 0) repeat the constants of the last real pair, so that they
      // take the removable-singularity fix-up only where that pair takes it anyway
      const int pair = min(geo.transposed ? (u - 1) * 4 + slot : u - 1, geo.real_pairs - 1);
      double Om = 0.0, dtg = 0.0;
      if (g < G) {
        int m, n;
        pair_from_index(pair, d, m, n);
        Om = eigvals[(size_t)g * d + m] - eigvals[(size_t)g * d + n];
        dtg = dt[g];
      }
      if (which == 0) {
        val = Om;
      } else {
        double sn, cs;
        sincos(0.5 * (Om * dtg), &sn, &cs);  // e^{i Omega dt / 2}
        val = which == 1 ? cs : sn;
      }
      out[geo.diag_unit + (size_t)(u - 1) * geo.pair_unit + 2 * col + c] = val;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// main kernel
// ------------------------------------------------------------------------------------------------
struct MainParams {
  const double* stream;
  const double* omega;
  double* partial;  // [S][rows_pad][n_omega] complex
  const int* n_live;  // banded route: frequency slots [*n_live, n_omega) are unused (nullptr: all used)
  int n_omega;
  int rows_pad;     // n_rb * MT * 8
  int n_pass;
  int n_pairs;
  int passes_per_chunk;
  // staging schedule
  int pps;          // whole passes per stage (>= 1) when n_sp == 1
  int n_sp;         // pieces per pass when a pass does not fit a stage
  int stage_doubles;  // shared-memory doubles per stage buffer
  size_t pass_doubles;
  size_t rb_doubles;
  int diag_unit;
  int pair_unit;
};

// unit boundary of piece j (in units, 0 .. 1 + n_pairs)
__host__ __device__ __forceinline__ int piece_begin(int j, int n_units, int n_sp) {
  return (int)(((long long)j * n_units) / n_sp);
}
__device__ __forceinline__ size_t unit_offset(int u, const MainParams& p) {
  return u == 0 ? 0 : (size_t)p.diag_unit + (size_t)(u - 1) * p.pair_unit;
}

// Per-lane state of the operand generator.  A lane owns ONE frequency w (of the warp's 8) and, within
// a pass, ONE segment (q = lane % 4 of the pass's 4).
struct Gen {
  double w, inv_w;        // frequency, 1/w (garbage if w_zero)
  bool w_zero;
  double ph_re, ph_im;    // e^{i w t_g} of the current pass's segment
  double dt, dt_prev;     // dt of the current segment / the one (hc, hs, J0) were computed for
  double hc, hs;          // sqrt(2) e^{i w dt / 2}
  double j0_re, j0_im;    // I(w) for dt_prev
};

// values a unit feeds to the tensor pipe: diag uses (a_re, a_im); pair uses all four (S then D)
struct Vals {
  double a_re, a_im, b_re, b_im;
};

// ---- diagonal unit: new segment -> (if dt changed) half-angle exponential and I(w); then the phase.
// Split in two so that the rarely taken branch does not cut the straight-line region in which the
// phase evaluation is interleaved with the previous unit's DMMAs.
__device__ __forceinline__ void gen_diag_slow(Gen& g, const double* unit_consts, int q) {
  g.dt = unit_consts[4 + q];
  if (__double_as_longlong(g.dt) != __double_as_longlong(g.dt_prev)) {  // never again on uniform grids
    double sn, cs;
    sincos_cw(0.5 * (g.w * g.dt), sn, cs);
    g.hc = SQRT2 * cs;
    g.hs = SQRT2 * sn;
    const double f = g.hs * g.inv_w;  // sqrt(2) sin(w dt / 2) / w
    g.j0_re = g.w_zero ? g.dt : g.hc * f;
    g.j0_im = g.w_zero ? 0.0 : g.hs * f;
    g.dt_prev = g.dt;
  }
}
__device__ __forceinline__ void gen_diag_fast(Gen& g, const double* unit_consts, int q, Vals& v) {
#ifdef FFB_EXP_NOGEN
  v.a_re = unit_consts[q]; v.a_im = g.j0_im; return;
#endif
  sincos_cw(g.w * unit_consts[q], g.ph_im, g.ph_re);
  v.a_re = g.ph_re * g.j0_re - g.ph_im * g.j0_im;
  v.a_im = g.ph_re * g.j0_im + g.ph_im * g.j0_re;
}
__device__ __forceinline__ void gen_diag(Gen& g, const double* unit_consts, int q, Vals& v) {
  gen_diag_slow(g, unit_consts, q);
  gen_diag_fast(g, unit_consts, q, v);
}

// ---- pair unit (product form): S = I(w + Om) + I(w - Om), D = i (I(w + Om) - I(w - Om)), times phase.
// Returns true if this lane needs the direct re-evaluation (cancellation in sin((w +- Om) dt / 2)).
__device__ __forceinline__ bool pair_values(const Gen& g, double Om, double Ch, double Sh, Vals& v) {
  const double t1 = g.hc * Ch, t3 = g.hs * Ch;
  const double zp_re = fma(-g.hs, Sh, t1), zp_im = fma(g.hc, Sh, t3);  // sqrt2 e^{i (w+Om) dt/2}
  const double zm_re = fma(g.hs, Sh, t1), zm_im = fma(-g.hc, Sh, t3);  // sqrt2 e^{i (w-Om) dt/2}
  const double fp = zp_im * rcp_nr(g.w + Om);
  const double fm = zm_im * rcp_nr(g.w - Om);
  const double jp_re = zp_re * fp, jp_im = zp_im * fp;
  const double jm_re = zm_re * fm, jm_im = zm_im * fm;
  const double s_re = jp_re + jm_re, s_im = jp_im + jm_im;
  const double d_re = jm_im - jp_im, d_im = jp_re - jm_re;
  v.a_re = g.ph_re * s_re - g.ph_im * s_im;
  v.a_im = g.ph_re * s_im + g.ph_im * s_re;
  v.b_re = g.ph_re * d_re - g.ph_im * d_im;
  v.b_im = g.ph_re * d_im + g.ph_im * d_re;
  return min(abs_hi(zp_im), abs_hi(zm_im)) < SMALL_SIN_HI;
}

__device__ __forceinline__ bool gen_pair(const Gen& g, const double* unit_consts, int q, Vals& v) {
#ifdef FFB_EXP_NOGEN
  v.a_re = unit_consts[q]; v.a_im = unit_consts[4 + q]; v.b_re = unit_consts[8 + q]; v.b_im = g.w; return false;
#endif
  return pair_values(g, unit_consts[q], unit_consts[4 + q], unit_consts[8 + q], v);
}

// rare path: at least one lane of the warp sits on the removable singularity.  Everything goes through
// registers (by value) so that the per-lane generator state never has its address taken.
struct Vals4 {
  double a_re, a_im, b_re, b_im;
};
__device__ __noinline__ Vals4 fix_pair(double w, double dt, double ph_re, double ph_im, double Om) {
  const cplx jp = integral_direct(w + Om, dt);
  const cplx jm = integral_direct(w - Om, dt);
  const double s_re = jp.re + jm.re, s_im = jp.im + jm.im;
  const double d_re = jm.im - jp.im, d_im = jp.re - jm.re;
  Vals4 r;
  r.a_re = ph_re * s_re - ph_im * s_im;
  r.a_im = ph_re * s_im + ph_im * s_re;
  r.b_re = ph_re * d_re - ph_im * d_im;
  r.b_im = ph_re * d_im + ph_im * d_re;
  return r;
}

template <int MT>
__device__ __forceinline__ void mma_diag(double (&acc_re)[MT][2], double (&acc_im)[MT][2],
                                         const double* unit, int lane, const Vals& v) {
#pragma unroll
  for (int mt = 0; mt < MT; ++mt) {
    const double a = unit[mt * 32 + lane];
    dmma884(acc_re[mt][0], acc_re[mt][1], a, v.a_re);
    dmma884(acc_im[mt][0], acc_im[mt][1], a, v.a_im);
  }
}

// (Experiment, round 2: the six rows (j, 0) of an identity basis element carry no pair terms, so the 96 rows of the
// d = 4 shapes need only 90 pair rows = 11.25 tiles.  Dropping the twelfth tile from the pair units outright buys 6.3 %
// (16.55 -> 15.51 ms, wrong results); the two pair rows left over would have to go through a DFMA side path costing
// about 2 % again, plus a row permutation in assemble / finalize -- not done.)
template <int MT>
__device__ __forceinline__ void mma_pair(double (&acc_re)[MT][2], double (&acc_im)[MT][2],
                                         const double* unit, int lane, const Vals& v) {
#pragma unroll
  for (int mt = 0; mt < MT; ++mt) {
    const double a = unit[mt * 32 + lane];
    dmma884(acc_re[mt][0], acc_re[mt][1], a, v.a_re);
    dmma884(acc_im[mt][0], acc_im[mt][1], a, v.a_im);
  }
#pragma unroll
  for (int mt = 0; mt < MT; ++mt) {
    const double a = unit[(MT + mt) * 32 + lane];
    dmma884(acc_re[mt][0], acc_re[mt][1], a, v.b_re);
    dmma884(acc_im[mt][0], acc_im[mt][1], a, v.b_im);
  }
}

template <int MT, int NW>
__global__ void __launch_bounds__(NW * 32, (MT <= 2 ? 3 : MT >= 10 ? 3 : 1))
ctrlmat_main_kernel(const MainParams p) {
  extern __shared__ __align__(16) double smem[];
  if (p.n_live && (int)blockIdx.x * NW * 8 >= __ldg(p.n_live)) return;  // whole CTA past the used slots
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int q = lane & 3;
  const int rb = blockIdx.y;
  const int pass_begin = blockIdx.z * p.passes_per_chunk;
  const int pass_end = min(p.n_pass, pass_begin + p.passes_per_chunk);
  const int n_units = 1 + p.n_pairs;

  Gen g;
  {
    const int w_idx = (blockIdx.x * NW + warp) * 8 + (lane >> 2);
    g.w = w_idx < p.n_omega ? p.omega[w_idx] : 1.0;
    g.w_zero = fabs(g.w) < TINY_OMEGA;
    g.inv_w = g.w_zero ? 0.0 : 1.0 / g.w;
    g.dt_prev = -1.0;
    g.dt = 0.0;
    g.hc = SQRT2;
    g.hs = 0.0;
    g.j0_re = g.j0_im = 0.0;
    g.ph_re = 1.0;
    g.ph_im = 0.0;
  }

  double acc_re[MT][2], acc_im[MT][2];
#pragma unroll
  for (int mt = 0; mt < MT; ++mt) {
    acc_re[mt][0] = acc_re[mt][1] = 0.0;
    acc_im[mt][0] = acc_im[mt][1] = 0.0;
  }

  const double* gstream = p.stream + (size_t)rb * p.rb_doubles;

  // ---- stage schedule: stage i of this chunk covers `len` doubles from `src`, holding `units` units
  const int n_passes = pass_end - pass_begin;
  const int n_stages = p.n_sp == 1 ? (n_passes + p.pps - 1) / p.pps : n_passes * p.n_sp;
  auto stage_range = [&](int i, size_t& src, int& len, int& units) {
    if (p.n_sp == 1) {
      const int p0 = pass_begin + i * p.pps;
      const int p1 = min(pass_end, p0 + p.pps);
      src = (size_t)p0 * p.pass_doubles;
      len = (int)((size_t)(p1 - p0) * p.pass_doubles);
      units = (p1 - p0) * n_units;
    } else {
      const int pass = pass_begin + i / p.n_sp;
      const int piece = i % p.n_sp;
      const int u0 = piece_begin(piece, n_units, p.n_sp);
      const int u1 = piece + 1 == p.n_sp ? n_units : piece_begin(piece + 1, n_units, p.n_sp);
      const size_t o0 = unit_offset(u0, p);
      const size_t o1 = piece + 1 == p.n_sp ? p.pass_doubles : unit_offset(u1, p);
      src = (size_t)pass * p.pass_doubles + o0;
      len = (int)(o1 - o0);
      units = u1 - u0;
    }
  };
  auto stage_load = [&](int i, double* buf) {
    size_t src;
    int len, units;
    stage_range(i, src, len, units);
    const double* gsrc = gstream + src;
    for (int e = threadIdx.x * 2; e < len; e += NW * 32 * 2) cp_async16(buf + e, gsrc + e);
  };
  auto stage_units = [&](int i) {
    size_t src;
    int len, units;
    stage_range(i, src, len, units);
    return units;
  };

  double* cur_buf = smem;
  double* nxt_buf = smem + p.stage_doubles;
  if (n_stages > 0) {
    stage_load(0, cur_buf);
    cp_async_commit();
    if (n_stages > 1) {
      stage_load(1, nxt_buf);
      cp_async_commit();
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
  }

  // ---- software-pipelined walk over the units of this chunk.  `v` always holds the operands of the
  // CURRENT unit; the operands of the next unit are generated in the same basic block as the current
  // unit's DMMAs.
  const int total_units = n_passes * n_units;
  if (p.n_pairs >= 1) {
    // fast path: tight loops over runs of pair units; all stage bookkeeping happens only on the unit
    // that ends a stage (which may be anywhere inside a pass when a pass is split into pieces).
    const int n_pairs = p.n_pairs;
    const int diag_unit = p.diag_unit, pair_unit = p.pair_unit;
    auto apply_fix = [&](bool fix, const double* consts, Vals& vn) {
      if (__any_sync(0xffffffffu, fix)) {
        if (fix) {
          const Vals4 r = fix_pair(g.w, g.dt, g.ph_re, g.ph_im, consts[q]);
          vn.a_re = r.a_re;
          vn.a_im = r.a_im;
          vn.b_re = r.b_re;
          vn.b_im = r.b_im;
        }
      }
    };
    int stage = 0;
    int left = n_stages > 0 ? stage_units(0) : 0;  // units left in the current stage (incl. current)
    // called before generating the operands of the unit that follows the LAST unit of a stage
    auto next_stage_ready = [&]() {
      cp_async_wait<0>();  // the only outstanding group is stage + 1
      __syncthreads();
    };
    // called after the DMMAs of the last unit of a stage
    auto retire_stage = [&]() {
      __syncthreads();  // everyone is done reading cur_buf
      if (stage + 2 < n_stages) {
        stage_load(stage + 2, cur_buf);
        cp_async_commit();
      }
      double* tmp = cur_buf;
      cur_buf = nxt_buf;
      nxt_buf = tmp;
      ++stage;
      left = stage_units(stage);
    };
    Vals v = {0.0, 0.0, 0.0, 0.0};
    const double* up = cur_buf;
    if (n_passes > 0) gen_diag(g, up + MT * 32, q, v);
    for (int pass = 0; pass < n_passes; ++pass) {
      Vals vn;
      // ---- diagonal unit  ||  operands of pair 0
      {
        const bool boundary = (left == 1);
        if (boundary) next_stage_ready();
        const double* pn = boundary ? nxt_buf : up + diag_unit;
        const bool fix = gen_pair(g, pn + 2 * MT * 32, q, vn);
        mma_diag<MT>(acc_re, acc_im, up, lane, v);
        apply_fix(fix, pn + 2 * MT * 32, vn);
        v = vn;
        if (boundary) retire_stage(); else --left;
        up = pn;
      }
      // ---- pair i  ||  operands of pair i + 1
      int pi = 0;
      while (pi + 1 < n_pairs) {
        const int run = min(n_pairs - 1 - pi, left - 1);  // steps that stay inside this stage
        for (int i = 0; i < run; ++i) {
          const double* pn = up + pair_unit;
          const bool fix = gen_pair(g, pn + 2 * MT * 32, q, vn);
          mma_pair<MT>(acc_re, acc_im, up, lane, v);
          apply_fix(fix, pn + 2 * MT * 32, vn);
          v = vn;
          up = pn;
        }
        pi += run;
        left -= run;
        if (pi + 1 < n_pairs) {  // left == 1: the next pair lives in the next stage
          next_stage_ready();
          const double* pn = nxt_buf;
          const bool fix = gen_pair(g, pn + 2 * MT * 32, q, vn);
          mma_pair<MT>(acc_re, acc_im, up, lane, v);
          apply_fix(fix, pn + 2 * MT * 32, vn);
          v = vn;
          retire_stage();
          up = pn;
          ++pi;
        }
      }
      // ---- last pair  ||  diagonal operands of the next pass
      if (pass + 1 < n_passes) {
        const bool boundary = (left == 1);
        if (boundary) next_stage_ready();
        const double* dn = boundary ? nxt_buf : up + pair_unit;
        gen_diag_slow(g, dn + MT * 32, q);
        gen_diag_fast(g, dn + MT * 32, q, vn);
        mma_pair<MT>(acc_re, acc_im, up, lane, v);
        v = vn;
        if (boundary) retire_stage(); else --left;
        up = dn;
      } else {
        mma_pair<MT>(acc_re, acc_im, up, lane, v);
      }
    }
  } else {
    // d == 1 (no pair units): flat walk over the units; unit k is a diagonal unit iff
    // k % n_units == 0.
    int stage = 0;
    int left_in_stage = n_stages > 0 ? stage_units(0) : 0;
    const double* up = cur_buf;
    int u = 0;  // unit index within the pass
    Vals v = {0.0, 0.0, 0.0, 0.0};
    if (total_units > 0) gen_diag(g, up + MT * 32, q, v);

    for (int k = 0; k < total_units; ++k) {
      const bool cur_diag = (u == 0);
      const bool last_in_stage = (left_in_stage == 1);
      const bool has_next = (k + 1 < total_units);
      const double* up_next = up + (cur_diag ? p.diag_unit : p.pair_unit);
      if (last_in_stage && has_next) {
        cp_async_wait<0>();  // the only outstanding group is stage + 1
        __syncthreads();
        up_next = nxt_buf;
      }
      const int u_next = (u + 1 == n_units) ? 0 : u + 1;
      Vals vn = v;
      // Six straight-line variants (current unit type x next unit type): the generator of the next
      // unit and the DMMAs of the current one share a basic block so that ptxas interleaves them.
      if (!has_next) {
        if (cur_diag) mma_diag<MT>(acc_re, acc_im, up, lane, v);
        else mma_pair<MT>(acc_re, acc_im, up, lane, v);
      } else if (u_next == 0) {
        const double* cn = up_next + MT * 32;
        gen_diag_slow(g, cn, q);
        if (cur_diag) {
          gen_diag_fast(g, cn, q, vn);
          mma_diag<MT>(acc_re, acc_im, up, lane, v);
        } else {
          gen_diag_fast(g, cn, q, vn);
          mma_pair<MT>(acc_re, acc_im, up, lane, v);
        }
      } else {
        const double* cn = up_next + 2 * MT * 32;
        bool fix;
        if (cur_diag) {
          fix = gen_pair(g, cn, q, vn);
          mma_diag<MT>(acc_re, acc_im, up, lane, v);
        } else {
          fix = gen_pair(g, cn, q, vn);
          mma_pair<MT>(acc_re, acc_im, up, lane, v);
        }
        if (__any_sync(0xffffffffu, fix)) {
          if (fix) {
            const Vals4 r = fix_pair(g.w, g.dt, g.ph_re, g.ph_im, cn[q]);
            vn.a_re = r.a_re;
            vn.a_im = r.a_im;
            vn.b_re = r.b_re;
            vn.b_im = r.b_im;
          }
        }
      }
      v = vn;
      if (last_in_stage && has_next) {
        __syncthreads();  // everyone is done reading cur_buf
        if (stage + 2 < n_stages) {
          stage_load(stage + 2, cur_buf);
          cp_async_commit();
        }
        double* tmp = cur_buf;
        cur_buf = nxt_buf;
        nxt_buf = tmp;
        ++stage;
        left_in_stage = stage_units(stage);
      } else {
        --left_in_stage;
      }
      up = up_next;
      u = u_next;
    }
  }

  // ---- epilogue: C fragment (row = lane/4, cols 2q, 2q+1) -> partial[z][row][w]
  const int w0 = (blockIdx.x * NW + warp) * 8 + 2 * q;
  double* out = p.partial + (size_t)blockIdx.z * p.rows_pad * p.n_omega * 2;
#pragma unroll
  for (int mt = 0; mt < MT; ++mt) {
    const int row = (rb * MT + mt) * 8 + (lane >> 2);
    double* dst = out + ((size_t)row * p.n_omega + w0) * 2;
    if (w0 < p.n_omega) {
      reinterpret_cast<double2*>(dst)[0] = make_double2(acc_re[mt][0], acc_im[mt][0]);
    }
    if (w0 + 1 < p.n_omega) {
      reinterpret_cast<double2*>(dst)[1] = make_double2(acc_re[mt][1], acc_im[mt][1]);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Statically scheduled variant of ctrlmat_main_kernel for the shapes that dominate config 3 and the
// north_star target (d = 4: NP = 6 level pairs, one pass per stage or a pass split into two pieces):
// the walk over the 1 + NP units of a pass is fully unrolled, so the stage boundaries, the unit sizes
// and the unit kinds are compile-time facts.  In the generic kernel that bookkeeping (run lengths,
// boundary tests, pointer arithmetic, the v = vn copies) costs ~1.3 issue slots per DMMA, and under the
// dispatch-port model (an FP64-pipe instruction blocks the scheduler's dispatch for its pipe time, see
// DESIGN.md 4.1) every one of them is a cycle the tensor pipe idles.
// Requires pps == 1 and n_sp == NSP with the generic piece boundaries piece_begin(j, 1 + NP, NSP).
// ------------------------------------------------------------------------------------------------
// the pair units of the first TP row tiles only (SPLIT variant below)
template <int MT, int TP>
__device__ __forceinline__ void mma_pair_tiles(double (&acc_re)[MT][2], double (&acc_im)[MT][2],
                                               const double* unit, int lane, const Vals& v) {
#pragma unroll
  for (int mt = 0; mt < TP; ++mt) {
    const double a = unit[mt * 32 + lane];
    dmma884(acc_re[mt][0], acc_re[mt][1], a, v.a_re);
    dmma884(acc_im[mt][0], acc_im[mt][1], a, v.a_im);
  }
#pragma unroll
  for (int mt = 0; mt < TP; ++mt) {
    const double a = unit[(MT + mt) * 32 + lane];
    dmma884(acc_re[mt][0], acc_re[mt][1], a, v.b_re);
    dmma884(acc_im[mt][0], acc_im[mt][1], a, v.b_im);
  }
}

// SPLIT (two qubits, six noise operators: 96 rows): basis element 0 of the Pauli / GGM basis is the identity,
// Cbar_0 = 1/2 is diagonal in every eigenbasis, so the six rows (j, 0) have no level-pair terms.  With the rows
// ordered [90 rows (j, k >= 1) | 6 rows (j, 0)] the twelfth row tile holds two pair rows and the six identity
// rows: its 24 pair DMMAs per pass are dropped and the two pair rows go through 48 DFMAs per lane instead (a
// lane owns (frequency, segment) = one B-fragment element, i.e. exactly the factor those rows need), added
// into the tile's accumulators by shuffles at the end.  Measured on d4: 16.55 -> 15.9 ms.
template <int MT, int NW, int NP, int NSP, bool SPLIT = false>
__global__ void __launch_bounds__(NW * 32, (MT <= 2 ? 3 : MT >= 10 ? 3 : 1))
ctrlmat_static_kernel(const MainParams p) {
  extern __shared__ __align__(16) double smem[];
  if (p.n_live && (int)blockIdx.x * NW * 8 >= __ldg(p.n_live)) return;  // whole CTA past the used slots
  constexpr int NU = 1 + NP;
  constexpr int DIAG_UNIT = MT * 32 + 8, PAIR_UNIT = 2 * MT * 32 + 12;
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int q = lane & 3;
  const int rb = blockIdx.y;
  const int pass_begin = blockIdx.z * p.passes_per_chunk;
  const int pass_end = min(p.n_pass, pass_begin + p.passes_per_chunk);
  const int n_passes = pass_end - pass_begin;

  Gen g;
  {
    const int w_idx = (blockIdx.x * NW + warp) * 8 + (lane >> 2);
    g.w = w_idx < p.n_omega ? p.omega[w_idx] : 1.0;
    g.w_zero = fabs(g.w) < TINY_OMEGA;
    g.inv_w = g.w_zero ? 0.0 : 1.0 / g.w;
    g.dt_prev = -1.0;
    g.dt = 0.0;
    g.hc = SQRT2;
    g.hs = 0.0;
    g.j0_re = g.j0_im = 0.0;
    g.ph_re = 1.0;
    g.ph_im = 0.0;
  }
  double acc_re[MT][2], acc_im[MT][2];
#pragma unroll
  for (int mt = 0; mt < MT; ++mt) {
    acc_re[mt][0] = acc_re[mt][1] = 0.0;
    acc_im[mt][0] = acc_im[mt][1] = 0.0;
  }
  double side_re[2] = {0.0, 0.0}, side_im[2] = {0.0, 0.0};   // SPLIT: pair terms of rows 0, 1 of the last tile

  // stage i = (pass i / NSP, piece i % NSP); piece j holds units [PB(j), PB(j + 1))
  auto PB = [](int j) constexpr { return (j * NU) / NSP; };
  auto UOFF = [](int u) constexpr { return u == 0 ? 0 : DIAG_UNIT + (u - 1) * PAIR_UNIT; };
  const double* gstream = p.stream + (size_t)rb * p.rb_doubles + (size_t)pass_begin * p.pass_doubles;
  const int n_stages = n_passes * NSP;
  // stage i lives in buffer i & 1; its mbarrier completes phase (i >> 1) & 1 when the bytes have landed
  unsigned long long* mbar = reinterpret_cast<unsigned long long*>(smem + 2 * (size_t)p.stage_doubles);
  auto stage_load = [&](int i) {  // called by thread 0 only
    const int pass = i / NSP, piece = i % NSP;
    const int o0 = UOFF(PB(piece));
    const int o1 = piece + 1 == NSP ? (int)p.pass_doubles : UOFF(PB(piece + 1));
    const unsigned bytes = (unsigned)(o1 - o0) * 8u;
    mbar_expect_tx(&mbar[i & 1], bytes);
    bulk_g2s(smem + (size_t)(i & 1) * p.stage_doubles, gstream + (size_t)pass * p.pass_doubles + o0, bytes,
             &mbar[i & 1]);
  };
  if (threadIdx.x == 0) {
    mbar_init(&mbar[0], 1);
    mbar_init(&mbar[1], 1);
    mbar_fence_init();
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    if (n_stages > 0) stage_load(0);
    if (n_stages > 1) stage_load(1);
  }
  if (n_stages > 0) mbar_wait(&mbar[0], 0);
  int stage = 0;
  Vals v = {0.0, 0.0, 0.0, 0.0};
  const double* up = smem;
  if (n_passes > 0) gen_diag(g, up + MT * 32, q, v);
  for (int pass = 0; pass < n_passes; ++pass) {
#pragma unroll
    for (int u = 0; u < NU; ++u) {
      // compile-time facts about unit u
      int piece = 0;
#pragma unroll
      for (int j = 1; j < NSP; ++j) piece += (u >= PB(j)) ? 1 : 0;
      const bool last_in_piece = (u + 1 == (piece + 1 == NSP ? NU : PB(piece + 1)));
      const bool last_of_pass = (u + 1 == NU);
      const bool has_next = !(last_of_pass && pass + 1 == n_passes);
      Vals vn = v;
      const double* pn = up + (u == 0 ? DIAG_UNIT : PAIR_UNIT);
      if (last_in_piece) {
        if (has_next) mbar_wait(&mbar[(stage + 1) & 1], ((stage + 1) >> 1) & 1);  // stage + 1 has landed
        pn = smem + (size_t)((stage + 1) & 1) * p.stage_doubles;
      }
      bool fix = false;
      if (!last_of_pass) {
        fix = gen_pair(g, pn + 2 * MT * 32, q, vn);
      } else if (has_next) {
        gen_diag_slow(g, pn + MT * 32, q);
        gen_diag_fast(g, pn + MT * 32, q, vn);
      }
      if (u == 0) {
        mma_diag<MT>(acc_re, acc_im, up, lane, v);
      } else if (SPLIT) {
        mma_pair_tiles<MT, MT - 1>(acc_re, acc_im, up, lane, v);
#pragma unroll
        for (int r = 0; r < 2; ++r) {   // this lane's (frequency, segment) term of rows r of the last tile
          const double a = up[(MT - 1) * 32 + r * 4 + q], b = up[(2 * MT - 1) * 32 + r * 4 + q];
          side_re[r] = fma(a, v.a_re, fma(b, v.b_re, side_re[r]));
          side_im[r] = fma(a, v.a_im, fma(b, v.b_im, side_im[r]));
        }
      } else {
        mma_pair<MT>(acc_re, acc_im, up, lane, v);
      }
      if (!last_of_pass) {
        if (__any_sync(0xffffffffu, fix)) {
          if (fix) {
            const Vals4 r = fix_pair(g.w, g.dt, g.ph_re, g.ph_im, pn[2 * MT * 32 + q]);
            vn.a_re = r.a_re;
            vn.a_im = r.a_im;
            vn.b_re = r.b_re;
            vn.b_im = r.b_im;
          }
        }
      }
      v = vn;
      if (last_in_piece && has_next) {
        __syncthreads();  // everyone is done reading the buffer of `stage`
        if (threadIdx.x == 0 && stage + 2 < n_stages) {
          fence_proxy_async();  // order the generic-proxy reads before the async overwrite
          stage_load(stage + 2);
        }
        ++stage;
      }
      up = pn;
    }
  }

  if (SPLIT) {
    // sum over the 4 segments of a pass slot (lanes 4 w .. 4 w + 3 hold frequency w), then hand the totals to
    // the lanes that own (row r, frequencies 2 q, 2 q + 1) of the last tile's accumulator fragment
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      side_re[r] += __shfl_xor_sync(0xffffffffu, side_re[r], 1);
      side_im[r] += __shfl_xor_sync(0xffffffffu, side_im[r], 1);
      side_re[r] += __shfl_xor_sync(0xffffffffu, side_re[r], 2);
      side_im[r] += __shfl_xor_sync(0xffffffffu, side_im[r], 2);
    }
    const int r_own = lane >> 2;
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int src = 4 * (2 * q + e);
      const double re0 = __shfl_sync(0xffffffffu, side_re[0], src), im0 = __shfl_sync(0xffffffffu, side_im[0], src);
      const double re1 = __shfl_sync(0xffffffffu, side_re[1], src), im1 = __shfl_sync(0xffffffffu, side_im[1], src);
      if (r_own == 0) {
        acc_re[MT - 1][e] += re0;
        acc_im[MT - 1][e] += im0;
      } else if (r_own == 1) {
        acc_re[MT - 1][e] += re1;
        acc_im[MT - 1][e] += im1;
      }
    }
  }
  const int w0 = (blockIdx.x * NW + warp) * 8 + 2 * q;
  double* out = p.partial + (size_t)blockIdx.z * p.rows_pad * p.n_omega * 2;
#pragma unroll
  for (int mt = 0; mt < MT; ++mt) {
    const int row = (rb * MT + mt) * 8 + (lane >> 2);
    double* dst = out + ((size_t)row * p.n_omega + w0) * 2;
    if (w0 < p.n_omega) reinterpret_cast<double2*>(dst)[0] = make_double2(acc_re[mt][0], acc_im[mt][0]);
    if (w0 + 1 < p.n_omega) reinterpret_cast<double2*>(dst)[1] = make_double2(acc_re[mt][1], acc_im[mt][1]);
  }
}

// ------------------------------------------------------------------------------------------------
// Small row counts (rows = n_nops * n_basis <= 16: a single qubit in the Pauli basis, config 2): DFMA
// variant.  With 12 rows the tensor path pads M to 16 (25 % of the DMMA work is wasted) and the mix of
// DMMA and the generator's DFMA/DMUL stream costs another ~12 % of the FP64 pipe (measured,
// profiles/fp64_peaks_r01.jsonl "mixed").  Here a THREAD owns one frequency and walks the segments; the
// coefficients of a segment are broadcast from shared memory (every lane reads the same address) and
// the 2 R accumulators live in registers: per (segment, frequency) R (2 + 4 n_pairs) DFMAs with no
// padding beyond R = 4 ceil(rows / 4), next to the same operand generator.  A warp = 32 frequencies x
// one contiguous range of segments; the 8 warps of a CTA split the CTA's segment chunk 8 ways (their
// partial sums are reduced through shared memory in a fixed order), each warp streams its own records
// through a private double-buffered cp.async pipeline -- no block-wide barrier in the main loop.
//
// Stream: one record per segment:  t, dt, diag[R], then per level pair: Omega, cos(Omega dt/2),
// sin(Omega dt/2), 0, Re[RFP], Im[RFP]  (RFP = RF rounded up to even).
//
// Rows without level-pair terms.  If basis element 0 is a multiple of the identity (Basis.pauli,
// Basis.ggm), Cbar_0 = U^+ C_0 U = C_0 is diagonal in every eigenbasis: its rows (j, 0) only have the
// diagonal term (and vanish altogether for traceless noise operators).  The accumulator slots are
// therefore ordered [RF rows (j, k >= 1) | rows (j, 0) | padding]: the diagonal coefficients cover
// all R slots, the pair coefficients only the first RF -- for config 2 (3 x 4 rows) 9 instead of 12
// rows take part in the 4 n_pairs DFMAs per row: 60 instead of 72 DFMAs per (segment, frequency).
// ------------------------------------------------------------------------------------------------
struct DfmaParams {
  const double* stream;
  const double* omega;
  double* partial;   // [S][R][n_omega] complex
  int n_omega;
  int G;
  int n_pairs;
  int rec_doubles;
  int segs_per_cta;  // segment chunk of one CTA (blockIdx.y)
  int segs_per_warp; // ceil(segs_per_cta / DFMA_WARPS)
  const double2* trig_table;  // (sin, cos)(k pi / 128), 256 entries
  int stage_smem_doubles;     // offset of the table copy in shared memory
};

constexpr int DFMA_WARPS = 8;
constexpr int DFMA_STAGE_SEGS = 8;

__host__ __device__ inline int dfma_rec_doubles(int R, int RF, int n_pairs) {
  return 2 + R + n_pairs * (4 + 2 * ((RF + 1) & ~1));
}
// accumulator slot -> row (j * n_krows + k) of the control matrix, -1 for padding.  split: slots
// [0, RF) are the rows with k >= 1, slots RF.. the rows with k == 0 (basis element 0 = identity)
__host__ __device__ inline int dfma_row_of_slot(int slot, int rows, int RF, bool split, int n_jrows,
                                                int n_krows) {
  if (!split) return slot < rows ? slot : -1;
  if (slot < RF) return (slot / (n_krows - 1)) * n_krows + 1 + slot % (n_krows - 1);
  return slot - RF < n_jrows ? (slot - RF) * n_krows : -1;
}

// element `off` of the record of a segment; Bseg / Cseg = the segment's transformed noise operators
// [n_jrows][d*d] and basis elements [n_krows][d*d] (complex, interleaved), ev = its eigenvalues
__device__ __forceinline__ double dfma_record_value(int off, int d, int rows, int R, int RF, bool split,
                                                    int n_jrows, int n_krows, const double* Bseg,
                                                    const double* Cseg, const double* ev, double tg,
                                                    double dtg) {
  const int dd = d * d;
  const int RFP = (RF + 1) & ~1;
  if (off < 2) return off == 0 ? tg : dtg;
  if (off < 2 + R) {
    const int row = dfma_row_of_slot(off - 2, rows, RF, split, n_jrows, n_krows);
    if (row < 0) return 0.0;
    const double* Bm = Bseg + (size_t)(row / n_krows) * 2 * dd;
    const double* Cm = Cseg + (size_t)(row % n_krows) * 2 * dd;
    double acc = 0.0;
    for (int m = 0; m < d; ++m) acc += Bm[2 * (m * d + m)] * Cm[2 * (m * d + m)];
    return acc;
  }
  off -= 2 + R;
  const int pair = off / (4 + 2 * RFP);
  off %= 4 + 2 * RFP;
  int m, n;
  pair_from_index(pair, d, m, n);
  if (off < 4) {
    const double Om = ev[m] - ev[n];
    if (off == 0) return Om;
    if (off == 3) return 0.0;
    double sn, cs;
    sincos(0.5 * (Om * dtg), &sn, &cs);
    return off == 1 ? cs : sn;
  }
  const int col = (off - 4) / RFP, slot = (off - 4) % RFP;
  const int row = slot < RF ? dfma_row_of_slot(slot, rows, RF, split, n_jrows, n_krows) : -1;
  if (row < 0) return 0.0;
  const double* Bm = Bseg + (size_t)(row / n_krows) * 2 * dd;
  const double* Cm = Cseg + (size_t)(row % n_krows) * 2 * dd;
  const cplx b = {Bm[2 * (m * d + n)], Bm[2 * (m * d + n) + 1]};
  const cplx c = {Cm[2 * (n * d + m)], Cm[2 * (n * d + m) + 1]};
  const cplx prod = cmul(b, c);
  return col == 0 ? prod.re : prod.im;
}

__global__ void __launch_bounds__(256)
assemble_dfma_kernel(int G, int d, int rows, int R, int RF, int split, int n_jrows, int n_krows,
                     const double* __restrict__ Bbar, const double* __restrict__ Cbar,
                     const double* __restrict__ eigvals, const double* __restrict__ dt,
                     const double* __restrict__ t, double* __restrict__ stream) {
  const int rec = dfma_rec_doubles(R, RF, d * (d - 1) / 2);
  const size_t total = (size_t)G * rec;
  const int dd = d * d;
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (size_t)gridDim.x * blockDim.x) {
    const int g = (int)(idx / rec);
    stream[idx] = dfma_record_value((int)(idx % rec), d, rows, R, RF, split != 0, n_jrows, n_krows,
                                    Bbar + (size_t)g * n_jrows * 2 * dd,
                                    Cbar + (size_t)g * n_krows * 2 * dd, eigvals + (size_t)g * d, t[g],
                                    dt[g]);
  }
}

// Fused prologue of the DFMA path (d <= 3): a block transforms the operators of DFMA_PRO_SEGS segments
// into shared memory (thread per (segment, operator), registers) and writes their records, which are
// contiguous in the stream -- one launch instead of two, and Bbar / Cbar never touch HBM
// (transform_small_kernel 5.6 us + assemble_dfma_kernel 10.9 us for config 2).
constexpr int DFMA_PRO_SEGS = 16;
template <int D>
__global__ void __launch_bounds__(128)
dfma_prologue_kernel(int G, int n_nops, int n_basis, int parts_j, int parts_k, int rows, int R, int RF,
                     int split, const double2* __restrict__ eigvecs,
                     const double2* __restrict__ propagators, const double2* __restrict__ n_opers,
                     const double* __restrict__ n_coeffs, const double2* __restrict__ basis,
                     const double* __restrict__ eigvals, const double* __restrict__ dt,
                     const double* __restrict__ t, double* __restrict__ stream) {
  extern __shared__ __align__(16) double2 xs[];  // [DFMA_PRO_SEGS][n_jrows + n_krows][D*D]
  constexpr int DD = D * D;
  const int n_ops = n_nops + n_basis;
  const int n_jrows = n_nops * parts_j, n_krows = n_basis * parts_k;
  const int per_seg = (n_jrows + n_krows) * DD;
  const int seg0 = blockIdx.x * DFMA_PRO_SEGS;
  const int n_seg = min(DFMA_PRO_SEGS, G - seg0);
  for (int idx = threadIdx.x; idx < n_seg * n_ops; idx += blockDim.x) {
    const int sl = idx / n_ops, op = idx % n_ops;
    const bool is_noise = op < n_nops;
    double2* dst = xs + (size_t)sl * per_seg +
                   (is_noise ? op * parts_j : n_jrows + (op - n_nops) * parts_k) * DD;
    transform_small_one<D>(G, seg0 + sl, op, n_nops, is_noise ? parts_j : parts_k, eigvecs, propagators,
                           n_opers, n_coeffs, basis, dst);
  }
  __syncthreads();
  const int rec = dfma_rec_doubles(R, RF, D * (D - 1) / 2);
  double* out = stream + (size_t)seg0 * rec;
  for (int e = threadIdx.x; e < n_seg * rec; e += blockDim.x) {
    const int sl = e / rec, g = seg0 + sl;
    const double* Bseg = reinterpret_cast<const double*>(xs + (size_t)sl * per_seg);
    out[e] = dfma_record_value(e % rec, D, rows, R, RF, split != 0, n_jrows, n_krows, Bseg,
                               Bseg + (size_t)n_jrows * 2 * DD, eigvals + (size_t)g * D, t[g], dt[g]);
  }
}

// The table-sincos constants enter through the KERNEL PARAMETERS: constant bank 0 can be a direct
// operand of DFMA/DMUL, whereas a __constant__ array (bank 3) is re-loaded by LDC/LDCU in every
// iteration (ncu r01c: 33 M of the 676 M warp instructions of config 2) -- and on sm_100 every
// non-FP64 instruction costs the issue slot of half a DFMA.
struct TrigConsts {
  double inv_step, magic, step_hi, step_lo, s5, s3, c6, c4;
};
inline TrigConsts trig_consts() {
  return {4.07436654315252084757e+01, 6755399441055744.0, 2.45436926061702587187e-02,
          9.56755311833869693105e-19, 1.0 / 120.0, -1.0 / 6.0, -1.0 / 720.0, 1.0 / 24.0};
}
__device__ __forceinline__ void sincos_tab_p(double x, const double2* __restrict__ table_smem,
                                             const TrigConsts& tc, double& sn, double& cs) {
  double kd = fma(x, tc.inv_step, tc.magic);
  const int k = __double2loint(kd) & (TRIG_TABLE_SIZE - 1);
  kd -= tc.magic;
  double r = fma(-kd, tc.step_hi, x);
  r = fma(-kd, tc.step_lo, r);
  const double2 sc = table_smem[k];
  const double r2 = r * r;
  const double ps = fma(r2, tc.s5, tc.s3);
  const double s = fma(r * r2, ps, r);
  double pc = fma(r2, tc.c6, tc.c4);
  pc = fma(pc, r2, -0.5);
  const double c = fma(pc, r2, 1.0);
  sn = fma(sc.x, c, sc.y * s);
  cs = fma(sc.y, c, -(sc.x * s));
}

// NP = number of level pairs d (d - 1) / 2 (compile time: record size and the walk over a record are
// constants, the pair loop is unrolled); RF <= R = number of leading accumulator slots that carry pair
// coefficients (see "rows without level-pair terms" above).
template <int R, int RF, int NP>
__global__ void __launch_bounds__(DFMA_WARPS * 32, 2)
ctrlmat_dfma_kernel(const DfmaParams p, const TrigConsts tc) {
  extern __shared__ __align__(16) double smem[];
  constexpr int RFP = (RF + 1) & ~1;
  constexpr int PAIR = 4 + 2 * RFP;
  constexpr int REC = 2 + R + NP * PAIR;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int w_idx = blockIdx.x * 32 + lane;
  double* wbuf = smem + (size_t)warp * 2 * DFMA_STAGE_SEGS * REC;  // this warp's two stage buffers
  double2* trig = reinterpret_cast<double2*>(smem + p.stage_smem_doubles);
  for (int k = threadIdx.x; k < TRIG_TABLE_SIZE; k += DFMA_WARPS * 32) trig[k] = p.trig_table[k];
  __syncthreads();

  Gen g;
  g.w = w_idx < p.n_omega ? p.omega[w_idx] : 1.0;
  g.w_zero = fabs(g.w) < TINY_OMEGA;
  g.inv_w = g.w_zero ? 0.0 : 1.0 / g.w;
  g.dt_prev = -1.0;
  g.dt = 0.0;
  g.hc = SQRT2;
  g.hs = 0.0;
  g.j0_re = g.j0_im = 0.0;
  g.ph_re = 1.0;
  g.ph_im = 0.0;

  double acc_re[R], acc_im[R];
#pragma unroll
  for (int r = 0; r < R; ++r) acc_re[r] = acc_im[r] = 0.0;

  const int seg_begin = min(p.G, blockIdx.y * p.segs_per_cta + warp * p.segs_per_warp);
  const int seg_end = min(min(p.G, (blockIdx.y + 1) * p.segs_per_cta), seg_begin + p.segs_per_warp);
  const int n_segs = max(0, seg_end - seg_begin);
  const int n_stages = (n_segs + DFMA_STAGE_SEGS - 1) / DFMA_STAGE_SEGS;
  const double* gsrc = p.stream + (size_t)seg_begin * REC;
  auto stage_load = [&](int st) {
    const int s0 = st * DFMA_STAGE_SEGS;
    const int len = min(DFMA_STAGE_SEGS, n_segs - s0) * REC;  // REC is even: whole 16-byte chunks
    double* dst = wbuf + (st & 1) * DFMA_STAGE_SEGS * REC;
    const double* src = gsrc + (size_t)s0 * REC;
    for (int e = lane * 2; e < len; e += 64) cp_async16(dst + e, src + e);
  };
  auto dt_update = [&](double dtg) {
    g.dt = dtg;
    if (__double_as_longlong(g.dt) != __double_as_longlong(g.dt_prev)) {  // warp-uniform
      double sn, cs;
      sincos_cw(0.5 * (g.w * g.dt), sn, cs);
      g.hc = SQRT2 * cs;
      g.hs = SQRT2 * sn;
      const double f = g.hs * g.inv_w;
      g.j0_re = g.w_zero ? g.dt : g.hc * f;
      g.j0_im = g.w_zero ? 0.0 : g.hs * f;
      g.dt_prev = g.dt;
    }
  };
  auto fma_diag = [&](const double* rp, double a_re, double a_im) {
    const double2* c2 = reinterpret_cast<const double2*>(rp + 2);
#pragma unroll
    for (int r = 0; r < R / 2; ++r) {
      const double2 c = c2[r];
      acc_re[2 * r] = fma(c.x, a_re, acc_re[2 * r]);
      acc_im[2 * r] = fma(c.x, a_im, acc_im[2 * r]);
      acc_re[2 * r + 1] = fma(c.y, a_re, acc_re[2 * r + 1]);
      acc_im[2 * r + 1] = fma(c.y, a_im, acc_im[2 * r + 1]);
    }
  };
  auto fma_pair = [&](const double* pp, const Vals& v) {
    const double2* cre = reinterpret_cast<const double2*>(pp + 4);
    const double2* cim = reinterpret_cast<const double2*>(pp + 4 + RFP);
#pragma unroll
    for (int r = 0; r < RF / 2; ++r) {
      const double2 a = cre[r], b = cim[r];
      acc_re[2 * r] = fma(a.x, v.a_re, fma(b.x, v.b_re, acc_re[2 * r]));
      acc_im[2 * r] = fma(a.x, v.a_im, fma(b.x, v.b_im, acc_im[2 * r]));
      acc_re[2 * r + 1] = fma(a.y, v.a_re, fma(b.y, v.b_re, acc_re[2 * r + 1]));
      acc_im[2 * r + 1] = fma(a.y, v.a_im, fma(b.y, v.b_im, acc_im[2 * r + 1]));
    }
    if (RF & 1) {  // odd number of pair rows: the last one alone (LDS.64)
      const double a = pp[4 + RF - 1], b = pp[4 + RFP + RF - 1];
      acc_re[RF - 1] = fma(a, v.a_re, fma(b, v.b_re, acc_re[RF - 1]));
      acc_im[RF - 1] = fma(a, v.a_im, fma(b, v.b_im, acc_im[RF - 1]));
    }
  };
  // one segment; the half-angle factors (hc, hs, j0) are valid for its dt
  auto one_segment = [&](const double* rp) {
    sincos_tab_p(g.w * rp[0], trig, tc, g.ph_im, g.ph_re);
    fma_diag(rp, g.ph_re * g.j0_re - g.ph_im * g.j0_im, g.ph_re * g.j0_im + g.ph_im * g.j0_re);
#pragma unroll
    for (int pi = 0; pi < NP; ++pi) {
      const double* pp = rp + 2 + R + pi * PAIR;
      Vals v;
      const double Om = pp[0];
      const bool fix = pair_values(g, Om, pp[1], pp[2], v);
      if (__any_sync(0xffffffffu, fix)) {  // rare; taken by the whole warp, so it never diverges
        const Vals4 rr = fix_pair(g.w, g.dt, g.ph_re, g.ph_im, Om);
        v.a_re = fix ? rr.a_re : v.a_re;
        v.a_im = fix ? rr.a_im : v.a_im;
        v.b_re = fix ? rr.b_re : v.b_re;
        v.b_im = fix ? rr.b_im : v.b_im;
      }
      fma_pair(pp, v);
    }
  };
  // (Generating the next unit's operands next to the current unit's DFMAs, as the tensor-path kernel
  // does, was measured SLOWER here: 1.33 vs 1.16 ms on config 2 -- the extra live values cost moves.
  // Generating the operands of two segments per iteration changed nothing: 1.073 vs 1.078 ms -- the
  // kernel is bound by issue slots, not by latency.)
  if (n_stages > 0) {
    stage_load(0);
    cp_async_commit();
  }
  for (int st = 0; st < n_stages; ++st) {
    if (st + 1 < n_stages) {
      stage_load(st + 1);
      cp_async_commit();
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncwarp();
    const double* rp = wbuf + (st & 1) * DFMA_STAGE_SEGS * REC;
    const int ns = min(DFMA_STAGE_SEGS, n_segs - st * DFMA_STAGE_SEGS);
    // dt is tested once per stage, not per segment: on a uniform time grid the half-angle factors never
    // change after the first segment
    const double dt_l = rp[(lane < ns ? lane : 0) * REC + 1];
    const bool same_dt =
        __all_sync(0xffffffffu, __double_as_longlong(dt_l) == __double_as_longlong(g.dt_prev));
    if (same_dt) {
      for (int sgm = 0; sgm < ns; ++sgm, rp += REC) one_segment(rp);
    } else {
      for (int sgm = 0; sgm < ns; ++sgm, rp += REC) {
        dt_update(rp[1]);
        one_segment(rp);
      }
    }
    __syncwarp();  // all lanes are done with this buffer before it is refilled
  }

  // ---- reduce the 8 warps' partial sums (fixed order) and write partial[z][row][w]
  __syncthreads();  // every warp is done with its stage buffers: reuse them
  double* red = smem;  // [DFMA_WARPS][2 R][32]
#pragma unroll
  for (int r = 0; r < R; ++r) {
    red[((size_t)warp * 2 * R + 2 * r) * 32 + lane] = acc_re[r];
    red[((size_t)warp * 2 * R + 2 * r + 1) * 32 + lane] = acc_im[r];
  }
  __syncthreads();
  if (w_idx < p.n_omega) {
    double2* out = reinterpret_cast<double2*>(p.partial) + (size_t)blockIdx.y * R * p.n_omega;
    for (int row = warp; row < R; row += DFMA_WARPS) {
      double re = 0.0, im = 0.0;
#pragma unroll
      for (int wi = 0; wi < DFMA_WARPS; ++wi) {
        re += red[((size_t)wi * 2 * R + 2 * row) * 32 + lane];
        im += red[((size_t)wi * 2 * R + 2 * row + 1) * 32 + lane];
      }
      out[(size_t)row * p.n_omega + w_idx] = make_double2(re, im);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// finalize: sum the split-K partials and undo the Hermitian/anti-Hermitian row expansion
//   out[j,k,w] = sum_z sum_{pj,pk} i^{pj+pk} partial[z][(j*parts_j+pj)*n_krows + k*parts_k+pk][w]
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
finalize_kernel(int S, int rows_pad, int n_nops, int n_basis, int parts_j, int parts_k, int n_omega,
                size_t ld_out, int split_rf, const double* __restrict__ partial,
                double* __restrict__ out) {
  const size_t total = (size_t)n_nops * n_basis * n_omega;
  const int n_krows = n_basis * parts_k;
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (size_t)gridDim.x * blockDim.x) {
    const int w = (int)(idx % n_omega);
    const int jk = (int)(idx / n_omega);
    const int j = jk / n_basis, k = jk % n_basis;
    double re = 0.0, im = 0.0;
    for (int pj = 0; pj < parts_j; ++pj) {
      for (int pk = 0; pk < parts_k; ++pk) {
        int row = (j * parts_j + pj) * n_krows + k * parts_k + pk;
        // DFMA kernel with the identity rows split off (parts_j = parts_k = 1): slot of row (j, k)
        if (split_rf > 0) row = k == 0 ? split_rf + j : j * (n_basis - 1) + k - 1;
        double pr = 0.0, pi = 0.0;
        for (int z = 0; z < S; ++z) {
          const double2 v = reinterpret_cast<const double2*>(
              partial)[((size_t)z * rows_pad + row) * n_omega + w];
          pr += v.x;
          pi += v.y;
        }
        switch ((pj + pk) & 3) {  // multiply by i^(pj+pk)
          case 0: re += pr; im += pi; break;
          case 1: re -= pi; im += pr; break;
          default: re -= pr; im -= pi; break;
        }
      }
    }
    reinterpret_cast<double2*>(out)[(size_t)jk * ld_out + w] = make_double2(re, im);
  }
}

// ------------------------------------------------------------------------------------------------
// banded route: Chebyshev interpolation of per-chunk partial sums on dense frequency bands (DESIGN 4.1.1)
//
// With the segments cut into chunks c of at most T_c and the stream's times taken relative to the chunk
// centres t_c (assemble_kernel, chunk_segs > 0), the main kernel's partial sum of chunk c is
//     Z_c(w) = e^{-i w t_c} B^(c)(w) = int_{|s| <= T_c/2} e^{i w s} f(t_c + s) ds,
// an entire function of exponential type T_c / 2.  On a band [k W, (k + 1) W) of width W = 4 sigma / T_c its
// Chebyshev coefficients beyond degree p are bounded by 2 |J_p(sigma)| ||f||_1, so the values at the
// BAND_P Chebyshev points of the second kind determine Z_c on the band to rounding level (BAND_P = 48,
// sigma = 16: max_{p >= 48} |J_p(16)| = 4.8e-19).  A band whose targets outnumber its proxies by the rule
// in band_plan_kernel is evaluated as
//     B(w) = sum_c e^{i w t_c} sum_p l_p(w) Z_c(w_p),
// every other frequency directly, B(w) = sum_c e^{i w t_c} Z_c(w).
// ------------------------------------------------------------------------------------------------
constexpr int BAND_P = 48;
constexpr double BAND_SIGMA = 16.0;
constexpr int BAND_MIN_G = 1024;       // shorter pulses: too few segments per chunk for the route to pay
constexpr int BAND_CHUNK_QUANTUM = 128;  // chunk length: a multiple of this many segments
constexpr int BAND_PLAN_THREADS = 1024;
constexpr int BAND_EVAL_OUTS = 8;      // (j, k) outputs per thread of band_eval_kernel

struct BandPlan {
  double* eval_omega;  // [n] frequencies the main kernel evaluates: proxies and direct targets, then 1.0
  int* target;         // [n] slot of a direct target, -(run + 1) of an interpolated one
  int* run_start;      // [n + 1] first target of each run of targets in one band
  int* run_base;       // [n] first slot of a run (its proxies if it pays, else its direct targets)
  int* counts;         // [3] used slots, interpolated bands, proxies
  int* log_counts;     // [2] bands and proxies for the dispatch record
};

__device__ __forceinline__ double band_of(double w, double W) { return floor(w / W); }
__device__ __forceinline__ bool band_pays(int len, double r_cost) { return len * (1.0 - r_cost) > BAND_P; }

// exclusive prefix sum over the block (blockDim.x == BAND_PLAN_THREADS); *total = sum over the block
__device__ int block_exclusive_scan(int v, int* total) {
  __shared__ int warp_sums[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int u = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += u;
  }
  if (lane == 31) warp_sums[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    int s = warp_sums[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int u = __shfl_up_sync(0xffffffffu, s, o);
      if (lane >= o) s += u;
    }
    warp_sums[lane] = s;
  }
  __syncthreads();
  const int before = (warp ? warp_sums[warp - 1] : 0) + incl - v;
  *total = warp_sums[31];
  __syncthreads();
  return before;
}

// One CTA: splits the frequency block into runs of consecutive targets that share a band of the global
// lattice [k W, (k + 1) W), decides per run whether interpolation pays, and writes the compacted list of
// frequencies the main kernel evaluates.  Enqueue-only: omega, t and dt stay on the device.
// r_cost = evaluation cost of an interpolated target in units of a direct one; a run of len targets pays
// when len (1 - r_cost) > BAND_P.
__global__ void __launch_bounds__(BAND_PLAN_THREADS)
band_plan_kernel(const double* __restrict__ omega, int n, const double* __restrict__ t,
                 const double* __restrict__ dt, int G, int L, int S, double r_cost, BandPlan plan) {
  __shared__ double tc_max[32];
  __shared__ double s_W;
  const int tid = threadIdx.x;
  // ---- longest chunk -> band width
  double dur = 0.0;
  for (int c = tid; c < S; c += blockDim.x) {
    const int g0 = c * L, g1 = min(G, g0 + L) - 1;
    dur = fmax(dur, (t[g1] + dt[g1]) - t[g0]);
  }
  for (int o = 16; o; o >>= 1) dur = fmax(dur, __shfl_xor_sync(0xffffffffu, dur, o));
  if ((tid & 31) == 0) tc_max[tid >> 5] = dur;
  __syncthreads();
  if (tid == 0) {
    double m = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) m = fmax(m, tc_max[w]);
    s_W = 4.0 * BAND_SIGMA / m;
  }
  __syncthreads();
  const double W = s_W;
  // ---- runs: target i starts a run when its band differs from that of target i - 1
  int n_runs = 0;
  for (int i0 = 0; i0 < n; i0 += blockDim.x) {
    const int i = i0 + tid;
    int flag = 0;
    if (i < n) flag = (i == 0 || band_of(omega[i], W) != band_of(omega[i - 1], W)) ? 1 : 0;
    int tile_runs;
    const int before = block_exclusive_scan(flag, &tile_runs);
    if (i < n) {
      const int run = n_runs + before + flag - 1;
      plan.target[i] = run;  // run index for now
      if (flag) plan.run_start[run] = i;
    }
    n_runs += tile_runs;
  }
  if (tid == 0) plan.run_start[n_runs] = n;
  __syncthreads();
  // ---- slots per run: BAND_P proxies if it pays, else its targets
  int n_slots = 0, n_bands = 0;
  for (int r0 = 0; r0 < n_runs; r0 += blockDim.x) {
    const int r = r0 + tid;
    int slots = 0, pays = 0;
    if (r < n_runs) {
      const int len = plan.run_start[r + 1] - plan.run_start[r];
      pays = band_pays(len, r_cost) ? 1 : 0;
      slots = pays ? BAND_P : len;
    }
    int tile_slots, tile_bands;
    const int base = block_exclusive_scan(slots, &tile_slots);
    block_exclusive_scan(pays, &tile_bands);
    if (r < n_runs) plan.run_base[r] = n_slots + base;
    n_slots += tile_slots;
    n_bands += tile_bands;
  }
  __syncthreads();
  // ---- targets and proxies
  for (int i = tid; i < n; i += blockDim.x) {
    const int r = plan.target[i];
    const int s0 = plan.run_start[r];
    if (band_pays(plan.run_start[r + 1] - s0, r_cost)) {
      plan.target[i] = -(r + 1);
      if (i - s0 < BAND_P) {  // proxy i - s0 of the run (a paying run has more than BAND_P targets)
        const int j = i - s0;
        const double h = 0.5 * W, c = (band_of(omega[s0], W) + 0.5) * W;
        plan.eval_omega[plan.run_base[r] + j] = fma(h, cospi((double)j / (BAND_P - 1)), c);
      }
    } else {
      const int slot = plan.run_base[r] + (i - s0);
      plan.target[i] = slot;
      plan.eval_omega[slot] = omega[i];
    }
  }
  for (int i = n_slots + tid; i < n; i += blockDim.x) plan.eval_omega[i] = 1.0;
  if (tid == 0) {
    plan.counts[0] = n_slots;
    plan.counts[1] = n_bands;
    plan.counts[2] = n_bands * BAND_P;
    plan.log_counts[0] = n_bands;
    plan.log_counts[1] = n_bands * BAND_P;
  }
}

// Replaces finalize_kernel on the banded route.  Thread = one target x BAND_EVAL_OUTS outputs (j, k):
//   out[j, k, w] = sum_c e^{i w t_c} sum_{pj, pk} i^{pj + pk} Zhat_c[row(j, k, pj, pk)](w)
// with Zhat_c(w) = partial_c(slot of w) for a direct target and sum_p l_p(w) partial_c(proxy p) for an
// interpolated one (barycentric weights of the second kind, real; a target on a proxy takes its value).
// Fixed summation order, no atomics: a second call repeats every bit.
__global__ void __launch_bounds__(128)
band_eval_kernel(int n, int S, int L, int G, int rows_pad, int n_nops, int n_basis, int parts_j,
                 int parts_k, size_t ld_out, int split_rf, const double* __restrict__ omega,
                 const double* __restrict__ t, const double* __restrict__ dt, BandPlan plan,
                 const double* __restrict__ partial, double* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int n_out = n_nops * n_basis;
  const int jk0 = blockIdx.y * BAND_EVAL_OUTS;
  const int n_krows = n_basis * parts_k;
  const size_t n_slots = (size_t)n;
  const double w = omega[i];
  const int tg = plan.target[i];
  int base;
  double l[BAND_P];
  if (tg >= 0) {
    base = tg;
  } else {
    const int r = -tg - 1;
    base = plan.run_base[r];
    const double* nodes = plan.eval_omega + base;
    int hit = -1;
#pragma unroll
    for (int p = 0; p < BAND_P; ++p) hit = nodes[p] == w ? p : hit;
    if (hit >= 0) {
#pragma unroll
      for (int p = 0; p < BAND_P; ++p) l[p] = p == hit ? 1.0 : 0.0;
    } else {
      // barycentric formula in the evaluated node frequencies themselves (it is invariant under the affine
      // map to [-1, 1]); weights (-1)^p, halved at the two ends
      double sum = 0.0;
#pragma unroll
      for (int p = 0; p < BAND_P; ++p) {
        const double wp = (p == 0 || p == BAND_P - 1) ? 0.5 : 1.0;
        const double q = ((p & 1) ? -wp : wp) / (w - nodes[p]);
        l[p] = q;
        sum += q;
      }
      const double inv = 1.0 / sum;
#pragma unroll
      for (int p = 0; p < BAND_P; ++p) l[p] *= inv;
    }
  }
  double acc_re[BAND_EVAL_OUTS], acc_im[BAND_EVAL_OUTS];
#pragma unroll
  for (int o = 0; o < BAND_EVAL_OUTS; ++o) acc_re[o] = acc_im[o] = 0.0;
  const double2* part = reinterpret_cast<const double2*>(partial);
  for (int c = 0; c < S; ++c) {
    double sn, cs;
    sincos(w * chunk_centre(t, dt, G, L, c), &sn, &cs);
#pragma unroll
    for (int o = 0; o < BAND_EVAL_OUTS; ++o) {
      const int jk = jk0 + o;
      if (jk >= n_out) break;
      const int j = jk / n_basis, k = jk % n_basis;
      double re = 0.0, im = 0.0;
      for (int pj = 0; pj < parts_j; ++pj) {
        for (int pk = 0; pk < parts_k; ++pk) {
          int row = (j * parts_j + pj) * n_krows + k * parts_k + pk;
          if (split_rf > 0) row = k == 0 ? split_rf + j : j * (n_basis - 1) + k - 1;
          const double2* src = part + ((size_t)c * rows_pad + row) * n_slots + base;
          double zr, zi;
          if (tg >= 0) {
            const double2 z = src[0];
            zr = z.x;
            zi = z.y;
          } else {
            zr = 0.0;
            zi = 0.0;
#pragma unroll
            for (int p = 0; p < BAND_P; ++p) {
              const double2 z = src[p];
              zr = fma(l[p], z.x, zr);
              zi = fma(l[p], z.y, zi);
            }
          }
          switch ((pj + pk) & 3) {  // multiply by i^(pj+pk)
            case 0: re += zr; im += zi; break;
            case 1: re -= zi; im += zr; break;
            default: re -= zr; im -= zi; break;
          }
        }
      }
      acc_re[o] = fma(cs, re, fma(-sn, im, acc_re[o]));
      acc_im[o] = fma(cs, im, fma(sn, re, acc_im[o]));
    }
  }
#pragma unroll
  for (int o = 0; o < BAND_EVAL_OUTS; ++o) {
    const int jk = jk0 + o;
    if (jk < n_out) reinterpret_cast<double2*>(out)[(size_t)jk * ld_out + i] = make_double2(acc_re[o], acc_im[o]);
  }
}

// ------------------------------------------------------------------------------------------------
// launch plumbing
// ------------------------------------------------------------------------------------------------
constexpr int STAGE_TARGET_BYTES = 32 * 1024;
constexpr int STAGE_MAX_BYTES = 48 * 1024;

template <int MT, int NW>
int launch_main(ffb_ctx* ctx, MainParams p, int n_wtiles, int n_rb, int S, ffb_dispatch_record& disp,
                bool timed) {
  auto kern = ctrlmat_main_kernel<MT, NW>;
  snprintf(disp.kernel, sizeof disp.kernel, "ctrlmat_main_kernel<%d, %d>", MT, NW);
  const size_t smem = (size_t)2 * p.stage_doubles * sizeof(double);
  FFB_TRY(ffb_func_smem(ctx, kern, smem));
  dim3 grid(n_wtiles, n_rb, S);
  int slot = -1;
  if (timed) FFB_TRY(ffb_time_begin(ctx, &slot));
  kern<<<grid, NW * 32, smem, ctx->stream>>>(p);
  FFB_LAUNCHED(ctx);
  FFB_TRY(ffb_time_end(ctx, slot));
  return FFB_OK;
}

template <int MT, int NW, int NP, int NSP, bool SPLIT = false>
int launch_static(ffb_ctx* ctx, MainParams p, int n_wtiles, int n_rb, int S, ffb_dispatch_record& disp,
                  bool timed) {
  auto kern = ctrlmat_static_kernel<MT, NW, NP, NSP, SPLIT>;
  snprintf(disp.kernel, sizeof disp.kernel, "ctrlmat_static_kernel<%d, %d, %d, %d, %s>", MT, NW, NP, NSP,
           SPLIT ? "true" : "false");
  const size_t smem = (size_t)2 * p.stage_doubles * sizeof(double) + 16;  // + two mbarriers
  FFB_TRY(ffb_func_smem(ctx, kern, smem));
  dim3 grid(n_wtiles, n_rb, S);
  int slot = -1;
  if (timed) FFB_TRY(ffb_time_begin(ctx, &slot));
  kern<<<grid, NW * 32, smem, ctx->stream>>>(p);
  FFB_LAUNCHED(ctx);
  FFB_TRY(ffb_time_end(ctx, slot));
  return FFB_OK;
}

template <int MT, int NW>
int occupancy(ffb_ctx* ctx, size_t smem, int* blocks) {
  auto kern = ctrlmat_main_kernel<MT, NW>;
  return ffb_occupancy(ctx, kern, NW * 32, smem, blocks);
}

int pick_mt(int mt_total) {
  // (5, 7, 10 row tiles: five noise operators in a two-qubit basis = 80 rows, four in a qutrit basis = 36
  // rows, ...: a whole padding tile would cost 8 - 17 % of the DMMAs)
  static const int avail[] = {1, 2, 3, 4, 5, 6, 7, 8, 10, 12};
  const int n_rb = (mt_total + 11) / 12;
  const int need = (mt_total + n_rb - 1) / n_rb;
  for (int a : avail)
    if (a >= need) return a;
  return 12;
}

// Row tiles per warp and warps per CTA.  Heavy accumulator tiles (MT >= 8, 130-160 registers) run with
// 4 warps per CTA (one per scheduler; 6 measured slower because the schedulers are then unevenly
// loaded) so that three or four INDEPENDENT CTAs share an SM: their barriers and unit boundaries are
// uncorrelated, which keeps the FP64 pipe fed while one warp does its bookkeeping.
#define FFB_DISPATCH_MT(MTV, CALL)                                  \
  switch (MTV) {                                                    \
    case 1: { constexpr int MT_ = 1, NW_ = 8; CALL; } break;        \
    case 2: { constexpr int MT_ = 2, NW_ = 8; CALL; } break;        \
    case 3: { constexpr int MT_ = 3, NW_ = 8; CALL; } break;        \
    case 4: { constexpr int MT_ = 4, NW_ = 8; CALL; } break;        \
    case 5: { constexpr int MT_ = 5, NW_ = 8; CALL; } break;        \
    case 6: { constexpr int MT_ = 6, NW_ = 8; CALL; } break;        \
    case 7: { constexpr int MT_ = 7, NW_ = 4; CALL; } break;        \
    case 8: { constexpr int MT_ = 8, NW_ = 4; CALL; } break;        \
    case 10: { constexpr int MT_ = 10, NW_ = 4; CALL; } break;      \
    default: { constexpr int MT_ = 12, NW_ = 4; CALL; } break;      \
  }
inline int warps_per_cta(int MT) { return MT >= 7 ? 4 : 8; }

}  // namespace

// fixed-point variant on the int8 tensor cores (ffb_ctrlmat_i8.cu; opt-in, d = 4)
bool ffbi_ctrlmat_i8_eligible(int G, int d, int rows, int parts_j, int parts_k);
int ffbi_ctrlmat_i8_prepare(ffb_ctx* ctx, int G, int rows, int n_krows, const double* Bbar,
                            const double* Cbar, const double* eigvals, const double* dt,
                            const double* t, DevBuf& stream, DevBuf& scales);
int ffbi_ctrlmat_i8_run(ffb_ctx* ctx, int G, const double* omega, int n_omega, const DevBuf& stream,
                        const DevBuf& scales, DevBuf& partial, int* S_out, int* stages_per_chunk,
                        int* n_stages_out, int* n_tiles_out);

int ffbi_control_matrix(ffb_ctx* ctx, int G, int d, int n_nops, int n_basis, int n_omega,
                        const double* eigvals, const double* eigvecs, const double* propagators,
                        const double* omega, const double* basis, const double* n_opers,
                        const double* n_coeffs, const double* dt, const double* t, int herm_flags,
                        double* out_all, const FreqBlocks* blocks) {
  const double* const omega_all = omega;
  const int n_omega_all = n_omega;
  FFB_CHECK_DIM(ctx, d);
  FFB_REQUIRE(ctx, G >= 1 && d >= 1 && d <= 32, "control matrix: G=%d, d=%d unsupported", G, d);
  FFB_REQUIRE(ctx, n_nops >= 1 && n_basis >= 1 && n_omega >= 1,
              "control matrix: n_nops=%d n_basis=%d n_omega=%d must all be positive", n_nops,
              n_basis, n_omega);
  const int dd = d * d;
  const int parts_j = (herm_flags & FFB_HERM_NOPERS) ? 1 : 2;
  const int parts_k = (herm_flags & FFB_HERM_BASIS) ? 1 : 2;
  const int n_jrows = n_nops * parts_j, n_krows = n_basis * parts_k;
  const int rows = n_jrows * n_krows;
  const int MT = pick_mt(ceil_div(rows, 8));
  const int NW = warps_per_cta(MT);
  const StreamGeom geo = make_geom(rows, G, d, MT);
  const int rows_pad = geo.n_rb * MT * 8;
  // rows <= 16 and few level pairs: the DFMA variant (thread per frequency), see ctrlmat_dfma_kernel
  bool use_dfma = rows <= 16 && d >= 2 && d <= 3;
  if (const char* e = getenv("FFB_CTRLMAT_DFMA")) use_dfma = use_dfma && atoi(e) != 0;
  const int R = 4 * ceil_div(rows, 4);
  // rows (j, 0) of an identity basis element carry no pair coefficients (instances that exist:
  // d = 2 with 2-4 noise operators in a 4-element basis, d = 3 with one in a 9-element basis)
  bool split = use_dfma && (herm_flags & FFB_BASIS_IDENTITY0) && parts_j == 1 && parts_k == 1 &&
               ((d == 2 && n_basis == 4 && n_nops >= 2 && n_nops <= 4) ||
                (d == 3 && n_basis == 9 && n_nops == 1));
  if (const char* e = getenv("FFB_DFMA_SPLIT_IDENTITY")) split = split && atoi(e) != 0;
  const int RF = split ? n_nops * (n_basis - 1) : R;
  const int rec = dfma_rec_doubles(R, RF, d * (d - 1) / 2);

  // DFMA path: transforms and records in one kernel (Bbar / Cbar stay in shared memory)
  static const bool fused_ok = !(getenv("FFB_DFMA_FUSED_PROLOGUE") && atoi(getenv("FFB_DFMA_FUSED_PROLOGUE")) == 0);
  const size_t pro_smem = (size_t)DFMA_PRO_SEGS * (n_jrows + n_krows) * dd * 16;
  const bool fused_prologue = use_dfma && fused_ok && pro_smem <= 160 * 1024;
  const bool use_i8 = !use_dfma && ffbi_ctrlmat_i8_eligible(G, d, rows, parts_j, parts_k);
  // tensor path, two qubits with six noise operators in a basis whose element 0 is the identity: rows ordered
  // [(j, k >= 1) | (j, 0)] so that the last of the 12 row tiles carries only two rows with level-pair terms
  // (ctrlmat_static_kernel<..., SPLIT>); any other kernel simply sees permuted rows
  bool split_tensor = !use_dfma && !use_i8 && d == 4 && (herm_flags & FFB_BASIS_IDENTITY0) && parts_j == 1 &&
                      parts_k == 1 && n_basis == 16 && n_nops == 6 && MT == 12 && geo.n_rb == 1 && !geo.transposed;
  if (const char* e = getenv("FFB_CTRLMAT_SPLIT_IDENTITY")) split_tensor = split_tensor && atoi(e) != 0;
  const int split_t = split_tensor ? n_nops * (n_basis - 1) : 0;
  // block boundaries on multiples of 64 frequencies (the frequency tiles of all kernel variants)
  const int n_blocks = blocks ? std::max(1, std::min(blocks->n_blocks, ceil_div(n_omega_all, 64))) : 1;
  const int per_block = ceil_div(ceil_div(n_omega_all, n_blocks), 64) * 64;
  // banded route (DESIGN 4.1.1): tensor path in the regular layout, long pulses, blocks that can hold a band
  // worth interpolating.  Chunks of band_L segments, the shortest multiple of BAND_CHUNK_QUANTUM (doubled) whose
  // partials [S][rows_pad][per_block] stay within 1 GiB.
  const bool banded = !use_dfma && !use_i8 && !geo.transposed && d >= 2 && G >= BAND_MIN_G &&
                      std::min(per_block, n_omega_all) > BAND_P;
  int band_L = 0;
  if (banded) {
    band_L = BAND_CHUNK_QUANTUM;
    while (band_L < G && (size_t)ceil_div(G, band_L) * rows_pad * per_block * 16 > ((size_t)1 << 30)) band_L *= 2;
  }
  DevBuf Bbar, Cbar, stream, partial, i8_scales, plan_buf;
  std::string prologue;  // for the dispatch record
  if (!fused_prologue) {
    FFB_TRY(Bbar.alloc(ctx, (size_t)G * n_jrows * dd * 16));
    FFB_TRY(Cbar.alloc(ctx, (size_t)G * n_krows * dd * 16));
  }
  if (!use_i8)
    FFB_TRY(stream.alloc(ctx, use_dfma ? (size_t)G * rec * sizeof(double)
                                       : geo.rb_doubles * geo.n_rb * sizeof(double)));

  if (fused_prologue) {
    auto launch = [&](auto kern) -> int {
      FFB_TRY(ffb_func_smem(ctx, kern, pro_smem));
      kern<<<ceil_div(G, DFMA_PRO_SEGS), 128, pro_smem, ctx->stream>>>(
          G, n_nops, n_basis, parts_j, parts_k, rows, R, RF, split ? 1 : 0,
          reinterpret_cast<const double2*>(eigvecs), reinterpret_cast<const double2*>(propagators),
          reinterpret_cast<const double2*>(n_opers), n_coeffs, reinterpret_cast<const double2*>(basis),
          eigvals, dt, t, stream.as<double>());
      return FFB_OK;
    };
    if (d == 2) FFB_TRY(launch(dfma_prologue_kernel<2>));
    else FFB_TRY(launch(dfma_prologue_kernel<3>));
    prologue = d == 2 ? "dfma_prologue_kernel<2>" : "dfma_prologue_kernel<3>";
    FFB_LAUNCHED(ctx);
  } else if (d >= 2 && d <= 4) {
    const long long n_threads = (long long)G * (n_nops + n_basis);
    const unsigned blocks = (unsigned)((n_threads + 127) / 128);
    auto args = [&](auto kern) {
      kern<<<blocks, 128, 0, ctx->stream>>>(
          G, n_nops, n_basis, parts_j, parts_k, reinterpret_cast<const double2*>(eigvecs),
          reinterpret_cast<const double2*>(propagators), reinterpret_cast<const double2*>(n_opers),
          n_coeffs, reinterpret_cast<const double2*>(basis), Bbar.as<double2>(), Cbar.as<double2>());
    };
    if (d == 2) args(transform_small_kernel<2>);
    else if (d == 3) args(transform_small_kernel<3>);
    else args(transform_small_kernel<4>);
    prologue = "transform_small_kernel<" + std::to_string(d) + ">";
    FFB_LAUNCHED(ctx);
  } else {
    const size_t smem = (size_t)8 * dd * sizeof(double);
    FFB_CUDA(ctx, cudaFuncSetAttribute(transform_kernel,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int slices = std::max(1, std::min(n_nops + n_basis, ceil_div(8 * ctx->sm_count, G)));
    transform_kernel<<<dim3(G, slices), 128, smem, ctx->stream>>>(G, d, n_nops, n_basis, parts_j, parts_k, eigvecs,
                                                    propagators, n_opers, n_coeffs, basis,
                                                    Bbar.as<double>(), Cbar.as<double>());
    FFB_LAUNCHED(ctx);
    prologue = "transform_kernel";
  }
  if (fused_prologue) {
    // records written by dfma_prologue_kernel
  } else if (use_dfma) {
    const size_t total = (size_t)G * rec;
    const unsigned blocks = (unsigned)std::min<size_t>(ceil_div_sz(total, 256), (size_t)ctx->sm_count * 32);
    assemble_dfma_kernel<<<blocks, 256, 0, ctx->stream>>>(G, d, rows, R, RF, split ? 1 : 0, n_jrows, n_krows,
                                                          Bbar.as<double>(), Cbar.as<double>(),
                                                          eigvals, dt, t, stream.as<double>());
    FFB_LAUNCHED(ctx);
    prologue += "+assemble_dfma_kernel";
  } else if (use_i8) {
    // digit stream of the coefficients + per-segment constants (ffb_ctrlmat_i8.cu)
    FFB_TRY(ffbi_ctrlmat_i8_prepare(ctx, G, rows, n_krows, Bbar.as<double>(), Cbar.as<double>(), eigvals,
                                    dt, t, stream, i8_scales));
    prologue += "+i8_rowmax_kernel+i8_coeff_kernel";
  } else {
    // operators of a pass's segments in shared memory when they fit
    const size_t stage_bytes = (size_t)(geo.transposed ? 1 : 4) * (n_jrows + n_krows) * 2 * dd * sizeof(double);
    const unsigned blocks = (unsigned)(geo.n_rb * geo.n_pass);
    if (stage_bytes <= 96 * 1024) {
      FFB_TRY(ffb_func_smem(ctx, assemble_kernel<true>, stage_bytes));
      assemble_kernel<true><<<blocks, 256, stage_bytes, ctx->stream>>>(
          geo, G, d, rows, n_jrows, n_krows, split_t, band_L, Bbar.as<double>(), Cbar.as<double>(), eigvals, dt, t,
          stream.as<double>());
      prologue += "+assemble_kernel<true>";
    } else {
      assemble_kernel<false><<<blocks, 256, 0, ctx->stream>>>(
          geo, G, d, rows, n_jrows, n_krows, split_t, band_L, Bbar.as<double>(), Cbar.as<double>(), eigvals, dt, t,
          stream.as<double>());
      prologue += "+assemble_kernel<false>";
    }
    FFB_LAUNCHED(ctx);
  }

  // ---- omega-dependent part, per block of frequencies (one block unless the caller asked for more)
  const size_t ld_out = (size_t)n_omega_all;
  auto run_block = [&](const double* omega, int n_omega, double* out, ffb_dispatch_record& disp) -> int {
  if (use_i8) {
    int S_i8 = 1;
    FFB_TRY(ffbi_ctrlmat_i8_run(ctx, G, omega, n_omega, stream, i8_scales, partial, &S_i8,
                                &disp.passes_per_chunk, &disp.n_pass, &disp.n_wtiles));
    snprintf(disp.kernel, sizeof disp.kernel, "ctrlmat_i8_kernel");
    disp.S = S_i8;
    const size_t total = (size_t)n_nops * n_basis * n_omega;
    const unsigned fblocks = (unsigned)std::min<size_t>(ceil_div_sz(total, 256), (size_t)ctx->sm_count * 16);
    finalize_kernel<<<fblocks, 256, 0, ctx->stream>>>(S_i8, 96, n_nops, n_basis, 1, 1, n_omega, ld_out, 0,
                                                      partial.as<double>(), out);
    FFB_LAUNCHED(ctx);
    return FFB_OK;
  }
  if (use_dfma) {
    DfmaParams q;
    q.stream = stream.as<double>();
    q.omega = omega;
    q.n_omega = n_omega;
    q.G = G;
    q.n_pairs = d * (d - 1) / 2;
    q.rec_doubles = rec;
    if (!ctx->trig_table) {
      FFB_CUDA(ctx, cudaMalloc(&ctx->trig_table, TRIG_TABLE_SIZE * sizeof(double2)));
      trig_table_kernel<<<1, TRIG_TABLE_SIZE, 0, ctx->stream>>>(reinterpret_cast<double2*>(ctx->trig_table));
      FFB_LAUNCHED(ctx);
    }
    q.trig_table = reinterpret_cast<const double2*>(ctx->trig_table);
    q.stage_smem_doubles = (int)std::max((size_t)DFMA_WARPS * 2 * DFMA_STAGE_SEGS * rec,
                                         (size_t)DFMA_WARPS * 2 * R * 32);
    const size_t smem = ((size_t)q.stage_smem_doubles + 2 * TRIG_TABLE_SIZE) * sizeof(double);
    FFB_REQUIRE(ctx, smem <= 200 * 1024, "control matrix: DFMA stage does not fit shared memory");
    const int n_wt = ceil_div(n_omega, 32);
    int blocks_per_sm = 1;
    auto pick = [&](auto kern) -> int {
      return ffb_occupancy(ctx, kern, DFMA_WARPS * 32, smem, &blocks_per_sm);
    };
#define FFB_DFMA_DISPATCH(CALL)                                                        \
  if (split) {                                                                        \
    if (d == 3) { CALL(12, 8, 3); }                                                   \
    else if (R == 8) { CALL(8, 6, 1); }                                               \
    else if (R == 12) { CALL(12, 9, 1); }                                             \
    else { CALL(16, 12, 1); }                                                         \
  } else {                                                                            \
    switch (R) {                                                                      \
      case 4: if (d == 2) { CALL(4, 4, 1); } else { CALL(4, 4, 3); } break;           \
      case 8: if (d == 2) { CALL(8, 8, 1); } else { CALL(8, 8, 3); } break;           \
      case 12: if (d == 2) { CALL(12, 12, 1); } else { CALL(12, 12, 3); } break;      \
      default: if (d == 2) { CALL(16, 16, 1); } else { CALL(16, 16, 3); } break;      \
    }                                                                                 \
  }
#define FFB_DFMA_PICK(R_, RF_, NP_) FFB_TRY(pick(ctrlmat_dfma_kernel<R_, RF_, NP_>))
    FFB_DFMA_DISPATCH(FFB_DFMA_PICK)
    blocks_per_sm = std::max(1, blocks_per_sm);
    // split the segment axis over CTAs so that whole waves of CTAs are filled (same cost model as below)
    const long long slots = (long long)ctx->sm_count * blocks_per_sm;
    const int min_chunk = DFMA_WARPS * 16;  // at least 16 segments per warp
    long long s_cap = std::max(1, G / min_chunk);
    s_cap = std::min(s_cap, 64 * slots / n_wt + 1);
    int S = 1, chunk = G;
    double best_cost = 1e300;
    for (int sp = 1; sp <= (int)s_cap; ++sp) {
      int c = ceil_div(G, sp);
      c = ceil_div(c, DFMA_WARPS) * DFMA_WARPS;
      const int s_eff = ceil_div(G, c);
      const long long waves = ((long long)n_wt * s_eff + slots - 1) / slots;
      const double cost = (double)waves * (c / DFMA_WARPS + 6.0);
      if (cost < best_cost * 0.999) {
        best_cost = cost;
        S = s_eff;
        chunk = c;
      }
    }
    q.segs_per_cta = chunk;
    q.segs_per_warp = ceil_div(chunk, DFMA_WARPS);
    FFB_TRY(partial.alloc(ctx, (size_t)S * R * n_omega * 16));
    q.partial = partial.as<double>();
    dim3 grid(n_wt, S);
    int slot = -1;
    FFB_TRY(ffb_time_begin(ctx, &slot));
    const TrigConsts tc = trig_consts();
#define FFB_DFMA_LAUNCH(R_, RF_, NP_)                                                             \
  ctrlmat_dfma_kernel<R_, RF_, NP_><<<grid, DFMA_WARPS * 32, smem, ctx->stream>>>(q, tc);        \
  snprintf(disp.kernel, sizeof disp.kernel, "ctrlmat_dfma_kernel<%d, %d, %d>", R_, RF_, NP_)
    FFB_DFMA_DISPATCH(FFB_DFMA_LAUNCH)
    FFB_LAUNCHED(ctx);
    FFB_TRY(ffb_time_end(ctx, slot));
    disp.S = S;
    disp.passes_per_chunk = chunk;
    disp.n_pass = G;
    disp.n_wtiles = n_wt;
    const size_t total_out = (size_t)n_nops * n_basis * n_omega;
    const unsigned fblocks = (unsigned)std::min<size_t>(ceil_div_sz(total_out, 256), (size_t)ctx->sm_count * 16);
    finalize_kernel<<<fblocks, 256, 0, ctx->stream>>>(S, R, n_nops, n_basis, parts_j, parts_k, n_omega,
                                                      ld_out, split ? RF : 0, partial.as<double>(), out);
    FFB_LAUNCHED(ctx);
    return FFB_OK;
  }

  MainParams p;
  p.stream = stream.as<double>();
  p.omega = omega;
  p.n_omega = n_omega;
  p.rows_pad = rows_pad;
  p.n_pass = geo.n_pass;
  p.n_pairs = geo.n_pairs;
  p.pass_doubles = geo.pass_doubles;
  p.rb_doubles = geo.rb_doubles;
  p.diag_unit = geo.diag_unit;
  p.pair_unit = geo.pair_unit;
  // Stage size: small enough that shared memory does not limit the number of resident CTAs below what
  // the register file allows (independent CTAs decorrelate the warps that share an FP64 pipe), large
  // enough to amortise the two barriers per stage.
  int ctas_by_regs = 1;
  FFB_DISPATCH_MT(MT, FFB_TRY((occupancy<MT_, NW_>(ctx, 0, &ctas_by_regs))));
  ctas_by_regs = std::max(1, std::min(ctas_by_regs, 8));
  const size_t stage_budget = std::min<size_t>(STAGE_MAX_BYTES,
                                               ((size_t)216 * 1024 / ctas_by_regs) / 2);
  const size_t pass_bytes = geo.pass_doubles * sizeof(double);
  if (pass_bytes <= stage_budget) {
    p.n_sp = 1;
    p.pps = (int)std::max<size_t>(1, std::min<size_t>(stage_budget, STAGE_TARGET_BYTES) / pass_bytes);
    p.pps = std::min(p.pps, 32);
    p.stage_doubles = (int)(p.pps * geo.pass_doubles);
  } else {
    p.pps = 1;
    const int n_units = 1 + geo.n_pairs;
    int n_sp = (int)ceil_div_sz(pass_bytes, stage_budget);
    n_sp = std::min(n_sp, n_units);
    // largest piece under this split
    int max_piece = 0;
    for (;;) {
      max_piece = 0;
      for (int j = 0; j < n_sp; ++j) {
        const int u0 = (int)(((long long)j * n_units) / n_sp);
        const int u1 = (int)(((long long)(j + 1) * n_units) / n_sp);
        int len = (u1 - u0) * geo.pair_unit;
        if (u0 == 0) len += geo.diag_unit - geo.pair_unit;
        max_piece = std::max(max_piece, len);
      }
      if ((size_t)max_piece * sizeof(double) <= stage_budget || n_sp == n_units) break;
      ++n_sp;
    }
    p.n_sp = n_sp;
    p.stage_doubles = max_piece;
  }
  FFB_REQUIRE(ctx, (size_t)2 * p.stage_doubles * sizeof(double) <= 200 * 1024,
              "control matrix: stage of %d doubles does not fit shared memory", p.stage_doubles);

  // split the segment axis so that the grid fills the machine a few times over
  const int n_wtiles = ceil_div(n_omega, NW * 8);
  int blocks_per_sm = 1;
  const size_t smem = (size_t)2 * p.stage_doubles * sizeof(double);
  FFB_DISPATCH_MT(MT, FFB_TRY((occupancy<MT_, NW_>(ctx, smem, &blocks_per_sm))));
  blocks_per_sm = std::max(1, blocks_per_sm);
  const long long slots = (long long)ctx->sm_count * blocks_per_sm;
  const long long base_ctas = (long long)n_wtiles * geo.n_rb;
  // Pick the split S that minimises the makespan estimate waves(S) * (passes per chunk + overhead):
  // whole waves of CTAs, so the last wave is not left mostly empty (ncu on the first version: 4.24
  // waves -> 15 % of the SM cycles idle).
  const int min_passes = std::max(p.pps * 2, 8);  // do not cut chunks shorter than this
  long long s_cap = (long long)geo.n_pass / min_passes;
  s_cap = std::min(s_cap, 64 * slots / base_ctas + 1);
  s_cap = std::min(s_cap, (long long)(((size_t)1 << 30) / ((size_t)rows_pad * n_omega * 16)) + 1);
  const int S_max = banded ? 0 : (int)std::max<long long>(1, s_cap);
  const double overhead_passes = 2.0;
  int S = banded ? ceil_div(G, band_L) : 1, ppc = banded ? band_L / 4 : geo.n_pass;
  double best_cost = 1e300;
  for (int s = 1; s <= S_max; ++s) {
    int c = ceil_div(geo.n_pass, s);
    c = ceil_div(c, p.pps) * p.pps;
    const int s_eff = ceil_div(geo.n_pass, c);
    const long long waves = (base_ctas * s_eff + slots - 1) / slots;
    const double cost = (double)waves * (c + overhead_passes);
    if (cost < best_cost * 0.999) {
      best_cost = cost;
      S = s_eff;
      ppc = c;
    }
  }
  p.passes_per_chunk = ppc;

  FFB_TRY(partial.alloc(ctx, (size_t)S * rows_pad * n_omega * 16));
  p.partial = partial.as<double>();
  p.n_live = nullptr;
  BandPlan plan = {};
  int stage_slot = -1;  // the banded route times plan, main kernel and evaluation as one stage
  if (banded) {
    const size_t n = (size_t)n_omega;
    FFB_TRY(plan_buf.alloc(ctx, n * sizeof(double) + (4 * n + 4) * sizeof(int)));
    plan.eval_omega = plan_buf.as<double>();
    plan.target = reinterpret_cast<int*>(plan.eval_omega + n);
    plan.run_start = plan.target + n;
    plan.run_base = plan.run_start + n + 1;
    plan.counts = plan.run_base + n;
    if (!ctx->band_counts)
      FFB_CUDA(ctx, cudaMalloc(&ctx->band_counts, (size_t)2 * FFB_DISPATCH_LOG_MAX * sizeof(int)));
    const int log_slot = (int)(ctx->band_counts_next++ % FFB_DISPATCH_LOG_MAX);
    plan.log_counts = ctx->band_counts + 2 * log_slot;
    disp.route = 1;
    disp.chunk_segs = band_L;
    disp.n_bands = -(log_slot + 1);  // filled from the device by ffb_dispatch_log
    // an interpolated target costs S (2 P + 4) real multiply-adds per row, a direct one 2 (1 + d (d - 1)) G
    const double r_cost = (double)S * (2 * BAND_P + 4) / (2.0 * (1 + d * (d - 1)) * G);
    FFB_TRY(ffb_time_begin(ctx, &stage_slot));
    band_plan_kernel<<<1, BAND_PLAN_THREADS, 0, ctx->stream>>>(omega, n_omega, t, dt, G, band_L, S, r_cost, plan);
    FFB_LAUNCHED(ctx);
    p.omega = plan.eval_omega;
    p.n_live = plan.counts;
  }

  // d = 4 (6 level pairs), one pass per stage or a pass in two pieces: statically scheduled variant
  bool use_static = geo.n_pairs == 6 && !geo.transposed && p.pps == 1 && p.n_sp <= 2 &&
                    (MT == 12 || MT == 10 || MT == 8 || MT == 6);
  if (const char* e = getenv("FFB_CTRLMAT_STATIC")) use_static = use_static && atoi(e) != 0;
  // d = 8 (28 level pairs; 3 qubits): a pass of 29 units is streamed in 5 - 7 pieces; same kernel, the walk
  // over the units of a pass fully unrolled
  bool use_static8 = geo.n_pairs == 28 && !geo.transposed && p.pps == 1 &&
                     ((MT == 12 && p.n_sp >= 5 && p.n_sp <= 7) || (MT == 8 && p.n_sp >= 4 && p.n_sp <= 6));
  if (const char* e = getenv("FFB_CTRLMAT_STATIC")) use_static8 = use_static8 && atoi(e) != 0;
  // d = 16 in the transposed layout (short pulses: the gate pulses and the joined pulse of config 5): 30 units
  // of four level pairs each + the diagonal unit per segment
  bool use_static16 = geo.n_pairs == 30 && geo.transposed && p.pps == 1 && MT == 12 && p.n_sp == 7;
  if (const char* e = getenv("FFB_CTRLMAT_STATIC")) use_static16 = use_static16 && atoi(e) != 0;
  disp.S = S;
  disp.passes_per_chunk = ppc;
  disp.n_pass = geo.n_pass;
  disp.n_sp = p.n_sp;
  disp.pps = p.pps;
  disp.transposed = geo.transposed;
  disp.n_rb = geo.n_rb;
  disp.n_wtiles = n_wtiles;
  disp.ctas_by_regs = ctas_by_regs;
  if (use_static16) {
    FFB_TRY((launch_static<12, 4, 30, 7>(ctx, p, n_wtiles, geo.n_rb, S, disp, !banded)));
  } else if (use_static8) {
    if (MT == 12 && p.n_sp == 5) FFB_TRY((launch_static<12, 4, 28, 5>(ctx, p, n_wtiles, geo.n_rb, S, disp, !banded)));
    else if (MT == 12 && p.n_sp == 6) FFB_TRY((launch_static<12, 4, 28, 6>(ctx, p, n_wtiles, geo.n_rb, S, disp, !banded)));
    else if (MT == 12) FFB_TRY((launch_static<12, 4, 28, 7>(ctx, p, n_wtiles, geo.n_rb, S, disp, !banded)));
    else if (p.n_sp == 4) FFB_TRY((launch_static<8, 4, 28, 4>(ctx, p, n_wtiles, geo.n_rb, S, disp, !banded)));
    else if (p.n_sp == 5) FFB_TRY((launch_static<8, 4, 28, 5>(ctx, p, n_wtiles, geo.n_rb, S, disp, !banded)));
    else FFB_TRY((launch_static<8, 4, 28, 6>(ctx, p, n_wtiles, geo.n_rb, S, disp, !banded)));
  } else if (use_static) {
    if (MT == 12 && p.n_sp == 2 && split_t) FFB_TRY((launch_static<12, 4, 6, 2, true>(ctx, p, n_wtiles, geo.n_rb, S, disp, !banded)));
    else if (MT == 12 && p.n_sp == 2) FFB_TRY((launch_static<12, 4, 6, 2>(ctx, p, n_wtiles, geo.n_rb, S, disp, !banded)));
    else if (MT == 12) FFB_TRY((launch_static<12, 4, 6, 1>(ctx, p, n_wtiles, geo.n_rb, S, disp, !banded)));
    else if (MT == 10 && p.n_sp == 2) FFB_TRY((launch_static<10, 4, 6, 2>(ctx, p, n_wtiles, geo.n_rb, S, disp, !banded)));
    else if (MT == 10) FFB_TRY((launch_static<10, 4, 6, 1>(ctx, p, n_wtiles, geo.n_rb, S, disp, !banded)));
    else if (MT == 8 && p.n_sp == 2) FFB_TRY((launch_static<8, 4, 6, 2>(ctx, p, n_wtiles, geo.n_rb, S, disp, !banded)));
    else if (MT == 8) FFB_TRY((launch_static<8, 4, 6, 1>(ctx, p, n_wtiles, geo.n_rb, S, disp, !banded)));
    else if (p.n_sp == 2) FFB_TRY((launch_static<6, 8, 6, 2>(ctx, p, n_wtiles, geo.n_rb, S, disp, !banded)));
    else FFB_TRY((launch_static<6, 8, 6, 1>(ctx, p, n_wtiles, geo.n_rb, S, disp, !banded)));
  } else {
    FFB_DISPATCH_MT(MT, FFB_TRY((launch_main<MT_, NW_>(ctx, p, n_wtiles, geo.n_rb, S, disp, !banded))));
  }

  if (banded) {
    const dim3 grid(ceil_div(n_omega, 128), ceil_div(n_nops * n_basis, BAND_EVAL_OUTS));
    band_eval_kernel<<<grid, 128, 0, ctx->stream>>>(n_omega, S, band_L, G, rows_pad, n_nops, n_basis, parts_j,
                                                    parts_k, ld_out, split_t, omega, t, dt, plan,
                                                    partial.as<double>(), out);
    FFB_LAUNCHED(ctx);
    FFB_TRY(ffb_time_end(ctx, stage_slot));
  } else {
    const size_t total = (size_t)n_nops * n_basis * n_omega;
    const unsigned blocks = (unsigned)std::min<size_t>(ceil_div_sz(total, 256), (size_t)ctx->sm_count * 16);
    finalize_kernel<<<blocks, 256, 0, ctx->stream>>>(S, rows_pad, n_nops, n_basis, parts_j, parts_k,
                                                     n_omega, ld_out, split_t, partial.as<double>(), out);
    FFB_LAUNCHED(ctx);
  }
  return FFB_OK;
  };  // run_block

  const bool trace = ffb_trace();
  for (int w0 = 0; w0 < n_omega_all; w0 += per_block) {
    const int w1 = std::min(n_omega_all, w0 + per_block);
    ffb_dispatch_record disp = {};
    snprintf(disp.prologue, sizeof disp.prologue, "%s", prologue.c_str());
    disp.block = w0 / per_block;
    disp.n_blocks = ceil_div(n_omega_all, per_block);
    disp.n_omega = w1 - w0;
    FFB_TRY(run_block(omega_all + w0, w1 - w0, out_all + 2 * (size_t)w0, disp));
    if (ctx->dispatch_log.size() >= FFB_DISPATCH_LOG_MAX) ctx->dispatch_log.pop_front();
    ctx->dispatch_log.push_back(disp);
    if (trace)
      fprintf(stderr,
              "[ffb trace] control matrix G %d d %d rows %d, block %d/%d (%d frequencies): %s after %s; S %d "
              "passes_per_chunk %d n_pass %d n_sp %d pps %d transposed %d n_rb %d n_wtiles %d ctas_by_regs %d "
              "route %d chunk_segs %d\n",
              G, d, rows, disp.block + 1, disp.n_blocks, disp.n_omega, disp.kernel, disp.prologue, disp.S,
              disp.passes_per_chunk, disp.n_pass, disp.n_sp, disp.pps, disp.transposed, disp.n_rb, disp.n_wtiles,
              disp.ctas_by_regs, disp.route, disp.chunk_segs);
    if (blocks && blocks->after_block) FFB_TRY(blocks->after_block(w0, w1));
  }
  return FFB_OK;
}
