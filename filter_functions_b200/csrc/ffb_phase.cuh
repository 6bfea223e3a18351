// Apart from ffb_device.cuh: SC_K must not enter units that do not use it, where it moves their own constant tables.
// Phase factor and first-order integral of the control-matrix kernels (ffb_ctrlmat.cu, ffb_ctrlmat_i8.cu).
#pragma once

#include "ffb_common.cuh"

namespace {

// sin/cos with a Cody-Waite reduction.  fma keeps x - k*pi/2 accurate to ~1e-16 ABSOLUTE,
// which is what a unit-modulus phase factor needs (CUDA's sincos switches to Payne-Hanek above 1e5
// to keep the RELATIVE error near zeros of sin, which is irrelevant here).  Branch free.  Verified
// against sincos() on B200 up to |x| = 1e7 (max abs deviation 1.1e-16); beyond ~1e9 the rounding of
// the argument itself (ulp(w t) > 1e-7 rad) has destroyed the phase in the reference too.
// The constants live in constant memory so that they enter the DFMAs as c[bank][offset] operands: as
// immediates each one costs two UMOV/IMAD.MOV issue slots per use (ncu: 53 of the 258 instructions per
// warp and segment of the DFMA kernel), and 16 doubles are too many to pin in registers.
__constant__ double SC_K[16] = {
    6.36619772367581382433e-01,   // 0: 2/pi
    6755399441055744.0,           // 1: 1.5 * 2^52, round-to-nearest-integer by addition
    1.57079632679489655800e+00,   // 2: pi/2 high
    6.12323399573676603587e-17,   // 3: pi/2 middle
    1.58969099521155010221e-10,   // 4..9: sin polynomial
    -2.50507602534068634195e-08, 2.75573137070700676789e-06, -1.98412698298579493134e-04,
    8.33333333332248946124e-03, -1.66666666666666324348e-01,
    -1.13596475577881948265e-11,  // 10..15: cos polynomial
    2.08757232129817482790e-09, -2.75573143513906633035e-07, 2.48015872894767294178e-05,
    -1.38888888888741095749e-03, 4.16666666666666019037e-02};

__device__ __forceinline__ void sincos_cw(double x, double& sn, double& cs) {
  double kd = fma(x, SC_K[0], SC_K[1]);
  const int q = __double2loint(kd);
  kd -= SC_K[1];
  // two-constant Cody-Waite: the third term of pi/2 (1.5e-33 k) is below 1e-17 for |x| < 1e16
  double r = fma(-kd, SC_K[2], x);
  r = fma(-kd, SC_K[3], r);
  const double r2 = r * r;
  double ps = fma(r2, SC_K[4], SC_K[5]);
  ps = fma(ps, r2, SC_K[6]);
  ps = fma(ps, r2, SC_K[7]);
  ps = fma(ps, r2, SC_K[8]);
  ps = fma(ps, r2, SC_K[9]);
  const double s = fma(r * r2, ps, r);
  double pc = fma(r2, SC_K[10], SC_K[11]);
  pc = fma(pc, r2, SC_K[12]);
  pc = fma(pc, r2, SC_K[13]);
  pc = fma(pc, r2, SC_K[14]);
  pc = fma(pc, r2, SC_K[15]);
  const double c = fma(r2 * r2, pc, fma(r2, -0.5, 1.0));
  // quadrant: swap for odd q, flip signs through the sign bit (integer ops, not the FP64 pipe)
  const double ss = (q & 1) ? c : s;
  const double cc = (q & 1) ? s : c;
  const int s_flip = (q & 2) << 30;        // bit 31 of the high word
  const int c_flip = ((q + 1) & 2) << 30;
  sn = __hiloint2double(__double2hiint(ss) ^ s_flip, __double2loint(ss));
  cs = __hiloint2double(__double2hiint(cc) ^ c_flip, __double2loint(cc));
}

// 1/x to ~1 ulp: MUFU.RCP64H seed + two Newton steps on the FP64 pipe.
__device__ __forceinline__ double rcp_nr(double x) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  double e = fma(-x, r, 1.0);
  r = fma(r, e, r);
  e = fma(-x, r, 1.0);
  r = fma(r, e, r);
  return r;
}

constexpr double SQRT2 = 1.41421356237309504880;
// |sqrt(2) sin(x dt / 2)| below 2^-10 sqrt(2) -> direct evaluation.  Compared on the high word only
// (integer pipe: a DSETP would take an FP64-pipe slot).
constexpr int SMALL_SIN_HI = 0x3F56A09E;  // high word of 2^-10 sqrt(2)
__device__ __forceinline__ int abs_hi(double x) { return __double2hiint(x) & 0x7fffffff; }

// I(x) = (e^{i x dt} - 1) / (i x) evaluated directly with the rounding sequence of numeric.py:156-165
// (y = x * dt); = dt for x == 0.  Only used by the rare fix-up paths.
__device__ __forceinline__ cplx integral_direct(double x, double dt) {
  if (x == 0.0) return {dt, 0.0};
  double sn, cs;
  sincos_cw(0.5 * (x * dt), sn, cs);
  const double f = 2.0 * sn / x;
  return {cs * f, sn * f};
}

}  // namespace
