// K2 on the 5th-generation tensor cores: the control-matrix GEMM of ffb_ctrlmat.cu
//     B[(j,k), w] = sum_{(g,kappa)} A[(j,k), (g,kappa)] * P[(g,kappa), w]        (numeric.py:846-869)
// evaluated in FIXED POINT with tcgen05.mma.kind::i8 (Ozaki-style splitting): both operands are scaled
// to 39-bit integers and cut into five balanced base-256 digits (int8); the product of two operands
// is the sum of digit products d^A_j d^P_i 256^(i+j), of which the five most significant levels
// (i + j >= 4; 15 of 25 digit pairs) are accumulated EXACTLY in int32 accumulators in tensor memory.  B200
// runs int8 MMAs at ~120x its FP64 rate, so 15 int8 products per FP64 product are still ~6x cheaper;
// the right operand P (phase factors times first-order integrals) is generated in FP64 registers exactly
// as in the FP64 kernels, cut into digits on the fly and written straight into the shared-memory operand
// tiles -- it never exists in global memory.
//
// Accuracy.  Every K term carries the quantisation of two operands (2^-39 of their scales) and the
// dropped digit levels (~2^-37.6 of scale_A scale_P); the errors are zero-mean (balanced digits, round
// to nearest) and add up like sqrt(K).  Expected deviation from the FP64 kernels:
// ~7e-12 * scale_A scale_P sqrt(K) / max|B| -- 3e-12 .. 1e-11 for the bench workloads (measured, tests),
// inside the 1e-10 of the north-star with an order of magnitude to spare but not the 1e-15 of the FP64
// path.  The path is therefore OPT-IN (FFB_CTRLMAT_INT8=1) and restricted to the shape it pays for:
// d = 4 (13 real A columns per segment, padded to 16 K entries), Hermitian operators, <= 96 rows.
//
// Mapping (one CTA = 64 frequencies x one chunk of segments, 1 CTA per SM because it owns all of TMEM):
//   MMA  D[M = 128, N] += A_mma[128, K = 32] B_mma[N, 32]^T with
//     M rows  = (re | im) x 64 frequencies: digit plane i of P,
//     N cols  = the 96 rows of the control matrix: digit planes j of the coefficients (two planes, 192
//               columns, per instruction where the target levels are adjacent: 9 instructions per K step),
//     K       = 2 segments x 16 entries [diag, S_0, D_0, ..., S_5, D_5, 0, 0, 0],
//     D       = level t = i + j at TMEM columns 96 (t - 4) .. (480 of the 512 columns).
//   12 generator warps (thread = one frequency x one segment of the stage; <= 128 registers, the digits of a
//     value are extracted as soon as it exists) -> P digit tiles in shared memory;
//   1 thread streams the coefficient digit tiles + per-segment constants with cp.async.bulk (mbarrier tx);
//   1 thread issues the MMAs and commits them to the stage's "empty" barrier; 2-stage ring of 6 segments
//     (3 K steps, 27 MMAs per stage; 106 KB per stage).
//   Epilogue: TMEM -> registers (tcgen05.ld), Horner over the 5 levels in FP64, scale, split-K partial.
#include <algorithm>
#include <cstdlib>

#include "ffb_common.cuh"

namespace {

constexpr int I8_ROWS = 96;      // coefficient rows per CTA (N of the MMA; fewer rows are zero padded)
constexpr int I8_W = 64;         // frequencies per CTA: M = 128 = (re | im) x 64
constexpr int I8_D = 5;          // digits per operand
constexpr int I8_SEGS = 6;       // segments per stage = 3 K steps of 32
constexpr int I8_KS = I8_SEGS / 2;
constexpr int I8_STAGES = 2;
constexpr int I8_GEN_WARPS = 2 * I8_SEGS;   // thread = (frequency, segment of the stage): 64 x I8_SEGS items
constexpr int I8_THREADS = I8_GEN_WARPS * 32 + 64;  // + producer warp + MMA warp
constexpr int NP = 6;            // level pairs of d = 4
constexpr int I8_CONSTS = 2 + 3 * NP;               // per segment: t, dt, Omega[6], cos[6], sin[6]
constexpr int P_PLANE = 128 * 32;                   // bytes of one digit plane of P, one K step
constexpr int P_KSTEP = I8_D * P_PLANE;
constexpr int C_KSTEP = I8_D * I8_ROWS * 32;        // all five coefficient planes: one 480-row tile
constexpr int C_LBO = I8_D * I8_ROWS * 16;          // 7680: between the two 16-byte K chunks
constexpr int STAGE_P = I8_KS * P_KSTEP;                                 // 61440
constexpr int STAGE_C = I8_KS * C_KSTEP + I8_SEGS * I8_CONSTS * 8;      // 46080 + 960
constexpr int STAGE_BYTES = STAGE_P + STAGE_C;
constexpr int I8_MAX_CHUNK_STAGES = 1536 / I8_SEGS;  // 1536 segments: 5 pairs x 24576 K entries x 2^14 < 2^31
constexpr double I8_MAGIC = 6755399441055744.0 + 551911719040.0;  // 1.5 2^52 + sum_i 128 256^i

// ---- math helpers (same formulas and constants as ffb_ctrlmat.cu) ------------------------------------
__constant__ double SCK[16] = {
    6.36619772367581382433e-01, 6755399441055744.0, 1.57079632679489655800e+00,
    6.12323399573676603587e-17, 1.58969099521155010221e-10, -2.50507602534068634195e-08,
    2.75573137070700676789e-06, -1.98412698298579493134e-04, 8.33333333332248946124e-03,
    -1.66666666666666324348e-01, -1.13596475577881948265e-11, 2.08757232129817482790e-09,
    -2.75573143513906633035e-07, 2.48015872894767294178e-05, -1.38888888888741095749e-03,
    4.16666666666666019037e-02};

__device__ __forceinline__ void sincos_cw(double x, double& sn, double& cs) {
  double kd = fma(x, SCK[0], SCK[1]);
  const int q = __double2loint(kd);
  kd -= SCK[1];
  double r = fma(-kd, SCK[2], x);
  r = fma(-kd, SCK[3], r);
  const double r2 = r * r;
  double ps = fma(r2, SCK[4], SCK[5]);
  ps = fma(ps, r2, SCK[6]);
  ps = fma(ps, r2, SCK[7]);
  ps = fma(ps, r2, SCK[8]);
  ps = fma(ps, r2, SCK[9]);
  const double s = fma(r * r2, ps, r);
  double pc = fma(r2, SCK[10], SCK[11]);
  pc = fma(pc, r2, SCK[12]);
  pc = fma(pc, r2, SCK[13]);
  pc = fma(pc, r2, SCK[14]);
  pc = fma(pc, r2, SCK[15]);
  const double c = fma(r2 * r2, pc, fma(r2, -0.5, 1.0));
  const double ss = (q & 1) ? c : s;
  const double cc = (q & 1) ? s : c;
  const int s_flip = (q & 2) << 30;
  const int c_flip = ((q + 1) & 2) << 30;
  sn = __hiloint2double(__double2hiint(ss) ^ s_flip, __double2loint(ss));
  cs = __hiloint2double(__double2hiint(cc) ^ c_flip, __double2loint(cc));
}

__device__ __forceinline__ double rcp_nr(double x) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  double e = fma(-x, r, 1.0);
  r = fma(r, e, r);
  e = fma(-x, r, 1.0);
  r = fma(r, e, r);
  return r;
}

// 1 / x to ~2^-46 (seed 2^-23, one Newton step): the operand is cut to 39 bits afterwards, so the second
// Newton step of rcp_nr would be wasted (12 reciprocals per segment and frequency)
__device__ __forceinline__ double rcp_nr1(double x) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  const double e = fma(-x, r, 1.0);
  return fma(r, e, r);
}

constexpr double SQRT2 = 1.41421356237309504880;
constexpr int SMALL_SIN_HI = 0x3F56A09E;  // high word of 2^-10 sqrt(2)
__device__ __forceinline__ int abs_hi(double x) { return __double2hiint(x) & 0x7fffffff; }

// I(x) = (e^{i x dt} - 1) / (i x) with the rounding sequence of numeric.py:156-165; = dt for x == 0
__device__ __forceinline__ cplx integral_direct(double x, double dt) {
  if (x == 0.0) return {dt, 0.0};
  double sn, cs;
  sincos_cw(0.5 * (x * dt), sn, cs);
  const double f = 2.0 * sn / x;
  return {cs * f, sn * f};
}

// ---- PTX wrappers ------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(void* mbar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(mbar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(void* mbar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(mbar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(void* mbar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(mbar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(void* mbar, unsigned parity) {
  unsigned ok = 0;
  const unsigned addr = smem_u32(mbar);
  while (!ok) {
    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                 : "=r"(ok) : "r"(addr), "r"(parity) : "memory");
  }
}
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, unsigned bytes, void* mbar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(mbar))
               : "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// K-major, no swizzle: 16-byte unit (row r, K chunk c) at  base + c LBO + (r / 8) SBO + (r % 8) 16
__device__ __forceinline__ unsigned long long umma_desc(unsigned smem_addr, unsigned lbo, unsigned sbo) {
  unsigned long long d = 0;
  d |= (unsigned long long)((smem_addr >> 4) & 0x3FFF);
  d |= (unsigned long long)((lbo >> 4) & 0x3FFF) << 16;
  d |= (unsigned long long)((sbo >> 4) & 0x3FFF) << 32;
  d |= 1ull << 46;  // descriptor version of sm_100
  return d;
}
__device__ __forceinline__ unsigned umma_idesc_s8(int n) {
  return (2u << 4) | (1u << 7) | (1u << 10) | ((unsigned)(n >> 3) << 17) | ((128u >> 4) << 24);
}
// COLL: use of the collector buffer of the A operand -- 0: none, 1: fill (keep A for the next MMA), 2: use
// (reuse the kept A and keep it), 3: lastuse.  Consecutive MMAs of one P digit plane share A, which is then
// read from shared memory once instead of once per instruction (the MMA phase is bound by operand reads).
template <int COLL>
__device__ __forceinline__ void umma_i8(unsigned tmem_d, unsigned long long da, unsigned long long db,
                                        unsigned idesc) {
  if (COLL == 1)
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, 1, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::i8.collector::a::fill [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc) : "memory");
  else if (COLL == 2)
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, 1, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::i8.collector::a::use [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc) : "memory");
  else if (COLL == 3)
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, 1, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::i8.collector::a::lastuse [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc) : "memory");
  else
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, 1, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc) : "memory");
}
__device__ __forceinline__ void umma_commit(void* mbar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];"
               ::"r"(smem_u32(mbar)) : "memory");
}

#define TMEM_LD16(taddr, v)                                                                              \
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 "                                                 \
               "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"           \
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),     \
                 "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), \
                 "=r"(v[14]), "=r"(v[15])                                                                 \
               : "r"(taddr))

// ------------------------------------------------------------------------------------------------
// prologue: row maxima of A (and the largest dt), then the coefficient digit stream
// ------------------------------------------------------------------------------------------------
// A values of (row, segment): [diag, Re M_0, Im M_0, ..., Re M_5, Im M_5] with M_p = Bbar_j[m,n] Cbar_k[n,m]
// (ffb_ctrlmat.cu assemble_kernel); Bm / Cm point at the 4 x 4 complex matrices of the row's (j, k)
__device__ __forceinline__ void a_values(const double2* Bm, const double2* Cm, double (&a)[13]) {
  double diag = 0.0;
#pragma unroll
  for (int m = 0; m < 4; ++m) diag += Bm[m * 4 + m].x * Cm[m * 4 + m].x;
  a[0] = diag;
  int p = 0;
#pragma unroll
  for (int m = 0; m < 4; ++m)
#pragma unroll
    for (int n = m + 1; n < 4; ++n) {
      const double2 b = Bm[m * 4 + n], c = Cm[n * 4 + m];
      a[1 + 2 * p] = b.x * c.x - b.y * c.y;
      a[2 + 2 * p] = b.x * c.y + b.y * c.x;
      ++p;
    }
}

// scales[0 .. 95] = max_k |A[r, k]| as raw bits (non-negative doubles order like integers),
// scales[96] = max dt.  One block per stage of 4 segments, thread = (row, segment slot).
__global__ void __launch_bounds__(I8_ROWS * I8_SEGS)
i8_rowmax_kernel(int G, int rows, int n_krows, const double2* __restrict__ Bbar,
                 const double2* __restrict__ Cbar, const double* __restrict__ dt,
                 unsigned long long* __restrict__ scales) {
  __shared__ unsigned long long smax[I8_ROWS];
  const int r = threadIdx.x % I8_ROWS, c = threadIdx.x / I8_ROWS;
  const int g = blockIdx.x * I8_SEGS + c;
  if (threadIdx.x < I8_ROWS) smax[threadIdx.x] = 0ull;
  __syncthreads();
  if (g < G && r < rows) {
    const int n_jrows = rows / n_krows;
    double a[13];
    a_values(Bbar + ((size_t)g * n_jrows + r / n_krows) * 16, Cbar + ((size_t)g * n_krows + r % n_krows) * 16, a);
    double m = 0.0;
#pragma unroll
    for (int i = 0; i < 13; ++i) m = fmax(m, fabs(a[i]));
    atomicMax(&smax[r], (unsigned long long)__double_as_longlong(m));
  }
  __syncthreads();
  if (threadIdx.x < I8_ROWS && smax[threadIdx.x]) atomicMax(&scales[threadIdx.x], smax[threadIdx.x]);
  if (threadIdx.x == 0) {
    double m = 0.0;
    for (int i = 0; i < I8_SEGS; ++i)
      if (blockIdx.x * I8_SEGS + i < G) m = fmax(m, fabs(dt[blockIdx.x * I8_SEGS + i]));
    atomicMax(&scales[I8_ROWS], (unsigned long long)__double_as_longlong(m));
  }
}

// five balanced digits of round(x * scale) (|x * scale| <= 2^38): byte i of the result word pair is
// digit i + 128; lo holds digits 0..3, the low byte of hi digit 4
__device__ __forceinline__ void to_digits(double x, double scale, unsigned& lo, unsigned& hi) {
  const double y = fma(x, scale, I8_MAGIC);
  lo = (unsigned)__double2loint(y);
  hi = (unsigned)__double2hiint(y);
}

// Stream layout per stage of I8_SEGS segments:  [K step 0 | K step 1 | K step 2 | consts],  a K step being the 480-row tile
// [chunk cc = segment within the step][60 row groups][8 rows][16 bytes = kappa 0..15] with tall row
// 96 j + r for digit plane j of row r;  consts = I8_SEGS x [t, dt, Omega[6], cos(Omega dt/2)[6], sin(..)[6]].
__global__ void __launch_bounds__(I8_ROWS * I8_SEGS)
i8_coeff_kernel(int G, int rows, int n_krows, const double2* __restrict__ Bbar,
                const double2* __restrict__ Cbar, const double* __restrict__ eigvals,
                const double* __restrict__ dt, const double* __restrict__ t,
                const unsigned long long* __restrict__ scales, unsigned char* __restrict__ stream) {
  const int r = threadIdx.x % I8_ROWS, c = threadIdx.x / I8_ROWS;
  const int g = blockIdx.x * I8_SEGS + c;
  unsigned char* const stage = stream + (size_t)blockIdx.x * STAGE_C;
  unsigned words[I8_D][4];
#pragma unroll
  for (int j = 0; j < I8_D; ++j)
#pragma unroll
    for (int w = 0; w < 4; ++w) words[j][w] = 0u;  // digit 0 everywhere (padding rows / segments / kappa)
  if (g < G && r < rows) {
    const int n_jrows = rows / n_krows;
    double a[13];
    a_values(Bbar + ((size_t)g * n_jrows + r / n_krows) * 16, Cbar + ((size_t)g * n_krows + r % n_krows) * 16, a);
    const double amax = __longlong_as_double((long long)scales[r]);
    const double scale = amax > 0.0 ? 274877906944.0 / amax : 0.0;  // 2^38 / max|A_r|
#pragma unroll
    for (int k = 0; k < 13; ++k) {
      unsigned lo, hi;
      to_digits(a[k], scale, lo, hi);
      lo ^= 0x80808080u;
      hi ^= 0x80u;
#pragma unroll
      for (int j = 0; j < 4; ++j) words[j][k >> 2] |= ((lo >> (8 * j)) & 0xFFu) << (8 * (k & 3));
      words[4][k >> 2] |= (hi & 0xFFu) << (8 * (k & 3));
    }
  }
  const int ks = c >> 1, cc = c & 1;
#pragma unroll
  for (int j = 0; j < I8_D; ++j) {
    const int R = I8_ROWS * j + r;
    uint4* dst = reinterpret_cast<uint4*>(stage + (size_t)ks * C_KSTEP + (size_t)cc * C_LBO + (R >> 3) * 128 + (R & 7) * 16);
    *dst = make_uint4(words[j][0], words[j][1], words[j][2], words[j][3]);
  }
  // per-segment constants
  if (threadIdx.x < I8_SEGS * I8_CONSTS) {
    const int s = threadIdx.x / I8_CONSTS, e = threadIdx.x % I8_CONSTS;
    const int gs = blockIdx.x * I8_SEGS + s;
    double val = 0.0;
    if (e >= 2 + NP && e < 2 + 2 * NP) val = 1.0;  // cos of a padding segment
    if (gs < G) {
      if (e == 0) val = t[gs];
      else if (e == 1) val = dt[gs];
      else {
        const int p = (e - 2) % NP, which = (e - 2) / NP;
        int m = 0, n = 0, q = p;
        for (m = 0; q >= 3 - m; ++m) q -= 3 - m;
        n = m + 1 + q;
        const double Om = eigvals[(size_t)gs * 4 + m] - eigvals[(size_t)gs * 4 + n];
        if (which == 0) val = Om;
        else {
          double sn, cs;
          sincos(0.5 * (Om * dt[gs]), &sn, &cs);
          val = which == 1 ? cs : sn;
        }
      }
    }
    reinterpret_cast<double*>(stage + I8_KS * C_KSTEP)[threadIdx.x] = val;
  }
}

// ------------------------------------------------------------------------------------------------
// main kernel
// ------------------------------------------------------------------------------------------------
struct I8Params {
  const unsigned char* stream;
  const double* omega;
  const unsigned long long* scales;  // [96] row maxima (bits), [96] max dt
  double* partial;                   // [S][96][n_omega] complex
  int n_omega;
  int n_stages;                      // ceil(G / 4)
  int stages_per_chunk;
  int debug;                         // FFB_I8_DEBUG (timing experiments only): 1 = no MMAs issued, 2 = no operand
                                     // generation, 4 = generation without the shared-memory stores, 8 = stores without
                                     // the FP64 work
};

// 4 x 4 byte transpose: words a..d (4 values, digits 0..3 in their bytes) -> one word per digit plane
__device__ __forceinline__ void transpose4(unsigned a, unsigned b, unsigned c, unsigned d, unsigned (&w)[4]) {
  const unsigned x0 = __byte_perm(a, b, 0x5140), x1 = __byte_perm(a, b, 0x7362);
  const unsigned y0 = __byte_perm(c, d, 0x5140), y1 = __byte_perm(c, d, 0x7362);
  w[0] = __byte_perm(x0, y0, 0x5410);
  w[1] = __byte_perm(x0, y0, 0x7632);
  w[2] = __byte_perm(x1, y1, 0x5410);
  w[3] = __byte_perm(x1, y1, 0x7632);
}

// Digits of the 13 values of one operand row, collected as the values are produced (so that the FP64 values
// do not stay live): lo[k] = digits 0..3 of value k (one per byte), hi[k / 4] = digit 4 of four values.
struct DigitRow {
  unsigned lo[13];
  unsigned hi[4];
  __device__ __forceinline__ void clear() {
#pragma unroll
    for (int q = 0; q < 4; ++q) hi[q] = 0u;
  }
  template <int K>
  __device__ __forceinline__ void put(double v, double scale) {
    unsigned l, h;
    to_digits(v, scale, l, h);
    lo[K] = l;
    hi[K >> 2] |= (h & 0xFFu) << (8 * (K & 3));
  }
  // five digit planes of 16 bytes each, stored as one row of the P tile (plane stride P_PLANE)
  __device__ __forceinline__ void store(unsigned char* tile) const {
    unsigned plane[4][4];
#pragma unroll
    for (int q = 0; q < 3; ++q) {
      unsigned w[4];
      transpose4(lo[4 * q], lo[4 * q + 1], lo[4 * q + 2], lo[4 * q + 3], w);
#pragma unroll
      for (int j = 0; j < 4; ++j) plane[j][q] = w[j];
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) plane[j][3] = __byte_perm(lo[12], 0u, 0x4440 + j);
    // balanced digits: byte - 128 (the padding kappa 13..15 meet zero coefficients, their value is irrelevant)
#pragma unroll
    for (int j = 0; j < 4; ++j)
      *reinterpret_cast<uint4*>(tile + j * P_PLANE) =
          make_uint4(plane[j][0] ^ 0x80808080u, plane[j][1] ^ 0x80808080u, plane[j][2] ^ 0x80808080u,
                     plane[j][3] ^ 0x80808080u);
    *reinterpret_cast<uint4*>(tile + 4 * P_PLANE) =
        make_uint4(hi[0] ^ 0x80808080u, hi[1] ^ 0x80808080u, hi[2] ^ 0x80808080u, hi[3] ^ 0x80808080u);
  }
};

__global__ void __launch_bounds__(I8_THREADS, 1) ctrlmat_i8_kernel(const I8Params p) {
  extern __shared__ __align__(1024) unsigned char smem[];
  __shared__ __align__(8) unsigned long long bar_full_p[I8_STAGES], bar_full_c[I8_STAGES],
      bar_empty[I8_STAGES], bar_done;
  __shared__ unsigned tmem_base_s;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int w0 = blockIdx.x * I8_W;
  const int chunk = blockIdx.y;
  const int st0 = chunk * p.stages_per_chunk;
  const int n_st = max(0, min(p.stages_per_chunk, p.n_stages - st0));

  if (tid == 0) {
    for (int s = 0; s < I8_STAGES; ++s) {
      mbar_init(&bar_full_p[s], I8_GEN_WARPS);
      mbar_init(&bar_full_c[s], 1);
      mbar_init(&bar_empty[s], 1);
    }
    mbar_init(&bar_done, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == I8_GEN_WARPS) {  // the producer warp owns the tensor memory
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(&tmem_base_s)));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const unsigned tmem = tmem_base_s;
  // zero the accumulators (every MMA accumulates)
  if (warp < 4) {
    const unsigned z = 0u;
    for (int c0 = 0; c0 < I8_D * I8_ROWS; c0 += 16) {
      const unsigned taddr = tmem + ((unsigned)(warp * 32) << 16) + (unsigned)c0;
      asm volatile(
          "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
          "{%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1};" ::"r"(taddr), "r"(z) : "memory");
    }
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();

  if (warp < I8_GEN_WARPS) {
    // ===== generators: thread = (frequency wl, segment slot c of the stage) =====
    const int wl = tid & (I8_W - 1), c = tid >> 6;
    const int wi = min(w0 + wl, p.n_omega - 1);  // lanes beyond the grid repeat the last frequency
    const double w = p.omega[wi];
    const bool w_zero = fabs(w) < 1e-290;
    const double inv_w = 1.0 / w;
    const double dt_max = __longlong_as_double((long long)p.scales[I8_ROWS]);
    const double p_scale = 274877906944.0 / (2.000001 * dt_max + 1e-300);  // 2^38 / scale_P
    double dt_prev = -1.0, hc = 0.0, hs = 0.0, j0_re = 0.0, j0_im = 0.0;
    const int ks = c >> 1, cc = c & 1;
    for (int it = 0; it < n_st; ++it) {
      const int s = it % I8_STAGES;
      const unsigned ph = (unsigned)(it / I8_STAGES) & 1u;
      unsigned char* const sP = smem + (size_t)s * STAGE_BYTES;
      const double* cst = reinterpret_cast<const double*>(sP + STAGE_P + I8_KS * C_KSTEP) + c * I8_CONSTS;
      if (p.debug & 16)   // timing experiment: per-segment constants straight from global memory (L1 / L2)
        cst = reinterpret_cast<const double*>(p.stream + (size_t)(st0 + it) * STAGE_C + I8_KS * C_KSTEP) + c * I8_CONSTS;
      mbar_wait(&bar_empty[s], ph ^ 1u);   // the MMAs of the previous use of this stage are done
      mbar_wait(&bar_full_c[s], ph);       // constants (and coefficients) of this stage have landed
      if (p.debug & 2) {
        __syncwarp();
        if (lane == 0) mbar_arrive(&bar_full_p[s]);
        continue;
      }
      if (p.debug & 8) {
        const uint4 z = make_uint4(tid, it, 0u, 0u);
        unsigned char* const tile = sP + (size_t)ks * P_KSTEP + (size_t)cc * 2048;
#pragma unroll
        for (int j = 0; j < I8_D; ++j) {
          *reinterpret_cast<uint4*>(tile + (size_t)wl * 16 + j * P_PLANE) = z;
          *reinterpret_cast<uint4*>(tile + (size_t)(I8_W + wl) * 16 + j * P_PLANE) = z;
        }
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bar_full_p[s]);
        continue;
      }
      const double tg = cst[0], dtg = cst[1];
      if (__double_as_longlong(dtg) != __double_as_longlong(dt_prev)) {
        double sn, cs;
        sincos_cw(0.5 * (w * dtg), sn, cs);
        hc = SQRT2 * cs;
        hs = SQRT2 * sn;
        const double f = hs * inv_w;
        j0_re = w_zero ? dtg : hc * f;
        j0_im = w_zero ? 0.0 : hs * f;
        dt_prev = dtg;
      }
      double ph_re, ph_im;
      sincos_cw(w * tg, ph_im, ph_re);
      // E = e^{i w t} sqrt2 e^{i w dt / 2}: the phase factor folded into the half-angle factor, so that the
      // products below come out rotated already (8 FP64 operations per level pair less than rotating S, D)
      const double e_re = ph_re * hc - ph_im * hs, e_im = ph_re * hs + ph_im * hc;
      DigitRow dre, dim;
      dre.clear();
      dim.clear();
      dre.put<0>(ph_re * j0_re - ph_im * j0_im, p_scale);
      dim.put<0>(ph_re * j0_im + ph_im * j0_re, p_scale);
      bool any_store = !(p.debug & 4);
#pragma unroll
      for (int q = 0; q < NP; ++q) {
        const double Om = cst[2 + q], Ch = cst[2 + NP + q], Sh = cst[2 + 2 * NP + q];
        const double u1 = e_re * Ch, u3 = e_im * Ch, t3 = hs * Ch;
        const double sp = fma(hc, Sh, t3), sm = fma(-hc, Sh, t3);     // sqrt2 sin((w +- Om) dt / 2)
        double jp_re, jp_im, jm_re, jm_im;                              // e^{i w t} I(w +- Om)
        if (min(abs_hi(sp), abs_hi(sm)) < SMALL_SIN_HI) {  // removable singularity: direct evaluation
          const cplx jp = integral_direct(w + Om, dtg), jm = integral_direct(w - Om, dtg);
          jp_re = ph_re * jp.re - ph_im * jp.im; jp_im = ph_re * jp.im + ph_im * jp.re;
          jm_re = ph_re * jm.re - ph_im * jm.im; jm_im = ph_re * jm.im + ph_im * jm.re;
        } else {
          const double fp = sp * rcp_nr1(w + Om);
          const double fm = sm * rcp_nr1(w - Om);
          jp_re = fma(-e_im, Sh, u1) * fp; jp_im = fma(e_re, Sh, u3) * fp;
          jm_re = fma(e_im, Sh, u1) * fm;  jm_im = fma(-e_re, Sh, u3) * fm;
        }
        // S = jp + jm, D = i (jp - jm)
        if (q == 0) { dre.put<1>(jp_re + jm_re, p_scale); dim.put<1>(jp_im + jm_im, p_scale);
                      dre.put<2>(jm_im - jp_im, p_scale); dim.put<2>(jp_re - jm_re, p_scale); }
        if (q == 1) { dre.put<3>(jp_re + jm_re, p_scale); dim.put<3>(jp_im + jm_im, p_scale);
                      dre.put<4>(jm_im - jp_im, p_scale); dim.put<4>(jp_re - jm_re, p_scale); }
        if (q == 2) { dre.put<5>(jp_re + jm_re, p_scale); dim.put<5>(jp_im + jm_im, p_scale);
                      dre.put<6>(jm_im - jp_im, p_scale); dim.put<6>(jp_re - jm_re, p_scale); }
        if (q == 3) { dre.put<7>(jp_re + jm_re, p_scale); dim.put<7>(jp_im + jm_im, p_scale);
                      dre.put<8>(jm_im - jp_im, p_scale); dim.put<8>(jp_re - jm_re, p_scale); }
        if (q == 4) { dre.put<9>(jp_re + jm_re, p_scale); dim.put<9>(jp_im + jm_im, p_scale);
                      dre.put<10>(jm_im - jp_im, p_scale); dim.put<10>(jp_re - jm_re, p_scale); }
        if (q == 5) { dre.put<11>(jp_re + jm_re, p_scale); dim.put<11>(jp_im + jm_im, p_scale);
                      dre.put<12>(jm_im - jp_im, p_scale); dim.put<12>(jp_re - jm_re, p_scale); }
      }
      unsigned char* const tile = sP + (size_t)ks * P_KSTEP + (size_t)cc * 2048;
      if (p.debug & 4) any_store = (dre.lo[12] ^ dim.lo[7] ^ dre.hi[1]) == 0x12345678u;  // timing experiment
      if (any_store) {
        dre.store(tile + (size_t)wl * 16);             // rows 0..63: real parts
        dim.store(tile + (size_t)(I8_W + wl) * 16);    // rows 64..127: imaginary parts
      }
      fence_proxy_async();  // generic-proxy stores -> visible to the tensor core's async proxy
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_full_p[s]);
    }
  } else if (warp == I8_GEN_WARPS) {
    // ===== producer: coefficient digits + constants of a stage in one bulk copy =====
    if (lane == 0) {
      for (int it = 0; it < n_st; ++it) {
        const int s = it % I8_STAGES;
        const unsigned ph = (unsigned)(it / I8_STAGES) & 1u;
        mbar_wait(&bar_empty[s], ph ^ 1u);
        mbar_expect_tx(&bar_full_c[s], STAGE_C);
        bulk_g2s(smem + (size_t)s * STAGE_BYTES + STAGE_P, p.stream + (size_t)(st0 + it) * STAGE_C, STAGE_C,
                 &bar_full_c[s]);
      }
    }
  } else {
    // ===== MMA issuer =====
    if (lane == 0) {
      const unsigned idesc96 = umma_idesc_s8(96), idesc192 = umma_idesc_s8(192);
      for (int it = 0; it < n_st; ++it) {
        const int s = it % I8_STAGES;
        const unsigned ph = (unsigned)(it / I8_STAGES) & 1u;
        mbar_wait(&bar_full_c[s], ph);
        mbar_wait(&bar_full_p[s], ph);
        tc_fence_after();
        const unsigned sP = smem_u32(smem + (size_t)s * STAGE_BYTES);
        const unsigned sC = sP + STAGE_P;
#pragma unroll
        for (int ks = 0; ks < I8_KS; ++ks) {
          if (p.debug & 1) break;
          // P plane i (digit i) x coefficient planes j with i + j >= 4; level t = i + j at column 96 (t - 4);
          // two adjacent planes (adjacent levels) per instruction where possible
#pragma unroll
          for (int i = 0; i < I8_D; ++i) {
            const unsigned long long da = umma_desc(sP + ks * P_KSTEP + i * P_PLANE, 2048, 128);
            const int n_mma = (i + 2) / 2;   // coefficient planes 4 - i .. 4 in groups of two
            int j = 4 - i, m = 0;
            while (j <= 4) {
              const int nj = (j + 1 <= 4) ? 2 : 1;
              const unsigned long long db = umma_desc(sC + ks * C_KSTEP + j * (I8_ROWS * 16), C_LBO, 128);
              const unsigned d_at = tmem + (unsigned)((i + j - 4) * I8_ROWS);
              const unsigned idesc = nj == 2 ? idesc192 : idesc96;
              if (n_mma == 1) umma_i8<0>(d_at, da, db, idesc);
              else if (m == 0) umma_i8<1>(d_at, da, db, idesc);
              else if (m == n_mma - 1) umma_i8<3>(d_at, da, db, idesc);
              else umma_i8<2>(d_at, da, db, idesc);
              j += nj;
              ++m;
            }
          }
        }
        umma_commit(&bar_empty[s]);  // frees the stage when these MMAs have read it
      }
      umma_commit(&bar_done);
    }
  }

  // ===== epilogue: TMEM -> registers, Horner over the levels, scale, partial sums =====
  if (warp < 4) {
    mbar_wait(&bar_done, 0u);
    tc_fence_after();
    const int m = warp * 32 + lane;          // row of D: (re | im) x frequency
    const int wl = m & (I8_W - 1), reim = m >> 6;
    const int wi = w0 + wl;
    const double dt_max = __longlong_as_double((long long)p.scales[I8_ROWS]);
    const double out_scale = (2.000001 * dt_max + 1e-300) * 5.6843418860808015e-14;  // scale_P 2^-44
    double* const out = p.partial + ((size_t)chunk * I8_ROWS * p.n_omega + wi) * 2 + reim;
    for (int c0 = 0; c0 < I8_ROWS; c0 += 16) {
      unsigned v[I8_D][16];
#pragma unroll
      for (int t = 0; t < I8_D; ++t) {
        const unsigned taddr = tmem + ((unsigned)(warp * 32) << 16) + (unsigned)(t * I8_ROWS + c0);
        TMEM_LD16(taddr, v[t]);
      }
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      if (wi < p.n_omega) {
#pragma unroll
        for (int jj = 0; jj < 16; ++jj) {
          double acc = (double)(int)v[4][jj];
#pragma unroll
          for (int t = 3; t >= 0; --t) acc = fma(acc, 256.0, (double)(int)v[t][jj]);
          const int r = c0 + jj;
          const double amax = __longlong_as_double((long long)p.scales[r]);
          out[(size_t)r * p.n_omega * 2] = acc * (amax * out_scale);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == I8_GEN_WARPS) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem));
  }
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// host side (called from ffbi_control_matrix)
// ------------------------------------------------------------------------------------------------
bool ffbi_ctrlmat_i8_eligible(int G, int d, int rows, int parts_j, int parts_k) {
  const char* e = getenv("FFB_CTRLMAT_INT8");
  if (!e || atoi(e) == 0) return false;
  return d == 4 && parts_j == 1 && parts_k == 1 && rows <= I8_ROWS && G >= 64;
}

int ffbi_ctrlmat_i8_prepare(ffb_ctx* ctx, int G, int rows, int n_krows, const double* Bbar,
                            const double* Cbar, const double* eigvals, const double* dt,
                            const double* t, DevBuf& stream, DevBuf& scales) {
  const int n_stages = ceil_div(G, I8_SEGS);
  FFB_TRY(stream.alloc(ctx, (size_t)n_stages * STAGE_C));
  FFB_TRY(scales.alloc(ctx, (I8_ROWS + 1) * sizeof(unsigned long long)));
  FFB_CUDA(ctx, cudaMemsetAsync(scales.p, 0, (I8_ROWS + 1) * sizeof(unsigned long long), ctx->stream));
  i8_rowmax_kernel<<<n_stages, I8_ROWS * I8_SEGS, 0, ctx->stream>>>(
      G, rows, n_krows, reinterpret_cast<const double2*>(Bbar), reinterpret_cast<const double2*>(Cbar), dt,
      scales.as<unsigned long long>());
  FFB_LAUNCHED(ctx);
  i8_coeff_kernel<<<n_stages, I8_ROWS * I8_SEGS, 0, ctx->stream>>>(
      G, rows, n_krows, reinterpret_cast<const double2*>(Bbar), reinterpret_cast<const double2*>(Cbar),
      eigvals, dt, t, scales.as<unsigned long long>(), stream.as<unsigned char>());
  FFB_LAUNCHED(ctx);
  return FFB_OK;
}

// Partial sums [S][96][n_omega] complex for one block of frequencies; *S_out chunks of the segment axis
// of *stages_per_chunk stages each, *n_stages_out stages, *n_tiles_out frequency tiles.
int ffbi_ctrlmat_i8_run(ffb_ctx* ctx, int G, const double* omega, int n_omega, const DevBuf& stream,
                        const DevBuf& scales, DevBuf& partial, int* S_out, int* stages_per_chunk,
                        int* n_stages_out, int* n_tiles_out) {
  const int n_stages = ceil_div(G, I8_SEGS);
  const int n_tiles = ceil_div(n_omega, I8_W);
  // split of the segment axis: whole waves of CTAs (one CTA per SM), chunks short enough for int32
  const int s_min = ceil_div(n_stages, I8_MAX_CHUNK_STAGES);
  const int s_max = std::max(s_min, std::min(64, n_stages / 8));
  int S = s_min;
  double best = 1e300;
  for (int s = s_min; s <= s_max; ++s) {
    const int spc = ceil_div(n_stages, s);
    const int s_eff = ceil_div(n_stages, spc);
    const long long waves = ((long long)n_tiles * s_eff + ctx->sm_count - 1) / ctx->sm_count;
    const double cost = (double)waves * (spc + 6.0);
    if (cost < best * 0.999) {
      best = cost;
      S = s_eff;
    }
  }
  const int spc = ceil_div(n_stages, S);
  S = ceil_div(n_stages, spc);
  FFB_TRY(partial.alloc(ctx, (size_t)S * I8_ROWS * n_omega * 16));
  I8Params p;
  p.stream = stream.as<unsigned char>();
  p.omega = omega;
  p.scales = scales.as<unsigned long long>();
  p.partial = partial.as<double>();
  p.n_omega = n_omega;
  p.n_stages = n_stages;
  p.stages_per_chunk = spc;
  static const int debug = getenv("FFB_I8_DEBUG") ? atoi(getenv("FFB_I8_DEBUG")) : 0;
  p.debug = debug;
  const size_t smem = (size_t)I8_STAGES * STAGE_BYTES + 1024;
  FFB_TRY(ffb_func_smem(ctx, ctrlmat_i8_kernel, smem));
  int slot = -1;
  FFB_TRY(ffb_time_begin(ctx, &slot));
  ctrlmat_i8_kernel<<<dim3(n_tiles, S), I8_THREADS, smem, ctx->stream>>>(p);
  FFB_LAUNCHED(ctx);
  FFB_TRY(ffb_time_end(ctx, slot));
  *S_out = S;
  *stages_per_chunk = spc;
  *n_stages_out = n_stages;
  *n_tiles_out = n_tiles;
  return FFB_OK;
}
