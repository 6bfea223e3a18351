/* ffb200 -- C ABI of the B200-native control-matrix / filter-function / infidelity engine.
 *
 * The reference (qutech/filter_functions v1.2.1) is pure Python and has no FFI seam; the drop-in
 * boundary is the set of Python signatures of its hot path.  Every entry point below replaces the
 * BODY of one of those functions and is bound from `filter_functions_b200/_lib.py` with ctypes.
 * The reference-side binding a maintainer would add is shown in INTEGRATION.md.
 *
 * Conventions
 *   - plain C, no C++ or torch types; all arrays are C-contiguous;
 *   - complex128 is `double[2]` (re, im interleaved), passed as `const double*` / `double*`;
 *   - `ffb_*`      : pointers are HOST pointers, the call is synchronous (results are in the output
 *                    buffers on return); host<->device copies happen inside the call;
 *   - `ffb_dev_*`  : pointers are DEVICE pointers on the context's GPU, the call only enqueues work
 *                    on the context's stream (see ffb_set_stream / ffb_sync);
 *   - every function returns 0 on success or a negative FFB_E* code; ffb_last_error(ctx) returns
 *     the message.  No C++ exception crosses the boundary.  There is no CPU fallback: without a
 *     usable sm_100 device ffb_init fails with FFB_ENODEVICE.
 *   - a context is bound to one GPU and must be used from one thread at a time (the reference is
 *     single-threaded Python, util.py:1103-1109).
 *
 * Citations are `file:line` relative to /root/reference/filter_functions.
 */
#ifndef FFB200_H
#define FFB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ffb_ctx ffb_ctx;

enum {
  FFB_OK = 0,
  FFB_EINVAL = -1,    /* -> ValueError  */
  FFB_ENODEVICE = -2, /* -> RuntimeError: no CUDA device / wrong architecture */
  FFB_ECUDA = -3,     /* -> RuntimeError: CUDA runtime error */
  FFB_ENOMEM = -4,    /* -> MemoryError */
  FFB_ENOTCONV = -5   /* -> util.CalculationError: eigensolver did not converge */
};

/* ---- context -------------------------------------------------------------------------------- */
int ffb_init(ffb_ctx** ctx, int device);
void ffb_destroy(ffb_ctx* ctx);
const char* ffb_last_error(const ffb_ctx* ctx);
const char* ffb_version(void);
/* external != 0: enqueue all subsequent work on the externally owned cudaStream_t `cuda_stream`
 * (e.g. torch's current stream; NULL is the legacy default stream).  external == 0: go back to the
 * context's own non-blocking stream. */
int ffb_set_stream(ffb_ctx* ctx, void* cuda_stream, int external);
int ffb_sync(ffb_ctx* ctx);
/* Number of kernels this library has launched on this context since creation. */
int64_t ffb_launch_count(const ffb_ctx* ctx);
int ffb_device_info(ffb_ctx* ctx, int* sm_count, int* cc_major, int* cc_minor, size_t* total_mem);
/* Measures the DFMA / DMMA peak of the device with a short register-resident kernel (TFLOP/s).
 * The FP64 roofline denominator; MEASURED_PEAKS.json only holds HBM and bf16. */
int ffb_measure_fp64_peak(ffb_ctx* ctx, double* dfma_tflops, double* dmma_tflops);

/* ---- a1: diagonalisation and propagators ------------------------------------------------------
 * Replaces PulseSequence.diagonalize (pulse_sequence.py:577-586) + numeric.diagonalize
 * (numeric.py:1886-1935).  H_g = sum_i c_coeffs[i,g] c_opers[i]; batched Hermitian Jacobi, ascending
 * eigenvalues; P_g = V exp(-i D dt_g) V^dagger; propagators = [1, P_0, P_1 P_0, ...].
 *   c_opers (n_cops,d,d) c128 | c_coeffs (n_cops,G) f64 | dt (G) f64
 *   eigvals (G,d) f64 | eigvecs (G,d,d) c128 (columns) | propagators (G+1,d,d) c128
 * If c_coeffs is NULL, c_opers is taken to be the Hamiltonian itself, shape (G,d,d)
 * (the numeric.diagonalize(hamiltonian, dt) signature, numeric.py:1886). */
int ffb_diagonalize(ffb_ctx* ctx, int G, int d, int n_cops, const double* c_opers,
                    const double* c_coeffs, const double* dt, double* eigvals, double* eigvecs,
                    double* propagators);

/* ---- a2: first-order control matrix from scratch ----------------------------------------------
 * Replaces numeric.calculate_control_matrix_from_scratch (numeric.py:707-881).
 *   eigvals (G,d) | eigvecs (G,d,d) | propagators (G+1,d,d) | omega (n_omega) | basis (n_basis,d,d)
 *   n_opers (n_nops,d,d) | n_coeffs (n_nops,G) | dt (G) | t (G+1)
 *   out (n_nops,n_basis,n_omega) c128, omega fastest. */
int ffb_control_matrix_from_scratch(ffb_ctx* ctx, int G, int d, int n_nops, int n_basis,
                                    int n_omega, const double* eigvals, const double* eigvecs,
                                    const double* propagators, const double* omega,
                                    const double* basis, const double* n_opers,
                                    const double* n_coeffs, const double* dt, const double* t,
                                    double* out);

/* ---- a3 / a4: filter functions -----------------------------------------------------------------
 * Replaces numeric.calculate_filter_function (numeric.py:1413-1467) and
 * numeric.calculate_pulse_correlation_filter_function (numeric.py:1821-1883).
 *   B (P,n_nops,n_basis,n_omega) c128 with P = 1 for the plain filter function
 *   F fidelity    : (P,P,n_nops,n_nops,n_omega)
 *   F generalized : (P,P,n_nops,n_nops,n_basis,n_basis,n_omega) */
int ffb_filter_function(ffb_ctx* ctx, int P, int n_nops, int n_basis, int n_omega, const double* B,
                        int generalized, double* F);

/* ---- a5: control matrix of a sequence from those of its parts ---------------------------------
 * Replaces numeric.calculate_control_matrix_from_atomic (numeric.py:621-704).
 *   phases (P-1,n_omega) c128 | B_atomic (P,n_nops,n_basis,n_omega) c128
 *   Q_liouville (P-1,n_basis,n_basis) f64, or c128 if q_is_complex
 *   out (n_nops,n_basis,n_omega), or (P,n_nops,n_basis,n_omega) if correlations != 0 */
int ffb_control_matrix_from_atomic(ffb_ctx* ctx, int P, int n_nops, int n_basis, int n_omega,
                                   const double* phases, const double* B_atomic,
                                   const double* Q_liouville, int q_is_complex, int correlations,
                                   double* out);

/* ---- a7: infidelity integral --------------------------------------------------------------------
 * Replaces the integrand + trapezoid of numeric.infidelity (numeric.py:2318-2320, :259-374,
 * util.py:880-906).  F (n_lead,n_nops,n_nops,n_omega) c128 (n_lead = P*P for pulse correlations,
 * else 1); idx (n_sel) noise-operator indices; spectrum, already broadcast by the caller, is
 *   spectrum_ndim 1: (n_omega) | 2: (n_sel,n_omega) | 3: (n_sel,n_sel,n_omega), f64 or c128;
 * out f64: (n_lead,n_sel) for ndim 1/2, (n_lead,n_sel,n_sel) for ndim 3.
 * out = trapezoid(Re(F[idx..]*S)) / (2 pi d). */
int ffb_infidelity(ffb_ctx* ctx, int n_lead, int n_nops, int n_sel, const int* idx, int n_omega,
                   const double* F, const double* spectrum, int spectrum_ndim,
                   int spectrum_is_complex, const double* omega, int d, double* out);

/* ---- gradient: derivative of the infidelity with respect to every control amplitude ----------------
 * ff.infidelity_derivative (DESIGN.md section 4.11): out[a, g, h] = dI_a / du_h(g) of the first-order
 * infidelity I_a = trapezoid(S_a F_aa) / (2 pi norm_d) of ffb_infidelity, for a traceless basis
 * (F_aa = sum_k |B_ak|^2), with H_g = sum_i c_coeffs[i,g] c_opers[i].  Inputs as in
 * ffb_control_matrix_from_scratch, plus
 *   c_opers (n_cops,d,d) c128 | c_coeffs (n_cops,G) f64, only read when eigvals is NULL
 *   eigvals, eigvecs, propagators: the pulse's diagonalisation, or all three NULL: diagonalised here
 *   control_matrix (n_nops,n_basis,n_omega) c128 of all noise operators, or NULL: computed here
 *   ctrl_idx (n_ctrl) rows of c_opers to differentiate by | sel_idx (n_sel) rows of n_opers
 *   spectrum f64: spectrum_ndim 1: (n_omega) | 2: (n_sel,n_omega)
 *   n_coeffs_deps (n_nops,n_ctrl,G) f64 d n_coeffs[a,g] / d c_coeffs[ctrl_idx[h],g], or NULL (zero)
 *   out (n_sel,G,n_ctrl) f64.
 * d <= 8.  Deterministic: the sums over frequencies and segments run in a fixed order. */
int ffb_infidelity_derivative(ffb_ctx* ctx, int G, int d, int n_cops, int n_nops, int n_basis,
                              int n_omega, const double* c_opers, const double* c_coeffs,
                              const double* eigvals, const double* eigvecs,
                              const double* propagators, const double* omega, const double* basis,
                              const double* n_opers, const double* n_coeffs, const double* dt,
                              const double* t, const double* control_matrix, int n_ctrl,
                              const int* ctrl_idx, int n_sel, const int* sel_idx,
                              const double* spectrum, int spectrum_ndim,
                              const double* n_coeffs_deps, int norm_d, double* out);

/* ---- f1 (SURVEY 8f rank 1): decay amplitudes ---------------------------------------------------
 * Replaces numeric.calculate_decay_amplitudes (numeric.py:1194-1337) with the integrand of
 * numeric._get_integrand for a control matrix (numeric.py:259-374, einsum '...ko,...o,...lo->...klo'):
 *   Gamma^{(gh)}_{ab,kl} = trapezoid_w Re(conj(B^{(g)}_{ak}) S_{ab} B^{(h)}_{bl}) / (2 pi)
 * B (P,n_nops,n_basis,n_omega) c128 (P = 1: control matrix; P > 1: pulse-correlation control matrix);
 * idx (n_sel) noise-operator indices; spectrum as in ffb_infidelity;
 * out f64 (P,P,n_pairs,n_basis,n_basis), n_pairs = n_sel for spectrum_ndim 1/2 (a == b) and n_sel^2
 * for spectrum_ndim 3.  The integrand (n_basis^2 n_omega values per pair) is never materialised. */
int ffb_decay_amplitudes(ffb_ctx* ctx, int P, int n_nops, int n_sel, const int* idx, int n_basis,
                         int n_omega, const double* B, const double* spectrum, int spectrum_ndim,
                         int spectrum_is_complex, const double* omega, double* out);

/* ---- f2 (SURVEY 8f rank 2): batched concatenation -----------------------------------------------
 * n_seq gate sequences of (up to) L gates each, drawn from a library of n_lib pulses whose control
 * matrices are cached on one frequency grid: what a loop of ff.concatenate(cliffords[row]) followed by
 * ff.infidelity does in examples/randomized_benchmarking.py:70-91, in one call (pulse_sequence.py:1745,
 * :1824-1858 + numeric.py:621-704, :1413-1467, :2318-2320 per sequence).
 *   indices (n_seq,L) int32, entries in [0,n_lib) or < 0 for padding (no gate)
 *   lib_control_matrix (n_lib,n_nops,n_basis,n_omega) c128 | lib_total_phases (n_lib,n_omega) c128
 *   lib_liouville (n_lib,n_basis,n_basis) f64 | lib_propagator (n_lib,d,d) c128 | basis (n_basis,d,d)
 *   spectrum/omega as in ffb_infidelity with all n_nops operators selected (NULL: no infidelity)
 *   tau (n_seq) f64: durations of the sequences, only needed for total_phases
 * Outputs (any may be NULL): total_propagator (n_seq,d,d) c128, total_propagator_liouville
 * (n_seq,n_basis,n_basis) c128, control_matrix (n_seq,n_nops,n_basis,n_omega) c128, filter_function
 * (n_seq,n_nops,n_nops,n_omega) c128, infidelity (n_seq,n_nops) or (n_seq,n_nops,n_nops) f64,
 * total_phases (n_seq,n_omega) c128 = exp(i omega tau) (util.cexp, pulse_sequence.py:1056-1084). */
int ffb_concatenate_many(ffb_ctx* ctx, int n_seq, int L, int n_lib, int d, int n_nops, int n_basis,
                         int n_omega, const int* indices, const double* lib_control_matrix,
                         const double* lib_total_phases, const double* lib_liouville,
                         const double* lib_propagator, const double* basis, const double* spectrum,
                         int spectrum_ndim, int spectrum_is_complex, const double* omega,
                         double* total_propagator, double* total_propagator_liouville,
                         double* control_matrix, double* filter_function, double* infidelity,
                         const double* tau, double* total_phases);

/* ---- a6 with differing noise operators (config 5: QFT from gate pulses) --------------------------
 * Control matrix of a sequence of P pulses that do NOT all carry the same noise operators, as
 * ff.concatenate builds it (pulse_sequence.py:1822-1866: rows of cached control matrices are copied into
 * the atomic stack, rows of operators a pulse does not carry are computed from scratch with the merged
 * sensitivities, :1843-1851; then calculate_control_matrix_from_atomic, :1858, and the filter function,
 * :1866).  The atomic stack is assembled and consumed in device memory: cached rows are uploaded,
 * missing rows are written by the from-scratch kernel, and for the total control matrix only two pulse
 * slots exist (running sum updated in place).
 *   row_of (P,n_nops) int32: row of pulse p's cached control matrix holding merged operator j, -1 = missing
 *   cached[P]: host pointers to (n_cached_p,n_basis,n_omega) c128 (NULL if the pulse has none)
 *   G[P] and eigvals/eigvecs/propagators/dt/t[P]: the pulses' own diagonalisation, shapes as in
 *     ffb_control_matrix_from_scratch (t starts at 0 for every pulse); only read for missing rows
 *   n_coeffs[P] -> (n_nops,G_p) f64 merged noise sensitivities on pulse p's segments
 *   n_opers (n_nops,d,d) c128 merged | basis (n_basis,d,d) c128 | omega (n_omega) f64
 *   phases (P-1,n_omega) c128 cumulative | liouville (P-1,n_basis,n_basis) f64 cumulative
 *   correlations: 0 -> control_matrix (n_nops,n_basis,n_omega); 1 -> (P,n_nops,n_basis,n_omega)
 *   filter_function_kind: 0 none, 1 fidelity, 2 generalized; shape as ffb_filter_function with
 *     P = 1 (total) or P (correlations).  control_matrix may be NULL. */
int ffb_concatenate_pulses(ffb_ctx* ctx, int P, int d, int n_nops, int n_basis, int n_omega,
                           const int* row_of, const double* const* cached, const int* G,
                           const double* const* eigvals, const double* const* eigvecs,
                           const double* const* propagators, const double* const* dt,
                           const double* const* t, const double* const* n_coeffs,
                           const double* n_opers, const double* basis, const double* omega,
                           const double* phases, const double* liouville, int correlations,
                           int filter_function_kind, double* control_matrix,
                           double* filter_function);

/* ---- f3 (SURVEY 8f rank 3): control matrix with cached intermediates -----------------------------
 * cache_intermediates=True of numeric.calculate_control_matrix_from_scratch (numeric.py:828-879): the
 * control matrix plus the arrays of the `intermediates` dict (keys numeric.py:872-878), all c128:
 *   n_opers_transformed (n_nops,G,d,d) | eigvecs_propagated (G,d,d) | basis_transformed (G,n_basis,d,d)
 *   phase_factors (G,n_omega) | first_order_integral (G,n_omega,d,d)
 *   control_matrix_step (G,n_nops,n_basis,n_omega) | control_matrix_step_cumulative (G-1,n_nops,n_basis,n_omega)
 * Inputs as in ffb_control_matrix_from_scratch.  Memory grows with G * n_omega (this is the variant the
 * fused kernel avoids); the call fails with FFB_ENOMEM if the device cannot hold the arrays. */
int ffb_control_matrix_intermediates(ffb_ctx* ctx, int G, int d, int n_nops, int n_basis,
                                     int n_omega, const double* eigvals, const double* eigvecs,
                                     const double* propagators, const double* omega,
                                     const double* basis, const double* n_opers,
                                     const double* n_coeffs, const double* dt, const double* t,
                                     double* out, double* n_opers_transformed,
                                     double* eigvecs_propagated, double* basis_transformed,
                                     double* phase_factors, double* first_order_integral,
                                     double* control_matrix_step,
                                     double* control_matrix_step_cumulative);

/* ---- f4 (SURVEY 8f rank 4): periodic repetition ---------------------------------------------------
 * Replaces numeric.calculate_control_matrix_periodic (numeric.py:884-954):
 *   out(w) = B(w) sum_{g < repeats} (phases(w) L)^g
 * phases (n_omega) c128 | B (n_nops,n_basis,n_omega) c128 | L (n_basis,n_basis) f64 (c128 if
 * l_is_complex) | out (n_nops,n_basis,n_omega) c128.  Binary doubling on the rows of B instead of one
 * linear solve per frequency; valid for every frequency (no invertibility condition). */
int ffb_control_matrix_periodic(ffb_ctx* ctx, int n_nops, int n_basis, int n_omega, int repeats,
                                const double* phases, const double* B, const double* L,
                                int l_is_complex, double* out);

/* ---- a8 helper: Liouville representation --------------------------------------------------------
 * Replaces superoperator.liouville_representation (superoperator.py:51-84):
 * out[n,i,j] = tr(C_i U_n C_j U_n^dagger); U (n,d,d) c128, basis (n_basis,d,d) c128,
 * out (n,n_basis,n_basis) c128 (the Python shell keeps the real part for Hermitian bases). */
int ffb_liouville_representation(ffb_ctx* ctx, int n, int d, int n_basis, const double* U,
                                 const double* basis, double* out);

/* exp(i * x * scale) element-wise (util.cexp, util.py:136-162); x (n) f64 -> out (n) c128. */
int ffb_cexp(ffb_ctx* ctx, int n, const double* x, double scale, double* out);
/* exp(i x) - 1 = -2 sin^2(x/2) + i sin(x) element-wise (util.cexpm1, util.py:165-182). */
int ffb_cexpm1(ffb_ctx* ctx, int n, const double* x, double* out);

/* ---- fused pulse pipeline ------------------------------------------------------------------------
 * What PulseSequence.get_filter_function (pulse_sequence.py:691-805) does on a cold cache, in one
 * call: the inputs are packed into ONE upload; diagonalize -> control matrix -> fidelity filter
 * function (-> infidelity if spectrum != NULL), plus the two by-products cache_control_matrix keeps
 * (pulse_sequence.py:674-677): total_phases = exp(i omega tau) (n_omega) c128 and the Liouville
 * representation of the total propagator (n_basis,n_basis) c128.  The eigensystem, propagators and
 * by-products are downloaded on a second stream while the control-matrix kernel runs, the control
 * matrix while the filter function and the integral are computed.  Any output pointer may be NULL
 * to skip it.  t may be NULL: then t = [0, cumsum(dt)] (sequential sum, as np.cumsum).  spectrum as
 * in ffb_infidelity with n_sel = n_nops, idx = 0..n_nops-1.
 * If all result pointers lie in ONE block obtained from ffb_host_alloc, results that are less than 256
 * bytes apart there are downloaded in one copy; the bytes between them are treated as padding and
 * overwritten (the Python shell carves its result arrays out of one such block, _lib.empty_many). */
int ffb_pulse_filter_function(ffb_ctx* ctx, int G, int d, int n_cops, int n_nops, int n_basis,
                              int n_omega, const double* c_opers, const double* c_coeffs,
                              const double* n_opers, const double* n_coeffs, const double* dt,
                              const double* t, const double* basis, const double* omega,
                              const double* spectrum, int spectrum_ndim, int spectrum_is_complex,
                              double* eigvals, double* eigvecs, double* propagators,
                              double* control_matrix, double* filter_function, double* infidelity,
                              double* total_phases, double* total_propagator_liouville);

/* ---- device-resident variants (pointers are device pointers; asynchronous on the stream) -------- */
int ffb_dev_diagonalize(ffb_ctx* ctx, int G, int d, int n_cops, const double* c_opers,
                        const double* c_coeffs, const double* dt, double* eigvals, double* eigvecs,
                        double* propagators);
int ffb_dev_control_matrix_from_scratch(ffb_ctx* ctx, int G, int d, int n_nops, int n_basis,
                                        int n_omega, const double* eigvals, const double* eigvecs,
                                        const double* propagators, const double* omega,
                                        const double* basis, const double* n_opers,
                                        const double* n_coeffs, const double* dt, const double* t,
                                        int herm_flags, double* out);
int ffb_dev_filter_function(ffb_ctx* ctx, int P, int n_nops, int n_basis, int n_omega,
                            const double* B, int generalized, double* F);
int ffb_dev_control_matrix_from_atomic(ffb_ctx* ctx, int P, int n_nops, int n_basis, int n_omega,
                                       const double* phases, const double* B_atomic,
                                       const double* Q_liouville, int q_is_complex,
                                       int correlations, double* out);
int ffb_dev_infidelity(ffb_ctx* ctx, int n_lead, int n_nops, int n_sel, const int* idx,
                       int n_omega, const double* F, const double* spectrum, int spectrum_ndim,
                       int spectrum_is_complex, const double* omega, int d, double* out);
int ffb_dev_decay_amplitudes(ffb_ctx* ctx, int P, int n_nops, int n_sel, const int* idx,
                             int n_basis, int n_omega, const double* B, const double* spectrum,
                             int spectrum_ndim, int spectrum_is_complex, const double* omega,
                             double* out);
/* herm_flags for ffb_dev_control_matrix_from_scratch: bit 0 = all noise operators exactly
 * Hermitian, bit 1 = all basis elements exactly Hermitian, bit 2 = basis element 0 is exactly a real
 * multiple of the identity (Basis.pauli, Basis.ggm: its rows of the control matrix only have the
 * level-diagonal term, sum_g s_j tr(B_j)/sqrt(d) e^{i w t} I(w); the host entry points check all
 * three themselves; pass 0 if unknown -- always correct, only more work). */
#define FFB_HERM_NOPERS 1
#define FFB_HERM_BASIS 2
#define FFB_BASIS_IDENTITY0 4

/* ---- e: peer group of the GPUs of one node (SURVEY.md 8e; nothing in the reference) ---------------
 * One process per GPU.  The frequency axis is sharded by the caller (every output element depends on
 * one frequency only); the exchanges of the path run over NVLink peer memory inside this library's own
 * kernels: the sum of the per-noise-operator partial integrals is the EPILOGUE of the infidelity
 * kernels (the thread that holds a finished partial integral stores it into all peers' windows and
 * adds up what the peers stored, in rank order -- identical bits on every rank), and the gather of
 * F(omega) column blocks stores every block straight into all peers' windows.
 * Set-up: every rank calls ffb_comm_create (allocates its exchange window, returns a 64-byte CUDA IPC
 * handle), the host program all-gathers the handles by any means (distributed.py: torch.distributed)
 * and passes the concatenation (world x 64 bytes, rank order) to ffb_comm_connect.  All ranks must
 * issue the same sequence of collectives.  A peer that does not arrive within FFB_PEER_TIMEOUT_MS
 * (default 20000) makes the call fail with FFB_ECUDA instead of hanging the GPU. */
#define FFB_COMM_HANDLE_BYTES 64
int ffb_comm_create(ffb_ctx* ctx, int rank, int world, void* handle_out);
int ffb_comm_connect(ffb_ctx* ctx, const void* handles);
int ffb_comm_destroy(ffb_ctx* ctx);
int ffb_comm_info(const ffb_ctx* ctx, int* rank, int* world, size_t* data_window_bytes);
/* enable != 0: every infidelity integral this context computes (ffb_infidelity, ffb_dev_infidelity,
 * ffb_pulse_filter_function) is summed over the ranks before it is stored: numeric.infidelity
 * (numeric.py:2318-2320) on a frequency shard then returns the integral over the whole grid. */
int ffb_comm_reduce_infidelity(ffb_ctx* ctx, int enable);
/* In-place sum over the ranks of n doubles (host / device pointer). */
int ffb_allreduce_sum(ffb_ctx* ctx, double* data, int n);
int ffb_dev_allreduce_sum(ffb_ctx* ctx, double* data, int n);
/* Symmetric data window for ffb_allgather_columns: (re)allocate `bytes` on this rank and return its
 * handle; the ranks must be synchronised by the caller around the call (nobody may still use the old
 * window), then exchange the handles and call ffb_comm_data_connect. */
int ffb_comm_data_window(ffb_ctx* ctx, size_t bytes, void* handle_out);
int ffb_comm_data_connect(ffb_ctx* ctx, const void* handles);
/* All-gather along the last (frequency) axis: this rank holds `local` (rows, counts[rank]) c128, on
 * return `out` (rows, sum(counts)) c128 holds the blocks of all ranks side by side, on every rank. */
int ffb_allgather_columns(ffb_ctx* ctx, int rows, const int* counts, const double* local,
                          double* out);

/* Raw device memory for the callers of ffb_dev_* that do not bring their own (e.g. torch). */
int ffb_dev_alloc(ffb_ctx* ctx, size_t bytes, void** ptr);
int ffb_dev_free(ffb_ctx* ctx, void* ptr);
int ffb_memcpy_h2d(ffb_ctx* ctx, void* dst_dev, const void* src_host, size_t bytes);
int ffb_memcpy_d2h(ffb_ctx* ctx, void* dst_host, const void* src_dev, size_t bytes);

/* Page-locked host memory from a caching pool.  Result arrays allocated here make the device->host
 * copies of the host-pointer entry points run at full PCIe speed (the library detects pinned
 * destinations by itself); pageable buffers work too, just slower.  ffb_host_free returns the block to
 * the pool. */
int ffb_host_alloc(ffb_ctx* ctx, size_t bytes, void** ptr);
int ffb_host_free(ffb_ctx* ctx, void* ptr);

/* ---- device-resident shadows of cached arrays (SURVEY.md 8b; the reference's cache is
 * pulse_sequence.py:262-271, :1158-1245) ----------------------------------------------------------------
 * ffb_shadow_enable_next(ctx, 1) before ffb_pulse_filter_function, ffb_control_matrix_from_scratch,
 * ffb_concatenate_pulses or a single-sequence ffb_concatenate_many: the device copy of the results that
 * land in page-locked blocks of ffb_host_alloc is kept after the call, keyed by the host address range it
 * mirrors.  Any later host-pointer call that is handed a pointer into such a range (ffb_infidelity,
 * ffb_decay_amplitudes, ffb_filter_function, ffb_concatenate_pulses, ...) reads the device copy instead
 * of uploading the bytes.  A shadow ends when its host block is returned (ffb_host_free), when a call
 * writes into the range, by ffb_shadow_drop, or -- oldest first -- when all shadows together exceed a
 * quarter of the device memory (FFB_SHADOW_BYTES).  The caller must not modify a shadowed host array
 * (ffb_shadow_query tells; the Python shell marks such arrays read-only). */
int ffb_shadow_enable_next(ffb_ctx* ctx, int enable);
/* Mirror an INPUT array the caller will pass again and again (the stacked control matrices of a gate
 * library): uploaded once, then found by address like a result shadow.  The array must lie in a block of
 * ffb_host_alloc and be at least 64 KiB, otherwise nothing is kept (and nothing breaks). */
int ffb_shadow_upload(ffb_ctx* ctx, const void* host, size_t bytes);
int ffb_shadow_query(ffb_ctx* ctx, const void* host, size_t bytes);
int ffb_shadow_drop(ffb_ctx* ctx, const void* host, size_t bytes);
int ffb_shadow_stats(ffb_ctx* ctx, int* count, size_t* bytes, int64_t* hits, size_t* hit_bytes);

/* Kernel-level timing of the control-matrix stage: total duration (ms) and number of the timed launches,
 * recorded with CUDA events on the launching stream since the last reset.  A timed launch is the main
 * kernel, or on the banded route the plan, main and evaluation kernels of a frequency block together. */
int ffb_kernel_timing_enable(ffb_ctx* ctx, int enable);
int ffb_kernel_timing_read(ffb_ctx* ctx, double* total_ms, int64_t* launches, int reset);

/* Record of the control-matrix dispatch: every control-matrix computation of a context (any entry point
 * that computes one from scratch) appends one record per block of frequencies, naming the kernel
 * instance it launched and the quantities that chose it.  Names are spelled as the demangled symbol
 * without namespace and argument list, e.g. "ctrlmat_static_kernel<12, 4, 6, 2, true>".  For the DFMA
 * kernels a "pass" is one segment, for the int8 kernel one stage of four segments; fields that do not
 * apply to a kernel family are 0.  ffb_dispatch_log copies up to `capacity` records, oldest first, to
 * `out` (may be NULL), clears the log and returns the number copied.  The log holds the last
 * FFB_DISPATCH_LOG_MAX records.
 * ffb_diag_dispatch_log does the same for a log of its own, with one record per diagonalisation
 * (ffb_diagonalize and the pulse entry points that diagonalise): `kernel` is the diagonaliser instance
 * ("scan_block_kernel<4, 128>" when the diagonalisation is fused into the block scan,
 * "diag_small_kernel<4>", "diag_kernel"), `prologue` the scan kernel instances it launched, each once, in
 * order of first launch, `n_pass` = G segments, `passes_per_chunk` the segments per scan block or chunk
 * (NT, or L for the generic scan) and `S` the number of scan levels (the block scan runs once per level);
 * the other fields are 0. */
#define FFB_DISPATCH_LOG_MAX 256
typedef struct {
  char kernel[64];       /* the omega-dependent kernel */
  char prologue[96];     /* the omega-independent kernels before it, joined by '+' */
  int S;                 /* chunks of the segment axis (partials summed by finalize_kernel) */
  int passes_per_chunk;  /* passes per chunk (DFMA: segs_per_cta; int8: stages_per_chunk) */
  int n_pass;
  int n_sp;              /* pieces a pass is staged in */
  int pps;               /* passes per stage */
  int transposed;        /* level pairs of one segment in the K slots */
  int n_rb;              /* row blocks */
  int n_wtiles;          /* frequency tiles of the block */
  int ctas_by_regs;      /* resident CTAs per SM the registers allow (sets the stage budget) */
  int block, n_blocks;   /* this frequency block and the number of blocks of the call */
  int n_omega;           /* frequencies in this block */
  int route;             /* 0: every frequency evaluated directly; 1: banded (Chebyshev interpolation of
                            per-chunk partial sums on dense bands, DESIGN 4.1.1) */
  int chunk_segs;        /* banded: segments per chunk L (S = ceil(G / L) chunks); else 0 */
  int n_bands;           /* banded: bands interpolated in this block; else 0 */
  int n_proxies;         /* banded: proxy frequencies evaluated for them (BAND_P per band); else 0 */
} ffb_dispatch_record;
int ffb_dispatch_log(ffb_ctx* ctx, ffb_dispatch_record* out, int capacity);
int ffb_diag_dispatch_log(ffb_ctx* ctx, ffb_dispatch_record* out, int capacity);

#ifdef __cplusplus
}
#endif
#endif /* FFB200_H */
