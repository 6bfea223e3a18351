#!/usr/bin/env python
"""Benchmark of the hot path: from-scratch control matrix -> filter function -> infidelity.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload d4|c2|c3] [--extra c2,c3|none]
                    [--impl reference] [--dump-outputs DIR]

A *step* is one pass of the whole path over one synthetic pulse (SURVEY.md 8d): diagonalise the
G-segment control Hamiltonian, build the first-order control matrix on n_omega frequencies, reduce it
to the fidelity filter function and integrate against the noise spectrum.  The metric is
BASELINE.json's: control-matrix throughput in segment*frequency pairs per second (fp64).

  headline : the north_star target shape ``d4`` (d = 4, G = 1e4 segments, n_omega = 1e4 frequencies, 6
          noise operators; the loop it replaces is numeric.py:846-869 of the reference).  BASELINE
          configs 2 and 3 are measured in the same run and reported under ``workloads``.
  value : whole-job seg*omega/s with all inputs resident in HBM (DevicePulse, ffb_dev_* entry points),
          device-timed with CUDA events, L2 flushed between steps, max over ranks.
  e2e   : the same metric through the public NumPy API (ff.infidelity on a cold PulseSequence; with
          N > 1 filter_functions_b200.distributed.infidelity on the GLOBAL grid), host buffers in, host
          arrays out, copies inside the timed region.
  N > 1 : STRONG scaling -- the global frequency grid is fixed and sharded over the ranks (contiguous
          blocks of trapezoid intervals), the per-segment operands are replicated, and the partial
          integrals are summed over the ranks in the epilogue of the infidelity kernel over NVLink peer
          memory (csrc/ffb_peer.cuh); no other exchange.
  --impl reference : the UNMODIFIED reference (baseline/_ref, staged by baseline/install_reference.py)
          through its own public API on the host cores, on a bounded sample (first G_cpu segments of the
          same pulse, all frequencies; the reference's cost is exactly linear in G) -- the printed
          ms_per_step is EXTRAPOLATED to the full pulse.  Falls back to the NumPy port in oracle/ if
          the reference has not been staged.
  --dump-outputs DIR : after the timed steps, write what the last timed step of the headline workload
          computed (device path: eigenvalues, eigenvectors, propagators, control matrix, filter function,
          infidelities; public API: its infidelities) as DIR/<name>.npy, so that the outputs of two builds
          can be compared on identical (seeded) inputs.  With N > 1 the frequency-resolved arrays are rank
          0's block of the grid.
"""
import argparse
import json
import os
import sys
import threading
import time

if '--impl' in sys.argv and 'reference' in sys.argv:
    # torchrun pins OMP_NUM_THREADS=1 for its workers; the reference arm is the reference's CPU path
    # on ALL host cores, so undo that before NumPy/OpenBLAS load.
    for _var in ('OMP_NUM_THREADS', 'OPENBLAS_NUM_THREADS', 'MKL_NUM_THREADS'):
        os.environ[_var] = str(os.cpu_count() or 1)

# The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version line to
# stdout at init, nvcc output of a first build, ...): keep a private handle on the real stdout for the
# result line and point file descriptor 1 at stderr for everything else, native code included.
sys.stdout.flush()
RESULT_OUT = os.fdopen(os.dup(1), 'w')
os.dup2(2, 1)

import numpy as np  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import workloads  # noqa: E402

METRIC = 'control-matrix throughput (segments*omega/s, fp64), control matrix + filter function + infidelity'
UNIT = 'seg*omega/s'
HEADLINE = 'd4'


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=30)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--workload', default=HEADLINE, choices=['c2', 'c3', 'd4'])
    ap.add_argument('--extra', default=None,
                    help="comma-separated workloads reported under 'workloads' (default: the other two "
                         "of c2, c3, d4; 'none' to skip)")
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--cpu-seconds', type=float, default=12.0,
                    help='target duration of the bounded CPU-baseline sample')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-int8', action='store_true',
                    help="skip the extra 'd4_int8' line (opt-in int8 tensor-core kernel)")
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the outputs of the last timed step of the headline workload as '
                         'DIR/<name>.npy (float64, complex arrays with a trailing (real, imag) axis, at '
                         'most 64 MB in all: larger frequency-resolved arrays keep a fixed, seeded sample '
                         'of frequencies)')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    if args.dump_outputs is not None and args.impl != 'b200':
        ap.error('--dump-outputs writes the outputs of the GPU path (--impl b200)')
    return args


def workload_config(wl, n_gpus, n_local):
    return {
        'workload': f'{wl.name}: {wl.description}',
        'G': wl.G, 'd': wl.d, 'n_nops': len(wl.n_opers), 'n_basis': len(wl.basis),
        'n_omega_total': len(wl.omega), 'n_omega_per_gpu': n_local,
        'parallelism': (f'omega-sharded x{n_gpus} (fixed global grid, one halo abscissa per block)'
                        if n_gpus > 1 else 'single GPU'),
        'l2': 'flushed between timed steps (256 MiB device write)',
    }


# ------------------------------------------------------------------------------------------------
# CPU leg: the reference itself (baseline/_ref) or, if it is not staged, the oracle port
# ------------------------------------------------------------------------------------------------
def _load_reference():
    """The unmodified reference package from baseline/_ref (opt_einsum / sparse: oracle/shim)."""
    sys.path.insert(0, os.path.join(ROOT, 'baseline'))
    try:
        import install_reference
        state = install_reference.install(verbose=False)
    except Exception:
        state = 'unavailable'
    if state == 'unavailable':
        return None
    sys.path.insert(0, os.path.join(ROOT, 'oracle', 'shim'))
    sys.path.insert(0, os.path.join(ROOT, 'baseline', '_ref'))
    import filter_functions
    if not os.path.abspath(filter_functions.__file__).startswith(os.path.join(ROOT, 'baseline', '_ref')):
        return None
    return filter_functions


def _blas_threads():
    try:
        from threadpoolctl import threadpool_info
        return max([p.get('num_threads', 1) for p in threadpool_info()] or [1])
    except Exception:
        return os.cpu_count() or 1


def cpu_sample(wl, seconds):
    """Time the reference on a bounded sample: the first G_cpu segments of the same pulse on all
    frequencies, through ff.infidelity on a cold PulseSequence (diagonalisation, control matrix,
    filter function, integral).  Returns a dict with the throughput and what the sample was."""
    ref = _load_reference()
    n_omega = len(wl.omega)
    if ref is not None:
        kind = 'reference'
        basis = ref.Basis.pauli(int(np.log2(wl.d)))

        def run(G_cpu):
            pulse = ref.PulseSequence(
                [[op, c[:G_cpu], i] for op, c, i in zip(wl.c_opers, wl.c_coeffs, wl.c_ids)],
                [[op, c[:G_cpu], i] for op, c, i in zip(wl.n_opers, wl.n_coeffs, wl.n_ids)],
                wl.dt[:G_cpu], basis)
            t0 = time.perf_counter()
            ref.infidelity(pulse, wl.spectrum, wl.omega)
            return time.perf_counter() - t0
        what = 'unmodified reference (baseline/_ref), ff.infidelity on a cold PulseSequence'
    else:
        kind = 'port'
        sys.path.insert(0, os.path.join(ROOT, 'oracle'))
        import ff_oracle as oracle

        def run(G_cpu):
            t0 = time.perf_counter()
            H = oracle.hamiltonian_from_coeffs(wl.c_opers, wl.c_coeffs[:, :G_cpu])
            ev, V, Q = oracle.diagonalize(H, wl.dt[:G_cpu])
            B = oracle.control_matrix_from_scratch(ev, V, Q, wl.omega, wl.basis, wl.n_opers,
                                                   wl.n_coeffs[:, :G_cpu], wl.dt[:G_cpu])
            F = oracle.filter_function(B)
            oracle.infidelity_from_filter_function(F, wl.spectrum, wl.omega, wl.d)
            return time.perf_counter() - t0
        what = 'NumPy port of the reference algorithm (oracle/ff_oracle.py)'
    n_cal = 8
    per_seg = run(n_cal)/n_cal
    G_cpu = int(max(16, min(wl.G, seconds/per_seg)))
    elapsed = run(G_cpu)
    threads = _blas_threads()
    return {
        'value': G_cpu*n_omega/elapsed, 'unit': UNIT, 'cores': threads, 'kind': kind,
        'sample': (f'{what}: first {G_cpu} of {wl.G} segments x {n_omega} frequencies in '
                   f'{elapsed:.1f} s, NumPy/OpenBLAS with {threads} BLAS threads on '
                   f'{os.cpu_count()} host cores; cost is linear in G (numeric.py:846)'),
        'sample_segments': G_cpu, 'sample_seconds': elapsed,
    }


def run_reference(args):
    rank = int(os.environ.get('RANK', 0))
    if rank != 0:
        return
    wl = workloads.get(args.workload)
    per_step = max(1.0, min(args.cpu_seconds, 150.0/max(1, args.steps + args.warmup)))
    vals, last = [], None
    for i in range(args.warmup + args.steps):
        last = cpu_sample(wl, per_step)
        if i >= args.warmup:
            vals.append(last['value'])
    value = float(np.mean(vals)) if vals else 0.0
    cpu = dict(last, value=value)
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': 1e3*wl.G*len(wl.omega)/value if value else None,
        'ms_per_step_note': (f'EXTRAPOLATED to the full pulse of {wl.G} segments from timed samples '
                             f'of {last["sample_segments"]} segments (linear in G); each timed step '
                             f'really took {1e3*last["sample_seconds"]:.0f} ms'),
        'extrapolated': True, 'sample_segments': last['sample_segments'],
        'sample_ms_per_step': 1e3*last['sample_seconds'],
        'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f64',
        'data': 'synthetic', 'config': workload_config(wl, args.gpus, len(wl.omega)),
        'cpu_baseline': cpu,
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), file=RESULT_OUT, flush=True)


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    REASONS = {0x8: 'hw_slowdown', 0x40: 'hw_thermal_slowdown', 0x20: 'sw_thermal_slowdown',
               0x4: 'sw_power_cap', 0x80: 'hw_power_brake_slowdown'}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self.stop_flag = threading.Event()
        self.active = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        while not self.stop_flag.is_set():
            if self.active.is_set():
                try:
                    self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                    mask = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                    for bit, name in self.REASONS.items():
                        if mask & bit:
                            self.reasons.add(name)
                except Exception:
                    pass
            time.sleep(0.002)

    def result(self):
        if not self.samples:
            return {'sm_mhz': None, 'sm_max_mhz': self.max_mhz, 'reasons': [],
                    'note': 'NVML unavailable'}
        return {'sm_mhz': float(np.median(self.samples)), 'sm_max_mhz': self.max_mhz,
                'reasons': sorted(self.reasons), 'samples': len(self.samples)}


# ------------------------------------------------------------------------------------------------
# GPU leg
# ------------------------------------------------------------------------------------------------
def golden_parity(name, order, infid):
    """Infidelities of the whole grid against the reference's own result for this workload
    (tests/golden/workload_full_<name>.npz, computed once by the unmodified reference)."""
    path = os.path.join(ROOT, 'tests', 'golden', f'workload_full_{name}.npz')
    if not os.path.exists(path):
        return None
    want = np.load(path)['infidelity']
    got = np.asarray(infid).ravel()
    if got.shape != want.shape:
        return None
    return float(np.abs(got - want).max()/np.abs(want).max())


def kernel_model(wl, n_omega_local, kernel_ms, peak, int8=False):
    """Which control-matrix kernel instance ran and how many multiply-add flops it really issued
    (Hermitian-pair formulation, csrc/ffb_ctrlmat.cu header)."""
    G, d = wl.G, wl.d
    n_nops, n_basis = len(wl.n_opers), len(wl.basis)
    rows = n_nops*n_basis
    if int8:
        # csrc/ffb_ctrlmat_i8.cu: per seg*omega 15 digit-plane products of (re | im) x 96 rows x 16 K entries
        ops = 2*2*15*96*16*G*n_omega_local/(kernel_ms*1e-3)*1e-12
        return ('ctrlmat_i8_kernel',
                'int8 tensor cores (tcgen05.mma.kind::i8, int32 accumulators in TMEM; 15 int8 digit-plane '
                'products per FP64 product) fed by an FP64 operand generator (~260 FP64 instructions per '
                'seg*omega); executed_tflops counts the int8 operations (TOP/s), executed_frac is against '
                'the NOMINAL dense int8 peak of 4500 TOP/s', ops, ops/4500.0*peak)
    use_dfma = rows <= 16 and 2 <= d <= 3 and os.environ.get('FFB_CTRLMAT_DFMA', '1') != '0'
    n_pairs = d*(d - 1)//2
    if use_dfma:
        rows_pad = -(-rows//4)*4
        kernel = 'ctrlmat_dfma_kernel'
        pipe = ('fp64 DFMA (thread per frequency; 64 lanes/clk/SM, the pipe DMMA shares); the '
                'operand generator adds ~52 FP64 instructions per seg*omega that are not counted in '
                'executed_tflops')
        # rows of an identity basis element carry no level-pair terms (csrc/ffb_ctrlmat.cu)
        ident0 = bool((wl.basis[0] == wl.basis[0][0, 0].real*np.eye(d)).all())
        split = (ident0 and os.environ.get('FFB_DFMA_SPLIT_IDENTITY', '1') != '0'
                 and ((d == 2 and n_basis == 4 and 2 <= n_nops <= 4)
                      or (d == 3 and n_basis == 9 and n_nops == 1)))
        pair_rows = n_nops*(n_basis - 1) if split else rows_pad
    else:
        rows_pad = -(-rows//8)*8
        tiles = rows_pad//8
        n_rb = -(-tiles//12)
        mt = next(a for a in (1, 2, 3, 4, 5, 6, 7, 8, 10, 12) if a >= -(-tiles//n_rb))
        static = (d == 4 and mt in (6, 8, 10, 12) and G >= 4
                  and os.environ.get('FFB_CTRLMAT_STATIC', '1') != '0')
        kernel = 'ctrlmat_static_kernel' if static else 'ctrlmat_main_kernel'
        rows_pad = n_rb*mt*8
        pipe = 'fp64 (DMMA.8x8x4; shares the 64 lane/clk/SM FP64 pipe with DFMA)'
        pair_rows = rows_pad
        # two qubits, six noise operators, identity basis element: the six rows (j, 0) take no part in the
        # pair units (88 rows through DMMA, 2 through the DFMA side path; csrc/ffb_ctrlmat.cu, SPLIT)
        ident0 = bool((wl.basis[0] == wl.basis[0][0, 0].real*np.eye(d)).all())
        if (static and d == 4 and n_nops == 6 and n_basis == 16 and ident0 and mt == 12 and n_rb == 1
                and os.environ.get('FFB_CTRLMAT_SPLIT_IDENTITY', '1') != '0'):
            kernel = 'ctrlmat_static_kernel (identity-row split)'
            pair_rows = n_nops*(n_basis - 1)
    # real multiply-adds per seg*omega: 2 per row for the diagonal unit, 4 per row and level pair
    executed = (2*rows_pad + 4*n_pairs*pair_rows)*2*G*n_omega_local/(kernel_ms*1e-3)*1e-12
    return kernel, pipe, executed, executed


def measure(name, steps, warmup, env, int8=False, dump=False):
    """One workload on this rank's GPU: device-resident value, e2e through the public API, roofline of
    the control-matrix kernel.  Collective over the ranks (every rank calls it with the same name).
    ``int8``: with the opt-in fixed-point control-matrix kernel on the int8 tensor cores
    (FFB_CTRLMAT_INT8=1, d = 4 only).  ``dump``: the result also holds, under 'outputs', host copies
    of what the last timed step computed."""
    if int8:
        old = os.environ.get('FFB_CTRLMAT_INT8')
        os.environ['FFB_CTRLMAT_INT8'] = '1'
        try:
            return _measure(name, steps, warmup, env, True, dump)
        finally:
            if old is None:
                os.environ.pop('FFB_CTRLMAT_INT8', None)
            else:
                os.environ['FFB_CTRLMAT_INT8'] = old
    return _measure(name, steps, warmup, env, os.environ.get('FFB_CTRLMAT_INT8', '0') not in ('', '0'),
                    dump)


DUMP_BYTES = 64_000_000
FREQUENCY_RESOLVED = ('control_matrix', 'filter_function')


def dump_outputs(directory, outputs):
    """Write ``outputs`` (name -> array) as ``directory/<name>.npy`` in float64, a complex array with a
    trailing axis (real, imag).  If the files would exceed DUMP_BYTES, the frequency-resolved arrays keep
    the same fixed, seeded sample of their frequencies (last axis), identical from run to run."""
    n_omega = outputs['control_matrix'].shape[-1]
    budget = DUMP_BYTES - 1024*len(outputs)     # room for the .npy headers
    total = sum(a.nbytes for a in outputs.values())
    if total > budget:
        per_omega = sum(outputs[k].nbytes for k in FREQUENCY_RESOLVED)//n_omega
        n_keep = (budget - (total - per_omega*n_omega))//per_omega
        if n_keep < 1:
            raise SystemExit(f'--dump-outputs: the arrays that do not depend on frequency alone exceed '
                             f'{DUMP_BYTES} bytes')
        keep =np.sort(np.random.default_rng(0).choice(n_omega, n_keep, replace=False))
        outputs = {k: a[..., keep] if k in FREQUENCY_RESOLVED else a for k, a in outputs.items()}
    os.makedirs(directory, exist_ok=True)
    for name, a in outputs.items():
        if np.iscomplexobj(a):
            a = np.stack([a.real, a.imag], axis=-1)
        np.save(os.path.join(directory, f'{name}.npy'), np.ascontiguousarray(a, dtype=np.float64))


def control_matrix_parity(name, B):
    """Worst normalised deviation (per noise operator, scale = max |B| over the whole grid) of the control
    matrix from the reference's own result on the frequencies the full-size fixture holds."""
    path = os.path.join(ROOT, 'tests', 'golden', f'workload_full_{name}.npz')
    if not os.path.exists(path):
        return None
    g = np.load(path)
    pick = g['pick']
    return float(max(np.abs(B[j][:, pick] - g['control_matrix'][j]).max()/g['scale'][j]
                     for j in range(len(B))))


def _measure(name, steps, warmup, env, int8, dump):
    import ctypes

    import torch
    import torch.distributed as dist
    ff, ffd, _lib, DevicePulse = env['ff'], env['ffd'], env['_lib'], env['DevicePulse']
    world, rank, local_rank, peers = env['world'], env['rank'], env['local_rank'], env['peers']
    L = _lib.lib()
    wl = workloads.get(name)
    n_total = len(wl.omega)
    start, stop = ffd.frequency_shard(n_total, rank, world)
    local = wl.with_omega(wl.omega[start:stop], wl.spectrum[..., start:stop])
    G, n_local = wl.G, stop - start

    dev = DevicePulse(local.c_opers, local.c_coeffs, local.n_opers, local.n_coeffs, local.dt,
                      local.basis, local.omega, local.spectrum, device=local_rank)
    ctx = dev.ctx
    stream = torch.cuda.current_stream()
    dev.bind_stream()
    total = torch.zeros_like(dev.infidelity)
    if peers is not None:   # the sum over the ranks is the epilogue of the infidelity kernel
        _lib.check(ctx, L.ffb_comm_reduce_infidelity(ctx, 1))

    def step():
        dev.step()
        if world > 1 and peers is None:     # no peer-memory path: NCCL on the same stream
            total.copy_(dev.infidelity)
            dist.all_reduce(total)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(3, warmup)):
        step()
    barrier()

    # ---- device-resident timing -------------------------------------------------------------------
    _lib.check(ctx, L.ffb_kernel_timing_enable(ctx, 1))
    _lib.check(ctx, L.ffb_kernel_timing_read(ctx, None, None, 1))
    launches0 = L.ffb_launch_count(ctx)
    events = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
              for _ in range(steps)]
    barrier()
    env['sampler'].active.set()
    for e0, e1 in events:
        env['flush'].zero_()
        e0.record(stream)
        step()
        e1.record(stream)
    barrier()
    env['sampler'].active.clear()
    launches = L.ffb_launch_count(ctx) - launches0
    k_ms, k_n = ctypes.c_double(), ctypes.c_int64()
    _lib.check(ctx, L.ffb_kernel_timing_read(ctx, ctypes.byref(k_ms), ctypes.byref(k_n), 1))
    _lib.check(ctx, L.ffb_kernel_timing_enable(ctx, 0))
    dev_ms = sum(e0.elapsed_time(e1) for e0, e1 in events)
    dev_inf = (total if (world > 1 and peers is None) else dev.infidelity).cpu().numpy()
    outputs = None
    if dump:    # what a caller of DevicePulse.step() holds after the last timed step
        outputs = {k: getattr(dev, k).cpu().numpy() for k in
                   ('eigvals', 'eigvecs', 'propagators', 'control_matrix', 'filter_function')}
        outputs['infidelity'] = dev_inf
    if peers is not None:
        _lib.check(ctx, L.ffb_comm_reduce_infidelity(ctx, 0))

    # ---- end to end through the public API ----------------------------------------------------------
    _lib.check(ctx, L.ffb_set_stream(ctx, None, 0))
    pulse = ff.PulseSequence(
        [[op, c, i] for op, c, i in zip(wl.c_opers, wl.c_coeffs, wl.c_ids)],
        [[op, c, i] for op, c, i in zip(wl.n_opers, wl.n_coeffs, wl.n_ids)],
        wl.dt, ff.Basis(wl.basis, btype='Pauli'))

    def e2e_step():
        # the user-facing call takes the GLOBAL grid; with N > 1 distributed.infidelity shards it
        pulse.cleanup('all')
        return ffd.infidelity(pulse, wl.spectrum, wl.omega)

    for _ in range(3):
        infid_e2e = e2e_step()
    barrier()
    env['sampler'].active.set()
    t0 = time.perf_counter()
    for _ in range(steps):
        infid_e2e = e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0
    env['sampler'].active.clear()

    d, n_cops, n_nops, n_basis = wl.d, len(wl.c_opers), len(wl.n_opers), len(wl.basis)
    # inputs of the fused pipeline (ffb_pulse_filter_function): operators, coefficients, dt, t, basis,
    # omega, spectrum -- one packed upload per step and rank
    h2d = (16*(n_cops + n_nops + n_basis)*d*d + 8*(n_cops + n_nops)*G + 8*G + 8*(G + 1)
           + 8*n_local + local.spectrum.nbytes)
    d2h = (8*G*d + 16*G*d*d + 16*(G + 1)*d*d + 16*n_nops*n_basis*n_local
           + 16*n_nops*n_nops*n_local + 16*n_basis*n_basis + 16*n_local + 8*n_nops)

    # ---- max over ranks ------------------------------------------------------------------------------
    times = torch.tensor([dev_ms, e2e_s*1e3, k_ms.value, h2d, d2h], dtype=torch.float64, device='cuda')
    if world > 1:
        sums = times.clone()
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
        dist.all_reduce(sums, op=dist.ReduceOp.SUM)
        h2d, d2h = sums[3].item(), sums[4].item()
    dev_ms_max, e2e_ms_max, k_ms_max = times.tolist()[:3]

    units_total = G*n_total            # seg*omega pairs of the whole job per step (halo not counted)
    value = units_total*steps/(dev_ms_max*1e-3)
    e2e_value = units_total*steps/(e2e_ms_max*1e-3)

    # ---- parity of what was timed ----------------------------------------------------------------------
    order = np.argsort(wl.n_ids)           # PulseSequence sorts operators by identifier
    dev_inf = dev_inf[order]
    api = np.asarray(infid_e2e).ravel()
    if dump:
        outputs['e2e_infidelity'] = np.asarray(infid_e2e)
    parity = {'device_vs_api': float(np.abs(dev_inf - api).max()/np.abs(api).max()),
              'vs_reference_fixture': golden_parity(name, order, api),
              'tolerance': 1e-10}
    if world == 1:   # the control matrix the last timed call cached on the pulse
        parity['control_matrix_vs_reference_fixture'] = control_matrix_parity(
            name, pulse.get_control_matrix(wl.omega))
    if world > 1:
        # rank 0 evaluates the SAME global grid on its own GPU alone, outside the timed region
        if rank == 0:
            pulse.cleanup('all')
            single = np.asarray(ff.infidelity(pulse, wl.spectrum, wl.omega)).ravel()
            parity['sharded_vs_single_gpu'] = float(np.abs(api - single).max()/np.abs(single).max())
        dist.barrier()

    # ---- roofline of the dominant kernel ---------------------------------------------------------------
    peak = env['peak']
    kernel_ms = k_ms_max/max(1, k_n.value)
    W = wl.flops_per_seg_omega
    n_local_max = -(-(n_total - 1)//world) + 1 if world > 1 else n_total
    achieved = W*G*n_local_max/(kernel_ms*1e-3)*1e-12
    kernel, pipe, executed, executed_vs_peak = kernel_model(wl, n_local_max, kernel_ms, peak, int8)
    ncu = env['ncu'].get(name + ('_int8' if int8 else ''), {}) if world == 1 else {}
    roofline = {
        'bound': 'tensor', 'pipe': pipe, 'kernel': kernel, 'arithmetic': 'int8 fixed point' if int8 else 'f64', 'achieved': achieved, 'peak': peak,
        'unit': 'TFLOP/s', 'frac': achieved/peak, 'traffic': ncu.get('dram_bytes_per_launch'),
        'peak_source': env['peak_source'],
        'algorithmic_flops_per_unit': W, 'units_per_launch': G*n_local_max,
        'kernel_ms': kernel_ms, 'kernel_share_of_step': k_ms_max/dev_ms_max,
        'executed_tflops': executed, 'executed_frac': executed_vs_peak/peak,
        'ncu_pipe_active_pct': ncu.get('pipe_active_pct'),
        'ncu_pipe_active_metric': ncu.get('pipe_active_metric'),
        'ncu_dmma_pipe_active_pct': ncu.get('dmma_pipe_active_pct'),
        'ncu_fp64_pipe_active_pct': ncu.get('fp64_pipe_active_pct'),
        'ncu_kernel': ncu.get('kernel'),
        'ncu_source': ncu.get('source'),
        'note': 'achieved counts the reference formulation (W = 8 n_nops n_basis d^2 + 12 d^2 per '
                'seg*omega, SURVEY 8d); the kernel executes fewer flops by pairing (m,n)/(n,m) terms '
                'of Hermitian operators, so frac can exceed executed_frac (and 1.0); '
                'ncu_pipe_active_pct is the FP64 / DMMA pipe-active share of the ncu capture in '
                'profiles/ (the utilisation figure); traffic is its DRAM bytes per launch '
                '(algorithmic: operand stream + split-K partials + output, DESIGN 4.1)',
    }
    return {
        'value': value, 'unit': UNIT, 'ms_per_step': dev_ms_max/steps, 'steps': steps,
        'config': workload_config(wl, world, n_local),
        'e2e': {'value': e2e_value, 'unit': UNIT, 'h2d_bytes_per_step': int(h2d),
                'd2h_bytes_per_step': int(d2h), 'ms_per_step': e2e_ms_max/steps,
                'api': ('ff.infidelity(PulseSequence, spectrum, omega) on a cold cache' if world == 1
                        else 'filter_functions_b200.distributed.infidelity(PulseSequence, spectrum, '
                             'omega) on a cold cache, global grid, every rank')},
        'gpu_launches': int(launches), 'roofline': roofline, 'parity': parity,
        'infidelity': api.tolist()[:6], **({'outputs': outputs} if dump else {}),
    }


def run_b200(args):
    import ctypes

    import torch
    import torch.distributed as dist
    import __graft_entry__ as entry
    entry.build()
    import filter_functions_b200 as ff
    from filter_functions_b200 import _lib
    from filter_functions_b200 import distributed as ffd
    from filter_functions_b200.device import DevicePulse

    world = int(os.environ.get('WORLD_SIZE', 1))
    rank = int(os.environ.get('RANK', 0))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit('launch N>1 with: python -m torch.distributed.run --nnodes=1 '
                             f'--nproc-per-node {args.gpus} --master-addr 127.0.0.1 bench.py '
                             f'--gpus {args.gpus} ...')
        raise SystemExit(f'--gpus {args.gpus} but WORLD_SIZE={world}')
    torch.cuda.set_device(local_rank)
    peers = None
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
        peers = ffd.peer_group()

    ctx = _lib.context(local_rank)
    L = _lib.lib()
    dfma, dmma = ctypes.c_double(), ctypes.c_double()
    _lib.check(ctx, L.ffb_measure_fp64_peak(ctx, ctypes.byref(dfma), ctypes.byref(dmma)))
    ncu = {}
    npath = os.path.join(ROOT, 'profiles', 'ncu_summary.json')
    if os.path.exists(npath):
        ncu = json.load(open(npath))
    sampler = ClockSampler(local_rank)
    sampler.start()
    env = dict(ff=ff, ffd=ffd, _lib=_lib, DevicePulse=DevicePulse, world=world, rank=rank,
               local_rank=local_rank, peers=peers, sampler=sampler, ncu=ncu,
               flush=torch.empty(256 << 20, dtype=torch.uint8, device='cuda'),
               peak=max(dfma.value, dmma.value),
               peak_source='measured live by ffb_measure_fp64_peak (DFMA %.2f, DMMA %.2f TFLOP/s); '
                           'MEASURED_PEAKS.json has no fp64 entry' % (dfma.value, dmma.value))

    head = measure(args.workload, args.steps, args.warmup, env, dump=args.dump_outputs is not None)
    if args.extra is None:
        extra = [w for w in ('c2', 'c3', 'd4') if w != args.workload]
    else:
        extra = [w for w in args.extra.split(',') if w and w != 'none']
    others = {}
    for name in extra:
        others[name] = measure(name, max(3, min(args.steps, 10)), min(args.warmup, 3), env)
    if not args.no_int8 and 'd4' in [args.workload] + extra:
        # the opt-in fixed-point kernel on the int8 tensor cores, same workload, its own parity figures
        others['d4_int8'] = measure('d4', max(3, min(args.steps, 10)), min(args.warmup, 3), env, int8=True)
        others['d4_int8']['note'] = (
            'OPT-IN path (FFB_CTRLMAT_INT8=1), not the default and not the headline: Ozaki-style splitting '
            'into five int8 digits per operand, tcgen05.mma.kind::i8 with exact int32 accumulation in TMEM; '
            'deviation from the FP64 kernels ~1e-11 (inside the 1e-10 tolerance, see parity), DESIGN 4.9')
    sampler.stop_flag.set()
    sampler.join(timeout=1.0)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.dump_outputs is not None:
        dump_outputs(args.dump_outputs, head['outputs'])

    cpu = None
    if not args.no_cpu_baseline and world == 1:
        cpu = cpu_sample(workloads.get(args.workload), args.cpu_seconds)

    line = {
        'metric': METRIC, 'value': head['value'], 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
        'warmup': max(3, args.warmup), 'ms_per_step': head['ms_per_step'],
        'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f64',
        'data': 'synthetic', 'config': head['config'],
        'clocks': sampler.result(),
        'e2e': head['e2e'], 'gpu_launches': head['gpu_launches'], 'roofline': head['roofline'],
        'cpu_baseline': cpu,
        'parity': head['parity'], 'infidelity': head['infidelity'],
        'exchange': ('none (single GPU)' if world == 1 else
                     'partial integrals summed in the epilogue of the infidelity kernel over NVLink '
                     'peer memory (csrc/ffb_peer.cuh)' if peers is not None else
                     'NCCL all-reduce of the partial integrals (no peer-memory path on this box)'),
        'workloads': others,
    }
    print(json.dumps(line), file=RESULT_OUT, flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_b200(args)


if __name__ == '__main__':
    main()
