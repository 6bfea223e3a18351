"""Time ff.infidelity_derivative against the forward step on the same inputs.

    python tools/bench_gradient.py [--workloads d4 c2] [--steps 5] [--warmup 1]

For each workload (d4: G = 1e4, n_omega = 1e4, 6 noise operators, 5 controls, with the J-dependent
sensitivities as n_coeffs_deps; c2: the single-qubit GRAPE pulse) it prints one JSON line with the device
time of the gradient call (CUDA events on the library's stream around the call, which synchronises), the
same for the forward step (ff.infidelity on a cold pulse: diagonalisation, control matrix, filter function,
integral), their ratio, the FP64 rate from the flop formula of DESIGN.md section 4.11, and the card's name
and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def flops_per_seg_omega(d, n_ctrl):
    """Per (segment, frequency, noise operator): 134 d^3 + (30 + 8 n_ctrl) d^2 (DESIGN.md 4.11)."""
    return 134*d**3 + (30 + 8*n_ctrl)*d**2


def power_limit():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader,nounits',
                              '-i', '0'], capture_output=True, text=True, timeout=30).stdout.strip()
        return float(out.splitlines()[0])
    except Exception:  # noqa: BLE001
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--workloads', nargs='+', default=['d4', 'c2'])
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=1)
    args = ap.parse_args()
    import torch

    import filter_functions_b200 as ff
    import workloads
    from filter_functions_b200 import _lib
    ctx = _lib.context()
    stream = torch.cuda.current_stream()
    _lib.lib().ffb_set_stream(ctx, stream.cuda_stream, 1)
    card, watts = torch.cuda.get_device_name(0), power_limit()

    def timed(fn):
        for _ in range(args.warmup):
            fn()
        times = []
        for _ in range(args.steps):
            start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            start.record(stream)
            fn()
            end.record(stream)
            torch.cuda.synchronize()
            times.append(start.elapsed_time(end))
        return float(np.median(times))

    try:
        for name in args.workloads:
            wl = workloads.get(name)
            n_nops, n_cops = len(wl.n_opers), len(wl.c_opers)
            deps = None
            if name in ('c3', 'd4'):   # n_coeffs[i] = J_i = c_coeffs[i], i < 3
                deps = np.zeros((n_nops, n_cops, wl.G))
                for i in range(3):
                    deps[i, i] = 1.0
            basis = ff.Basis.pauli(int(np.log2(wl.d)))

            def pulse():
                return ff.PulseSequence(list(zip(wl.c_opers, wl.c_coeffs, wl.c_ids)),
                                        list(zip(wl.n_opers, wl.n_coeffs, wl.n_ids)), wl.dt, basis)

            ms_fwd = timed(lambda: ff.infidelity(pulse(), wl.spectrum, wl.omega))
            ms_grad = timed(lambda: ff.infidelity_derivative(pulse(), wl.spectrum, wl.omega,
                                                             n_coeffs_deps=deps))
            flops = flops_per_seg_omega(wl.d, n_cops)*wl.G*len(wl.omega)*n_nops
            print(json.dumps({
                'workload': name, 'G': wl.G, 'n_omega': len(wl.omega), 'd': wl.d, 'n_nops': n_nops,
                'n_ctrl': n_cops, 'gradient_ms': round(ms_grad, 3), 'forward_ms': round(ms_fwd, 3),
                'gradient_over_forward': round(ms_grad/ms_fwd, 2),
                'flops_per_seg_omega_nop': flops_per_seg_omega(wl.d, n_cops),
                'fp64_tflops': round(flops/ms_grad/1e9, 3), 'card': card, 'power_limit_w': watts}),
                flush=True)
    finally:
        _lib.lib().ffb_set_stream(ctx, None, 0)


if __name__ == '__main__':
    main()
