"""filter_functions_b200 -- B200-native engine for the control-matrix / filter-function /
infidelity path of qutech/filter_functions, behind the reference's Python API.

>>> import filter_functions_b200 as ff
>>> pulse = ff.PulseSequence(H_c, H_n, dt)
>>> F = pulse.get_filter_function(omega)
>>> ff.infidelity(pulse, spectrum, omega)

NumPy arrays in, NumPy arrays out; the arithmetic runs in hand-written sm_100a CUDA kernels
(``csrc/``) reached through the C ABI of ``include/ffb200.h``.  There is no CPU fallback.
"""
from . import basis, gradient, numeric, pulse_sequence, superoperator, util
from .basis import Basis
from .gradient import infidelity_derivative
from .numeric import error_transfer_matrix, infidelity
from .pulse_sequence import (PulseSequence, SequenceBatch, concatenate, concatenate_many,
                             concatenate_periodic, concatenate_without_filter_function)
from .superoperator import liouville_representation

__all__ = ['Basis', 'PulseSequence', 'SequenceBatch', 'basis', 'concatenate', 'concatenate_many',
           'concatenate_periodic', 'concatenate_without_filter_function',
           'error_transfer_matrix', 'gradient', 'infidelity', 'infidelity_derivative',
           'liouville_representation', 'numeric',
           'pulse_sequence', 'superoperator', 'util']

__version__ = '0.1.0'
