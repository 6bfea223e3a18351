"""ctypes binding of ``libffb200.so`` (C ABI declared in ``include/ffb200.h``).

The library is built in-tree by ``__graft_entry__.build()`` (plain ``nvcc`` for sm_100a).  There is
NO CPU fallback: if the shared object is missing, or no sm_100 GPU is visible, every compute call
raises.  Importing this module never touches the GPU, so the package can be imported on a CPU-only
box (the ``-m "not gpu"`` tests check that the library loads and exports every declared symbol).
"""
import ctypes
import os
import threading
import weakref
from ctypes import POINTER, byref, c_char_p, c_double, c_int, c_int64, c_size_t, c_void_p

import numpy as np

__all__ = ['lib', 'context', 'check', 'library_path', 'FFBError', 'EXPORTED_SYMBOLS']

_HERE = os.path.dirname(os.path.abspath(__file__))
#: FFB200_LIBRARY selects another build of the same sources (kernel experiments), never another backend
library_path = os.environ.get('FFB200_LIBRARY') or os.path.join(_HERE, 'csrc', 'libffb200.so')

FFB_OK, FFB_EINVAL, FFB_ENODEVICE, FFB_ECUDA, FFB_ENOMEM, FFB_ENOTCONV = 0, -1, -2, -3, -4, -5

_dp = POINTER(c_double)
_ip = POINTER(c_int)

#: every ``extern "C"`` symbol declared in include/ffb200.h with its (restype, argtypes)
EXPORTED_SYMBOLS = {
    'ffb_init': (c_int, [POINTER(c_void_p), c_int]),
    'ffb_destroy': (None, [c_void_p]),
    'ffb_last_error': (c_char_p, [c_void_p]),
    'ffb_version': (c_char_p, []),
    'ffb_set_stream': (c_int, [c_void_p, c_void_p, c_int]),
    'ffb_sync': (c_int, [c_void_p]),
    'ffb_launch_count': (c_int64, [c_void_p]),
    'ffb_device_info': (c_int, [c_void_p, _ip, _ip, _ip, POINTER(c_size_t)]),
    'ffb_measure_fp64_peak': (c_int, [c_void_p, _dp, _dp]),
    'ffb_diagonalize': (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                c_void_p, c_void_p, c_void_p]),
    'ffb_control_matrix_from_scratch': (c_int, [c_void_p] + [c_int]*5 + [c_void_p]*10),
    'ffb_control_matrix_intermediates': (c_int, [c_void_p] + [c_int]*5 + [c_void_p]*17),
    'ffb_filter_function': (c_int, [c_void_p] + [c_int]*4 + [c_void_p, c_int, c_void_p]),
    'ffb_control_matrix_from_atomic': (c_int, [c_void_p] + [c_int]*4 + [c_void_p]*3
                                       + [c_int, c_int, c_void_p]),
    'ffb_control_matrix_periodic': (c_int, [c_void_p] + [c_int]*4 + [c_void_p]*3
                                    + [c_int, c_void_p]),
    'ffb_infidelity': (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p,
                               c_int, c_int, c_void_p, c_int, c_void_p]),
    'ffb_infidelity_derivative': (c_int, [c_void_p] + [c_int]*6 + [c_void_p]*12
                                  + [c_int, c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p,
                                     c_int, c_void_p]),
    'ffb_decay_amplitudes': (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_int,
                                     c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    'ffb_dev_decay_amplitudes': (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_int,
                                         c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    'ffb_concatenate_many': (c_int, [c_void_p] + [c_int]*7 + [c_void_p]*7 + [c_int, c_int]
                             + [c_void_p]*8),
    'ffb_concatenate_pulses': (c_int, [c_void_p] + [c_int]*5 + [c_void_p]*14 + [c_int, c_int]
                               + [c_void_p]*2),
    'ffb_liouville_representation': (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p,
                                             c_void_p]),
    'ffb_cexp': (c_int, [c_void_p, c_int, c_void_p, c_double, c_void_p]),
    'ffb_cexpm1': (c_int, [c_void_p, c_int, c_void_p, c_void_p]),
    'ffb_pulse_filter_function': (c_int, [c_void_p] + [c_int]*6 + [c_void_p]*9 + [c_int, c_int]
                                  + [c_void_p]*8),
    'ffb_dev_diagonalize': (c_int, [c_void_p, c_int, c_int, c_int] + [c_void_p]*6),
    'ffb_dev_control_matrix_from_scratch': (c_int, [c_void_p] + [c_int]*5 + [c_void_p]*9
                                            + [c_int, c_void_p]),
    'ffb_dev_filter_function': (c_int, [c_void_p] + [c_int]*4 + [c_void_p, c_int, c_void_p]),
    'ffb_dev_control_matrix_from_atomic': (c_int, [c_void_p] + [c_int]*4 + [c_void_p]*3
                                           + [c_int, c_int, c_void_p]),
    'ffb_dev_infidelity': (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_void_p,
                                   c_void_p, c_int, c_int, c_void_p, c_int, c_void_p]),
    'ffb_dev_alloc': (c_int, [c_void_p, c_size_t, POINTER(c_void_p)]),
    'ffb_dev_free': (c_int, [c_void_p, c_void_p]),
    'ffb_memcpy_h2d': (c_int, [c_void_p, c_void_p, c_void_p, c_size_t]),
    'ffb_memcpy_d2h': (c_int, [c_void_p, c_void_p, c_void_p, c_size_t]),
    'ffb_host_alloc': (c_int, [c_void_p, c_size_t, POINTER(c_void_p)]),
    'ffb_host_free': (c_int, [c_void_p, c_void_p]),
    'ffb_kernel_timing_enable': (c_int, [c_void_p, c_int]),
    'ffb_kernel_timing_read': (c_int, [c_void_p, _dp, POINTER(c_int64), c_int]),
    'ffb_dispatch_log': (c_int, [c_void_p, c_void_p, c_int]),
    'ffb_diag_dispatch_log': (c_int, [c_void_p, c_void_p, c_int]),
    'ffb_shadow_enable_next': (c_int, [c_void_p, c_int]),
    'ffb_shadow_upload': (c_int, [c_void_p, c_void_p, c_size_t]),
    'ffb_shadow_query': (c_int, [c_void_p, c_void_p, c_size_t]),
    'ffb_shadow_drop': (c_int, [c_void_p, c_void_p, c_size_t]),
    'ffb_shadow_stats': (c_int, [c_void_p, _ip, POINTER(c_size_t), POINTER(c_int64), POINTER(c_size_t)]),
    'ffb_comm_create': (c_int, [c_void_p, c_int, c_int, c_void_p]),
    'ffb_comm_connect': (c_int, [c_void_p, c_void_p]),
    'ffb_comm_destroy': (c_int, [c_void_p]),
    'ffb_comm_info': (c_int, [c_void_p, _ip, _ip, POINTER(c_size_t)]),
    'ffb_comm_reduce_infidelity': (c_int, [c_void_p, c_int]),
    'ffb_allreduce_sum': (c_int, [c_void_p, c_void_p, c_int]),
    'ffb_dev_allreduce_sum': (c_int, [c_void_p, c_void_p, c_int]),
    'ffb_comm_data_window': (c_int, [c_void_p, c_size_t, c_void_p]),
    'ffb_comm_data_connect': (c_int, [c_void_p, c_void_p]),
    'ffb_allgather_columns': (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
}

COMM_HANDLE_BYTES = 64


class FFBError(RuntimeError):
    """CUDA / device failure inside libffb200."""


_lib = None
_lib_lock = threading.Lock()
_contexts = {}
#: A context (device pools, staging block, ticket counters) must be used by one thread at a time
#: (include/ffb200.h) and ctypes drops the GIL during a call, so every entry into the library --
#: including the ``ffb_host_free`` a garbage-collected result array triggers from whatever thread
#: the collector happens to run on -- takes this re-entrant lock.
_call_lock = threading.RLock()


class _SerialisedLibrary:
    """The loaded library with every exported function wrapped to hold ``_call_lock``."""

    def __init__(self, handle):
        self._handle = handle
        for name, (restype, argtypes) in EXPORTED_SYMBOLS.items():
            fn = getattr(handle, name)
            fn.restype = restype
            fn.argtypes = argtypes
            setattr(self, name, self._serialised(fn))

    @staticmethod
    def _serialised(fn):
        def call(*args):
            with _call_lock:
                return fn(*args)
        call.__name__ = fn.__name__
        return call


def lib():
    """Load (once) and return the shared library.  Raises if it has not been built."""
    global _lib
    if _lib is None:
        with _lib_lock:
            if _lib is None:
                if not os.path.exists(library_path):
                    raise FFBError(
                        f'{library_path} not found. Build it with '
                        '`python -c "import __graft_entry__ as g; g.build()"` from the repository '
                        'root (needs nvcc). filter_functions_b200 has no CPU fallback.')
                _lib = _SerialisedLibrary(ctypes.CDLL(library_path))
    return _lib


def context(device=None):
    """The (cached) engine context for ``device`` (default: ``FFB200_DEVICE``, else ``LOCAL_RANK``,
    else 0)."""
    if device is None:
        device = int(os.environ.get('FFB200_DEVICE', os.environ.get('LOCAL_RANK', 0)))
    ctx = _contexts.get(device)
    if ctx is None:
        handle = c_void_p()
        rc = lib().ffb_init(byref(handle), device)
        if rc != FFB_OK:
            msg = lib().ffb_last_error(None).decode()
            raise FFBError(f'ffb_init(device={device}) failed: {msg}')
        ctx = _contexts[device] = handle
    return ctx


def check(ctx, rc):
    """Map a negative return code to the Python exception the reference would raise."""
    if rc == FFB_OK:
        return
    msg = lib().ffb_last_error(ctx).decode()
    if rc == FFB_EINVAL:
        raise ValueError(msg)
    if rc == FFB_ENOMEM:
        raise MemoryError(msg)
    if rc == FFB_ENOTCONV:
        from .util import CalculationError
        raise CalculationError(msg)
    raise FFBError(msg)


#: result arrays at least this large are allocated in page-locked memory (download at PCIe speed)
PINNED_THRESHOLD = 256 << 10
PINNED_LIMIT = 1 << 30
#: results of one call that are smaller than this in total are not page-locked (nor mirrored on the device)
SMALL_RESULT_BYTES = 64 << 10


def _host_free(ctx, address):
    try:
        lib().ffb_host_free(ctx, address)
    except Exception:  # interpreter shutdown
        pass


def empty(shape, dtype=np.complex128, ctx=None):
    """``np.empty`` for result arrays of the engine.  Large arrays live in page-locked memory taken
    from the library's pool, so the device->host copy that fills them runs at full PCIe speed; the
    block goes back to the pool when the array (and all views of it) are garbage collected."""
    shape = tuple(int(s) for s in (shape if np.iterable(shape) else (shape,)))
    dtype = np.dtype(dtype)
    nbytes = int(np.prod(shape, dtype=np.int64))*dtype.itemsize
    if nbytes < PINNED_THRESHOLD or nbytes > PINNED_LIMIT:
        return np.empty(shape, dtype=dtype)
    ctx = context() if ctx is None else ctx
    address = c_void_p()
    if lib().ffb_host_alloc(ctx, nbytes, byref(address)) != FFB_OK:
        return np.empty(shape, dtype=dtype)   # pageable still works, only slower
    buf = (ctypes.c_char*nbytes).from_address(address.value)
    weakref.finalize(buf, _host_free, ctx, address.value)
    return np.frombuffer(buf, dtype=dtype).reshape(shape)


def empty_many(specs, ctx=None):
    """Several result arrays carved out of ONE page-locked block (one pool round trip instead of one
    per array); ``specs`` is a list of ``(shape, dtype)``.  The block returns to the pool when the
    last of the arrays is garbage collected.  Falls back to ``empty`` per array when the total is
    small or too large."""
    shapes = [tuple(int(s) for s in (sh if np.iterable(sh) else (sh,))) for sh, _ in specs]
    dtypes = [np.dtype(dt) for _, dt in specs]
    sizes = [int(np.prod(sh, dtype=np.int64))*dt.itemsize for sh, dt in zip(shapes, dtypes)]
    offsets, total = [], 0
    for n in sizes:
        offsets.append(total)
        total += (n + 255) & ~255
    if total > PINNED_LIMIT:
        return [empty(sh, dt, ctx) for sh, dt in zip(shapes, dtypes)]
    if total < SMALL_RESULT_BYTES:
        # small results live in ordinary memory (thousands of small pulses must not pin host memory);
        # the library downloads them in one copy through its own staging block and memcpy's them here
        buf = np.empty(total, dtype=np.uint8)
        return [np.frombuffer(buf, dtype=dt, count=n//dt.itemsize, offset=off).reshape(sh)
                for sh, dt, n, off in zip(shapes, dtypes, sizes, offsets)]
    ctx = context() if ctx is None else ctx
    address = c_void_p()
    if lib().ffb_host_alloc(ctx, total, byref(address)) != FFB_OK:
        return [np.empty(sh, dtype=dt) for sh, dt in zip(shapes, dtypes)]
    buf = (ctypes.c_char*total).from_address(address.value)
    weakref.finalize(buf, _host_free, ctx, address.value)
    return [np.frombuffer(buf, dtype=dt, count=n//dt.itemsize, offset=off).reshape(sh)
            for sh, dt, n, off in zip(shapes, dtypes, sizes, offsets)]


def keep_on_device(ctx):
    """The results of the NEXT library call stay mirrored in device memory (``ffb_shadow_*`` of
    include/ffb200.h), so that later calls that are handed those arrays skip the upload."""
    lib().ffb_shadow_enable_next(ctx, 1)


def freeze_shadowed(ctx, *arrays):
    """Arrays that have a device mirror become read-only: the mirror is what later library calls read,
    so an in-place edit of the host copy would silently not be seen (copy the array to modify it)."""
    query = lib().ffb_shadow_query
    for arr in arrays:
        if arr is not None and arr.nbytes >= (64 << 10) and query(ctx, arr.ctypes.data, arr.nbytes):
            arr.flags.writeable = False


def mirror_input(ctx, arr):
    """Upload ``arr`` (allocated by :func:`empty`) once and keep the device copy for later calls that are
    handed the same array; the array becomes read-only if the mirror was kept."""
    lib().ffb_shadow_upload(ctx, arr.ctypes.data, arr.nbytes)
    freeze_shadowed(ctx, arr)


def shadow_stats(ctx=None):
    """(number of shadows, bytes held, uploads avoided, bytes not uploaded) of a context."""
    ctx = context() if ctx is None else ctx
    n, nbytes, hits, hit_bytes = c_int(), c_size_t(), c_int64(), c_size_t()
    lib().ffb_shadow_stats(ctx, byref(n), byref(nbytes), byref(hits), byref(hit_bytes))
    return n.value, nbytes.value, hits.value, hit_bytes.value


DISPATCH_LOG_MAX = 256


class DispatchRecord(ctypes.Structure):
    """``ffb_dispatch_record`` of include/ffb200.h."""
    _fields_ = [('kernel', ctypes.c_char*64), ('prologue', ctypes.c_char*96)] + [
        (name, c_int) for name in ('S', 'passes_per_chunk', 'n_pass', 'n_sp', 'pps', 'transposed', 'n_rb',
                                   'n_wtiles', 'ctas_by_regs', 'block', 'n_blocks', 'n_omega', 'route',
                                   'chunk_segs', 'n_bands', 'n_proxies')]


def dispatch_log(ctx=None):
    """What the control-matrix calls of a context launched since the last call, one dict per frequency
    block, oldest first (``ffb_dispatch_log``); clears the record."""
    return _read_log(lib().ffb_dispatch_log, ctx)


def diag_dispatch_log(ctx=None):
    """What the diagonalisations of a context launched since the last call, one dict per call, oldest
    first (``ffb_diag_dispatch_log``); clears the record."""
    return _read_log(lib().ffb_diag_dispatch_log, ctx)


def _read_log(fn, ctx):
    ctx = context() if ctx is None else ctx
    records = (DispatchRecord*DISPATCH_LOG_MAX)()
    n = fn(ctx, ctypes.addressof(records), DISPATCH_LOG_MAX)
    return [{name: (getattr(rec, name).decode() if name in ('kernel', 'prologue') else getattr(rec, name))
             for name, _ in DispatchRecord._fields_} for rec in records[:n]]


def ptr(arr):
    """Raw pointer of a C-contiguous ndarray (``None`` -> NULL)."""
    if arr is None:
        return None
    return arr.ctypes.data   # plain integer address: argtypes are c_void_p (no cast object per call)


def as_c128(x):
    return np.ascontiguousarray(x, dtype=np.complex128)


def as_f64(x):
    return np.ascontiguousarray(x, dtype=np.float64)
