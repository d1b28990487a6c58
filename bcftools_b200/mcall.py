"""Thin ctypes wrapper over the C-ABI (include/mcall_b200.h) -- used by tests and bench.py.

It mirrors the reference's hook trio (call.h:131-147): `MCaller(params)` = mcall_init,
`MCaller.call_host / call_device` = mcall over a batch of records, `MCaller.close` = mcall_destroy.
No computation happens in Python and there is no fallback: a missing library or a missing GPU raises.
"""
import ctypes as C
import os

import numpy as np

from . import abi

_LIB_PATH = os.environ.get("MCALL_B200_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", "libmcall_b200.so")
_lib = None

EXPORTS = ["mcb_init", "mcb_destroy", "mcb_set_ploidy", "mcb_call_device", "mcb_call_host", "mcb_host_alloc",
           "mcb_host_free", "mcb_strerror", "mcb_last_cuda_error", "mcb_get_theta", "mcb_get_pl2p", "mcb_get_stats",
           "mcb_set_option", "mcb_version", "mcb_selftest_div", "mcb_get_kernel_times", "mcb_get_fallback_counts"]


JOB_EXPORTS = ["mcb_job_init", "mcb_job_destroy", "mcb_job_ndevices", "mcb_job_set_ploidy", "mcb_job_set_option",
               "mcb_job_call_host", "mcb_job_partition", "mcb_job_last_error"]


class McallError(RuntimeError):
    pass


def lib():
    """Load libmcall_b200.so; built in-tree when it is MISSING.  A stale library is not rebuilt here (file times do not survive the
    copy to a GPU box): `python -m bcftools_b200.build` / `__graft_entry__.build()` rebuild what is older than its sources."""
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            from . import build
            build.build()
        L = C.CDLL(_LIB_PATH)
        L.mcb_init.restype = C.c_int
        L.mcb_init.argtypes = [C.POINTER(C.c_void_p), C.POINTER(abi.McbParams)]
        L.mcb_destroy.restype = None
        L.mcb_destroy.argtypes = [C.c_void_p]
        L.mcb_set_ploidy.restype = C.c_int
        L.mcb_set_ploidy.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.mcb_call_device.restype = C.c_int
        L.mcb_call_device.argtypes = [C.c_void_p, C.POINTER(abi.McbBatch), C.POINTER(abi.McbResult), C.c_void_p]
        L.mcb_call_host.restype = C.c_int
        L.mcb_call_host.argtypes = [C.c_void_p, C.POINTER(abi.McbBatch), C.POINTER(abi.McbResult)]
        L.mcb_host_alloc.restype = C.c_void_p
        L.mcb_host_alloc.argtypes = [C.c_size_t]
        L.mcb_host_free.restype = None
        L.mcb_host_free.argtypes = [C.c_void_p]
        L.mcb_strerror.restype = C.c_char_p
        L.mcb_strerror.argtypes = [C.c_int]
        L.mcb_last_cuda_error.restype = C.c_char_p
        L.mcb_last_cuda_error.argtypes = [C.c_void_p]
        L.mcb_get_theta.restype = C.c_double
        L.mcb_get_theta.argtypes = [C.c_void_p]
        L.mcb_get_pl2p.restype = C.c_int
        L.mcb_get_pl2p.argtypes = [C.c_void_p, C.c_void_p]
        L.mcb_get_stats.restype = C.c_int
        L.mcb_get_stats.argtypes = [C.c_void_p, C.c_void_p]
        L.mcb_set_option.restype = C.c_int
        L.mcb_set_option.argtypes = [C.c_void_p, C.c_char_p, C.c_int64]
        L.mcb_version.restype = C.c_int
        L.mcb_get_kernel_times.restype = C.c_int
        L.mcb_get_kernel_times.argtypes = [C.c_void_p, C.c_void_p]
        L.mcb_get_fallback_counts.restype = C.c_int
        L.mcb_get_fallback_counts.argtypes = [C.c_void_p, C.c_void_p]
        L.mcb_selftest_div.restype = C.c_int
        L.mcb_selftest_div.argtypes = [C.c_void_p, C.c_int, C.c_uint64, C.c_uint64, C.POINTER(C.c_uint64)]
        L.mcb_job_init.restype = C.c_int
        L.mcb_job_init.argtypes = [C.POINTER(C.c_void_p), C.POINTER(abi.McbParams), C.POINTER(C.c_int), C.c_int]
        L.mcb_job_destroy.restype = None
        L.mcb_job_destroy.argtypes = [C.c_void_p]
        L.mcb_job_ndevices.restype = C.c_int
        L.mcb_job_ndevices.argtypes = [C.c_void_p]
        L.mcb_job_set_ploidy.restype = C.c_int
        L.mcb_job_set_ploidy.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.mcb_job_set_option.restype = C.c_int
        L.mcb_job_set_option.argtypes = [C.c_void_p, C.c_char_p, C.c_int64]
        L.mcb_job_call_host.restype = C.c_int
        L.mcb_job_call_host.argtypes = [C.c_void_p, C.POINTER(abi.McbBatch), C.POINTER(abi.McbResult), C.c_void_p]
        L.mcb_job_partition.restype = C.c_int
        L.mcb_job_partition.argtypes = [C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]
        L.mcb_job_last_error.restype = C.c_char_p
        L.mcb_job_last_error.argtypes = [C.c_void_p]
        _lib = L
    return _lib


def partition(nsmpl, nals, nparts):
    """mcb_job_partition: contiguous site ranges of about equal PL volume (host arithmetic of the product library)."""
    nals = np.ascontiguousarray(nals, np.uint8)
    first = np.zeros(nparts + 1, np.int32)
    rc = lib().mcb_job_partition(int(nsmpl), nals.ctypes.data, len(nals), int(nparts), first.ctypes.data)
    if rc != 0:
        raise McallError(f"mcb_job_partition failed: {rc}")
    return first


class MJob:
    """mcall_job.h: one job over several devices (contiguous site ranges, ordered results)."""

    def __init__(self, params, devices, ploidy_tab=None, options=None):
        self.params = params
        self._job = C.c_void_p()
        L = lib()
        p = params.c_struct()
        devs = (C.c_int * len(devices))(*[int(d) for d in devices])
        rc = L.mcb_job_init(C.byref(self._job), C.byref(p), devs, len(devices))
        if rc != 0:
            msg = L.mcb_strerror(rc).decode()
            if self._job:
                msg += " / " + L.mcb_job_last_error(self._job).decode()
                L.mcb_job_destroy(self._job)
                self._job = C.c_void_p()
            raise McallError(f"mcb_job_init failed: {msg}")
        if ploidy_tab is not None:
            tab = np.ascontiguousarray(ploidy_tab, np.uint8).reshape(-1, params.nsmpl)
            for i in range(tab.shape[0]):
                self._check(L.mcb_job_set_ploidy(self._job, i, tab[i].ctypes.data), "mcb_job_set_ploidy")
        for k, v in (options or {}).items():
            self._check(L.mcb_job_set_option(self._job, k.encode(), int(v)), f"mcb_job_set_option({k})")

    def _check(self, rc, what):
        if rc != 0:
            L = lib()
            raise McallError(f"{what} failed: {L.mcb_strerror(rc).decode()} / {L.mcb_job_last_error(self._job).decode()}")

    def call_host(self, batch, result=None, want_gp=False, compact=False, typed=False):
        res = result if result is not None else abi.HostResult(batch, want_gp=want_gp, compact=compact, typed=typed)
        b, r = batch.c_struct(), res.c_struct()
        first = np.zeros(lib().mcb_job_ndevices(self._job) + 1, np.int32)
        self._check(lib().mcb_job_call_host(self._job, C.byref(b), C.byref(r), first.ctypes.data), "mcb_job_call_host")
        res.first_site = first
        return res

    def close(self):
        if self._job:
            lib().mcb_job_destroy(self._job)
            self._job = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


def pinned_empty(shape, dtype):
    """numpy array backed by pinned host memory from mcb_host_alloc (kept alive by the returned array)."""
    dtype = np.dtype(dtype)
    n = int(np.prod(shape)) if np.ndim(shape) else int(shape)
    nbytes = max(1, n * dtype.itemsize)
    ptr = lib().mcb_host_alloc(nbytes)
    if not ptr:
        raise McallError("mcb_host_alloc failed")
    buf = (C.c_char * nbytes).from_address(ptr)
    arr = np.frombuffer(buf, dtype=dtype, count=n).reshape(shape)
    _PINNED[arr.ctypes.data] = ptr
    return arr


_PINNED = {}


def pin_batch(batch):
    """Copy every array of a HostBatch into pinned memory (in place)."""
    for name in abi.BATCH_FIELDS:
        a = getattr(batch, name)
        if a is not None:
            p = pinned_empty(a.shape, a.dtype)
            p[...] = a
            setattr(batch, name, p)
    return batch


def pin_result(res):
    for name in abi.RESULT_FIELDS:
        a = getattr(res, name)
        if a is not None:
            p = pinned_empty(a.shape, a.dtype)
            p[...] = a
            setattr(res, name, p)
    return res


class MCaller:
    def __init__(self, params, ploidy_tab=None, options=None):
        self.params = params
        self._ctx = C.c_void_p()
        L = lib()
        p = params.c_struct()
        rc = L.mcb_init(C.byref(self._ctx), C.byref(p))
        if rc != 0:
            msg = L.mcb_strerror(rc).decode()
            if self._ctx:
                msg += " / " + L.mcb_last_cuda_error(self._ctx).decode()
                L.mcb_destroy(self._ctx)
                self._ctx = C.c_void_p()
            raise McallError(f"mcb_init failed: {msg}")
        if ploidy_tab is not None:
            tab = np.ascontiguousarray(ploidy_tab, np.uint8).reshape(-1, params.nsmpl)
            for i in range(tab.shape[0]):
                self.set_ploidy(i, tab[i])
        for k, v in (options or {}).items():
            self.set_option(k, v)

    def _check(self, rc, what):
        if rc != 0:
            L = lib()
            raise McallError(f"{what} failed: {L.mcb_strerror(rc).decode()} / {L.mcb_last_cuda_error(self._ctx).decode()}")

    def set_ploidy(self, idx, ploidy):
        v = np.ascontiguousarray(ploidy, np.uint8)
        assert v.size == self.params.nsmpl
        self._check(lib().mcb_set_ploidy(self._ctx, int(idx), v.ctypes.data), "mcb_set_ploidy")

    def set_option(self, key, value):
        self._check(lib().mcb_set_option(self._ctx, key.encode(), int(value)), f"mcb_set_option({key})")

    @property
    def theta(self):
        return lib().mcb_get_theta(self._ctx)

    def pl2p(self):
        out = np.zeros(256, np.float64)
        lib().mcb_get_pl2p(self._ctx, out.ctypes.data)
        return out

    def stats(self):
        out = np.zeros(4, np.int64)
        lib().mcb_get_stats(self._ctx, out.ctypes.data)
        return out

    def call_host(self, batch, result=None, want_gp=False, compact=False, typed=False):
        """mcb_call_host on numpy (host) arrays; returns an abi.HostResult.  typed=True: GT/GQ/PL come back as the BCF
        typed vectors gt8/gq8/pl16 (mcb_result.gt8 ...); HostResult.widen() maps them to the int32 arrays."""
        res = result if result is not None else abi.HostResult(batch, want_gp=want_gp, compact=compact, typed=typed)
        b, r = batch.c_struct(), res.c_struct()
        self._check(lib().mcb_call_host(self._ctx, C.byref(b), C.byref(r)), "mcb_call_host")
        return res

    def call_device(self, batch_struct, result_struct, stream=0):
        """mcb_call_device on already-built McbBatch/McbResult structs holding DEVICE pointers."""
        self._check(lib().mcb_call_device(self._ctx, C.byref(batch_struct), C.byref(result_struct), C.c_void_p(stream)),
                    "mcb_call_device")

    def kernel_times_ms(self):
        """Per allele-count class device time of the last call_device (option time_kernels=1): array[6], [0]=sum."""
        out = np.zeros(6, np.float32)
        self._check(lib().mcb_get_kernel_times(self._ctx, out.ctypes.data), "mcb_get_kernel_times")
        return out

    def fallback_counts(self):
        """Sites per allele-count class that the multi-allelic kernels of the last call_device handed to the general kernel: array[6]."""
        out = np.zeros(6, np.int32)
        self._check(lib().mcb_get_fallback_counts(self._ctx, out.ctypes.data), "mcb_get_fallback_counts")
        return out

    def selftest_div(self, mode, n=0, seed=1):
        """Number of quotients of the shared-reciprocal division that differ from IEEE a/b (must be 0)."""
        bad = C.c_uint64(0)
        self._check(lib().mcb_selftest_div(self._ctx, int(mode), int(n), int(seed), C.byref(bad)), "mcb_selftest_div")
        return bad.value

    def close(self):
        if self._ctx:
            lib().mcb_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
