"""Context and storage: the device-resident `Box<[T]>` of `Array` (src/array.rs:5-8).

One `Context` per GPU per process (include/mdim.h).  `Storage` is a flat run of elements that
lives either in host memory (numpy, optionally pinned) or in HBM; an `Array` owns one Storage
(or a tuple of them for tuple-typed elements, stored as a structure of arrays).
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import _ffi as F

NP_OF = {F.U8: np.uint8, F.I32: np.int32, F.U32: np.uint32, F.I64: np.int64, F.U64: np.uint64, F.F32: np.float32, F.F64: np.float64,
         F.I8: np.int8, F.I16: np.int16, F.U16: np.uint16}


class Context:
    """mdim_ctx.  Raises when the library or an sm_100 device is missing: there is no CPU path."""

    def __init__(self, device=None):
        if device is None:
            device = int(os.environ.get("LOCAL_RANK", "0"))
        self.lib = F.lib()
        h = C.c_void_p()
        st = self.lib.mdim_init(int(device), C.byref(h))
        if st != F.OK:
            raise F.MdimError(st, f"mdim_init(device={device}): {self.lib.mdim_status_string(st).decode()} "
                                  f"(this library runs only on an sm_100 GPU; there is no CPU fallback)")
        self.handle = h
        self.device = int(device)
        self._closed = False

    # -- errors ---------------------------------------------------------------------------------
    def check(self, st):
        if st == F.OK:
            return
        info = F.ErrorInfo()
        self.lib.mdim_last_error(self.handle, C.byref(info))
        msg = info.message.decode(errors="replace") if info.status == st and info.message else self.lib.mdim_status_string(st).decode()
        cls = F.Panic if st in (F.ERR_OOB, F.ERR_ARITH, F.ERR_SIZE) else F.MdimError
        raise cls(st, msg, info)

    # -- plumbing -------------------------------------------------------------------------------
    def set_stream(self, cuda_stream):
        self.check(self.lib.mdim_set_stream(self.handle, C.c_void_p(cuda_stream or 0)))

    def stream_handle(self):
        """cudaStream_t the collects are launched on (wrap it with torch.cuda.ExternalStream to record events on it)."""
        p = C.c_void_p()
        self.check(self.lib.mdim_get_stream(self.handle, C.byref(p)))
        return p.value or 0

    def sync(self):
        self.check(self.lib.mdim_sync(self.handle))

    def last_kernel(self):
        """Name of the kernel the last collect launched (`mdim_jit_kernel[ops+shape]` when NVRTC specialised the chain)."""
        buf = C.create_string_buffer(96)
        self.check(self.lib.mdim_last_kernel(self.handle, buf, 96))
        return buf.value.decode()

    def launch_count(self):
        return int(self.lib.mdim_launch_count(self.handle))

    def device_info(self):
        sm, a, b, hbm = C.c_int(), C.c_int(), C.c_int(), C.c_size_t()
        self.check(self.lib.mdim_device_info(self.handle, C.byref(sm), C.byref(a), C.byref(b), C.byref(hbm)))
        return {"sm_count": sm.value, "cc": (a.value, b.value), "hbm_bytes": hbm.value}

    def alloc(self, nbytes):
        p = C.c_void_p()
        self.check(self.lib.mdim_buf_alloc(self.handle, nbytes, C.byref(p)))
        return p.value

    def free(self, ptr):
        if not self._closed and ptr:
            self.lib.mdim_buf_free(self.handle, C.c_void_p(ptr))

    def host_alloc(self, nbytes):
        p = C.c_void_p()
        self.check(self.lib.mdim_host_alloc(self.handle, nbytes, C.byref(p)))
        return p.value

    def host_free(self, ptr):
        if not self._closed and ptr:
            self.lib.mdim_host_free(self.handle, C.c_void_p(ptr))

    def upload(self, dptr, host_array):
        a = np.ascontiguousarray(host_array)
        self.check(self.lib.mdim_upload(self.handle, C.c_void_p(dptr), C.c_void_p(a.ctypes.data), a.nbytes))

    def download(self, host_array, dptr):
        assert host_array.flags["C_CONTIGUOUS"]
        self.check(self.lib.mdim_download(self.handle, C.c_void_p(host_array.ctypes.data), C.c_void_p(dptr), host_array.nbytes))

    def collect(self, expr, out_dptr, flags=0):
        self.check(self.lib.mdim_collect(self.handle, C.byref(expr), C.c_void_p(out_dptr), flags))

    def collect_tuple(self, expr, out_dptrs, flags=0):
        """mdim_collect_tuple: one launch fills the run of every scalar leaf of a tuple-typed element."""
        outs = (C.c_void_p * len(out_dptrs))(*out_dptrs)
        self.check(self.lib.mdim_collect_tuple(self.handle, C.byref(expr), outs, len(out_dptrs), flags))

    def collect_host(self, expr, out_hptr, flags=0):
        self.check(self.lib.mdim_collect_host(self.handle, C.byref(expr), C.c_void_p(out_hptr), flags))

    def describe(self, expr, flags=0):
        buf = C.create_string_buffer(256)
        st = self.lib.mdim_plan_describe(self.handle, C.byref(expr), flags, buf, 256)
        return st, buf.value.decode()

    def ipc_export(self, dptr):
        h = (C.c_uint8 * F.IPC_HANDLE_BYTES)()
        self.check(self.lib.mdim_ipc_export(self.handle, C.c_void_p(dptr), h))
        return bytes(h)

    def ipc_open(self, handle_bytes):
        h = (C.c_uint8 * F.IPC_HANDLE_BYTES).from_buffer_copy(handle_bytes)
        p = C.c_void_p()
        self.check(self.lib.mdim_ipc_open(self.handle, h, C.byref(p)))
        return p.value

    def ipc_close(self, dptr):
        self.check(self.lib.mdim_ipc_close(self.handle, C.c_void_p(dptr)))

    def close(self):
        if not self._closed:
            self._closed = True
            self.lib.mdim_shutdown(self.handle)


_default = None


def default_context():
    global _default
    if _default is None:
        _default = Context()
    return _default


def set_default_context(ctx):
    global _default
    _default = ctx


def describe_nodevice(expr, flags=0):
    """Which kernel the planner would pick; needs the library but no GPU."""
    buf = C.create_string_buffer(256)
    st = F.lib().mdim_plan_describe_nodevice(C.byref(expr), flags, buf, 256)
    return st, buf.value.decode()


class Storage:
    """A flat run of `n` elements of `dtype`, in host memory and/or in HBM."""

    def __init__(self, dtype, n, host=None, dptr=None, ctx=None, owns_device=True, pinned_ptr=None, keep=None):
        self.dtype, self.n = dtype, int(n)
        self.host = host      # numpy 1-D array or None
        self.dptr = dptr      # device pointer or None
        self.ctx = ctx
        self.owns_device = owns_device
        self.pinned_ptr = pinned_ptr
        self.keep = keep      # e.g. a torch tensor whose memory `dptr` points into
        self.home = "device" if (dptr is not None and host is None) else "host"

    @property
    def nbytes(self):
        return self.n * F.DTYPE_SIZE[self.dtype]

    @staticmethod
    def from_host(dtype, array):
        a = np.ascontiguousarray(array, dtype=NP_OF[dtype]).reshape(-1)
        return Storage(dtype, a.size, host=a)

    @staticmethod
    def pinned(ctx, dtype, n):
        nbytes = max(int(n) * F.DTYPE_SIZE[dtype], 1)
        p = ctx.host_alloc(nbytes)
        raw = (C.c_uint8 * nbytes).from_address(p)
        a = np.frombuffer(raw, dtype=NP_OF[dtype], count=int(n))
        return Storage(dtype, n, host=a, ctx=ctx, pinned_ptr=p)

    @staticmethod
    def device(ctx, dtype, n):
        return Storage(dtype, n, dptr=ctx.alloc(int(n) * F.DTYPE_SIZE[dtype]), ctx=ctx)

    @staticmethod
    def wrap_device(ctx, dtype, n, dptr, keep=None):
        return Storage(dtype, n, dptr=dptr, ctx=ctx, owns_device=False, keep=keep)

    def pointer(self, location):
        if location == "any":  # planning only: alignment matters, residence does not
            return self.dptr if self.dptr is not None else self.host.ctypes.data
        if location == "host":
            if self.host is None:
                raise F.MdimError(F.ERR_INVALID, "device-resident operand in a host collect")
            return self.host.ctypes.data
        if self.dptr is None:
            raise F.MdimError(F.ERR_INVALID, "host-resident operand in a device collect (call to_device())")
        return self.dptr

    def ensure_device(self, ctx):
        if self.dptr is None:
            self.ctx = self.ctx or ctx
            self.dptr = self.ctx.alloc(self.nbytes)
            self.ctx.upload(self.dptr, self.host)
        return self

    def to_numpy(self):
        if self.home == "host":
            return self.host
        out = np.empty(self.n, dtype=NP_OF[self.dtype])
        if self.n:
            self.ctx.download(out, self.dptr)
        return out

    def __del__(self):
        try:
            if self.dptr is not None and self.owns_device and self.ctx is not None:
                self.ctx.free(self.dptr)
            if self.pinned_ptr is not None and self.ctx is not None:
                self.host = None
                self.ctx.host_free(self.pinned_ptr)
        except Exception:
            pass
