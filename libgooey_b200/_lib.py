"""ctypes binding of libgooey_b200.so (the C ABI in include/gooey_batch.h and include/gooey.h).

The shared library is built in-tree by ``__graft_entry__.build()`` into
``libgooey_b200/lib/``.  There is no CPU fallback: if the library is missing the
import of any compute entry raises, and on a box without a CUDA device every
compute call returns GOOEY_E_NO_DEVICE which is raised as ``GooeyError``.
"""
import ctypes
import os

# One hardware queue per stream the library uses (type buckets x {front, back, general} + copy): with the default 8
# connections independent kernels alias onto one queue and serialise (measured 83 -> 77 ms per C2 step).  Only effective
# if the process has not created its CUDA context yet; the shared library does the same at load time.
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

_HERE = os.path.dirname(os.path.abspath(__file__))
# GOOEY_B200_LIB selects another build of the same library (kernel tuning experiments); never a different backend.
LIB_PATH = os.environ.get("GOOEY_B200_LIB") or os.path.join(_HERE, "lib", "libgooey_b200.so")


class GooeyError(RuntimeError):
    pass


class VoicePatch(ctypes.Structure):
    """GooeyVoicePatch (include/gooey_batch.h)."""
    _fields_ = [("instrument", ctypes.c_uint32), ("aux", ctypes.c_uint32), ("params", ctypes.c_float * 24)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise GooeyError(
                f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). libgooey_b200 has no CPU fallback.")
        L = ctypes.CDLL(LIB_PATH)
        c = ctypes
        L.gooey_b200_last_error.restype = c.c_char_p
        L.gooey_b200_device_count.restype = c.c_int
        L.gooey_b200_launch_count.restype = c.c_uint64
        L.gooey_b200_last_kernel_ms.restype = c.c_float
        L.gooey_voice_batch_new.argtypes = [c.c_float, c.c_uint32, c.POINTER(VoicePatch), c.c_int, c.POINTER(c.c_void_p)]
        L.gooey_voice_batch_free.argtypes = [c.c_void_p]
        L.gooey_voice_batch_free.restype = None
        L.gooey_voice_batch_trigger.argtypes = [c.c_void_p, c.c_uint32, c.c_uint32, c.c_float]
        L.gooey_voice_batch_trigger_all.argtypes = [c.c_void_p, c.c_uint32, c.POINTER(c.c_float)]
        L.gooey_voice_batch_set_param.argtypes = [c.c_void_p, c.c_uint32, c.c_uint32, c.c_uint32, c.c_float, c.c_int]
        L.gooey_voice_batch_note_on.argtypes = [c.c_void_p, c.c_uint32, c.c_uint32, c.c_uint32, c.c_float]
        L.gooey_voice_batch_release.argtypes = [c.c_void_p, c.c_uint32, c.c_uint32]
        L.gooey_voice_batch_set_buffer.argtypes = [c.c_void_p, c.c_uint32, c.c_uint32, c.c_void_p, c.c_uint32, c.c_float]
        L.gooey_voice_batch_share_buffer.argtypes = [c.c_void_p, c.c_uint32, c.c_uint32, c.c_uint32]
        L.gooey_voice_batch_set_seed.argtypes = [c.c_void_p, c.c_uint32, c.c_uint32, c.c_uint32]
        L.gooey_voice_batch_render.argtypes = [c.c_void_p, c.c_uint32, c.c_void_p]
        L.gooey_voice_batch_render_device.argtypes = [c.c_void_p, c.c_uint32, c.c_void_p, c.c_size_t]
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise GooeyError(f"libgooey_b200 error {rc}: {lib().gooey_b200_last_error().decode(errors='replace')}")


class HostBuffer:
    """Pinned host memory from gooey_b200_host_alloc: placed on the NUMA node the device hangs off, so that several ranks
    draining at once do not all write into one node.  `.array(shape, dtype)` views it as numpy; free with close()."""

    def __init__(self, nbytes, device=0):
        L = lib()
        L.gooey_b200_host_alloc.restype = ctypes.c_void_p
        L.gooey_b200_host_alloc.argtypes = [ctypes.c_size_t, ctypes.c_int, ctypes.POINTER(ctypes.c_int)]
        L.gooey_b200_host_free.argtypes = [ctypes.c_void_p]
        L.gooey_b200_host_free.restype = None
        node = ctypes.c_int(-1)
        self.nbytes = int(nbytes)
        self.ptr = L.gooey_b200_host_alloc(self.nbytes, int(device), ctypes.byref(node))
        if not self.ptr:
            raise GooeyError("gooey_b200_host_alloc failed: " + L.gooey_b200_last_error().decode(errors="replace"))
        self.numa_node = node.value

    def array(self, shape, dtype):
        import numpy as np
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        assert n <= self.nbytes
        buf = (ctypes.c_char * n).from_address(self.ptr)
        return np.frombuffer(buf, dtype=dtype).reshape(shape)

    def close(self):
        if getattr(self, "ptr", None):
            lib().gooey_b200_host_free(self.ptr)
            self.ptr = None

    __del__ = close
