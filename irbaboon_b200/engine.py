"""ctypes binding of libirb_b200.so (include/irb_b200.h) -- the host-side driver used by tests and bench.py.

This module is plumbing: it loads the C-ABI library, turns its status codes into exceptions and moves numpy
arrays (or raw device pointers from torch) across the boundary.  All arithmetic happens in the CUDA library;
there is no CPU fallback here -- if the library is missing, or no B200 is visible, calls raise.
"""
import ctypes
import os
import weakref

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("IRB_LIB") or os.path.join(_HERE, "libirb_b200.so")      # IRB_LIB: another build of the library (A/B measurements)
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "irb_b200.h")
BENCH_HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "irb_b200_bench.h")      # measurement aids, not the drop-in boundary

_f32p = ctypes.POINTER(ctypes.c_float)
_vp = ctypes.c_void_p
_lib = None


class IrbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("irb status %d: %s" % (code, msg))
        self.code = code


IRB_ERR_ARG, IRB_ERR_LAYOUT, IRB_ERR_CUDA, IRB_ERR_STATE = -1, -2, -3, -4

_SIGS = {
    "irb_last_error": (ctypes.c_char_p, []),
    "irb_version": (ctypes.c_int, []),
    "irb_device_count": (ctypes.c_int, []),
    "irb_set_device": (ctypes.c_int, [ctypes.c_int]),
    "irb_max_block_size": (ctypes.c_int, []),
    "irb_host_alloc": (_vp, [ctypes.c_size_t]),
    "irb_host_alloc_write_combined": (_vp, [ctypes.c_size_t]),
    "irb_host_free": (None, [_vp]),
    "irb_engine_create": (ctypes.c_int, [ctypes.POINTER(_vp)] + [ctypes.c_int] * 5),
    "irb_engine_destroy": (ctypes.c_int, [_vp]),
    "irb_engine_set_stream": (ctypes.c_int, [_vp, _vp]),
    "irb_engine_set_ir": (ctypes.c_int, [_vp, ctypes.c_int, _vp, _vp, ctypes.c_int]),
    "irb_engine_stage_ir": (ctypes.c_int, [_vp, ctypes.c_int, _vp, _vp, ctypes.c_int, ctypes.c_int]),
    "irb_engine_set_irs": (ctypes.c_int, [_vp, ctypes.c_int, _vp, _vp, _vp, ctypes.c_longlong, _vp]),
    "irb_engine_stage_irs": (ctypes.c_int, [_vp, ctypes.c_int, _vp, _vp, _vp, ctypes.c_longlong, _vp, ctypes.c_int]),
    "irb_engine_mac_plan": (ctypes.c_int, [_vp, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int)]),
    "irb_engine_set_mac_split": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int]),
    "irb_engine_set_fused_step": (ctypes.c_int, [_vp, ctypes.c_int]),
    "irb_engine_bind": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int]),
    "irb_engine_tile_channels": (ctypes.c_int, [_vp]),
    "irb_engine_reset": (ctypes.c_int, [_vp]),
    "irb_engine_set_active_channels": (ctypes.c_int, [_vp, ctypes.c_int]),
    "irb_engine_active_channels": (ctypes.c_int, [_vp]),
    "irb_engine_process": (ctypes.c_int, [_vp, _vp, _vp, ctypes.c_int]),
    "irb_engine_process_callback": (ctypes.c_int, [_vp, _vp, _vp, ctypes.c_int]),
    "irb_engine_process_device": (ctypes.c_int, [_vp, _vp, _vp, ctypes.c_int]),
    "irb_engine_synchronize": (ctypes.c_int, [_vp]),
    "irb_engine_submit": (ctypes.c_int, [_vp, _vp, _vp, ctypes.c_int]),
    "irb_engine_wait": (ctypes.c_int, [_vp]),
    "irb_engine_process_pcm": (ctypes.c_int, [_vp, _vp, ctypes.c_int, _vp, ctypes.c_int, ctypes.c_int]),
    "irb_engine_submit_pcm": (ctypes.c_int, [_vp, _vp, ctypes.c_int, _vp, ctypes.c_int, ctypes.c_int]),
    "irb_engine_process_device_pcm": (ctypes.c_int, [_vp, _vp, ctypes.c_int, _vp, ctypes.c_int, ctypes.c_int]),
    "irb_engine_set_timing": (ctypes.c_int, [_vp, ctypes.c_int]),
    "irb_engine_get_timings": (ctypes.c_int, [_vp, _vp, _vp, ctypes.c_int]),
    "irb_engine_state_bytes": (ctypes.c_size_t, [_vp]),
    "irb_engine_fft_size": (ctypes.c_int, [_vp]),
    "irb_engine_partitions": (ctypes.c_int, [_vp, ctypes.c_int]),
    "irb_engine_read_ir_spectrum": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, _vp]),
    "irb_engine_read_fdl_spectrum": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, _vp]),
    "irb_engine_launch_count": (ctypes.c_longlong, [_vp]),
    "irb_launch_count": (ctypes.c_longlong, []),
    "irb_release_workspace": (ctypes.c_size_t, []),
    "irb_last_compute_ms": (ctypes.c_double, []),
    "irb_engine_create_matrix": (ctypes.c_int, [ctypes.POINTER(_vp)] + [ctypes.c_int] * 7),
    "irb_engine_bind_matrix": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_int)]),
    "irb_group_create": (ctypes.c_int, [ctypes.POINTER(_vp), ctypes.POINTER(ctypes.c_int)] + [ctypes.c_int] * 5),
    "irb_group_destroy": (ctypes.c_int, [_vp]),
    "irb_group_device_count": (ctypes.c_int, [_vp]),
    "irb_group_channel_range": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int)]),
    "irb_group_set_ir": (ctypes.c_int, [_vp, ctypes.c_int, _vp, _vp, ctypes.c_int]),
    "irb_group_stage_ir": (ctypes.c_int, [_vp, ctypes.c_int, _vp, _vp, ctypes.c_int, ctypes.c_int]),
    "irb_group_set_irs": (ctypes.c_int, [_vp, ctypes.c_int, _vp, _vp, _vp, ctypes.c_longlong, _vp]),
    "irb_group_stage_irs": (ctypes.c_int, [_vp, ctypes.c_int, _vp, _vp, _vp, ctypes.c_longlong, _vp, ctypes.c_int]),
    "irb_group_bind": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int]),
    "irb_group_reset": (ctypes.c_int, [_vp]),
    "irb_group_process": (ctypes.c_int, [_vp, _vp, _vp, ctypes.c_int]),
    "irb_group_process_pcm": (ctypes.c_int, [_vp, _vp, ctypes.c_int, _vp, ctypes.c_int, ctypes.c_int]),
    "irb_group_state_bytes": (ctypes.c_size_t, [_vp]),
    "irb_convolve_periodic": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, _vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp]),
    "irb_convolve_nonperiodic": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, _vp, ctypes.c_int, ctypes.c_int, _vp]),
    "irb_convolve_batch": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, _vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp]),
    "irb_convolve_batch_device": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, _vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp]),
    "irb_deconvolve": (ctypes.c_int, [_vp, ctypes.c_int, _vp, ctypes.c_int, ctypes.c_double, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp]),
    "irb_deconvolve_batch": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, _vp, ctypes.c_int, ctypes.c_double, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp]),
    "irb_deconvolve_batch_device": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, _vp, ctypes.c_int, ctypes.c_double, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp]),
    "irb_ir_chop_batch_device": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_int, ctypes.c_int, ctypes.c_float, _vp, _vp]),
    "irb_deconvolve_chop_batch": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, _vp, ctypes.c_int, ctypes.c_double, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                                 ctypes.c_int, ctypes.c_float, ctypes.c_int, ctypes.c_int, ctypes.c_float, _vp, _vp]),
    "irb_invert_filter": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, _vp]),
    "irb_averaging_filter": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_double, ctypes.c_double, ctypes.c_int, ctypes.c_int, ctypes.c_int]),
    "irb_fft_transform": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp]),
    "irb_fft_inv_transform": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, _vp]),
    "irb_ir_to_real_fft_raw": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, _vp]),
    "irb_ess_generate": (ctypes.c_int, [ctypes.c_double] * 5 + [ctypes.c_int, _vp, ctypes.c_int]),
}

# include/irb_b200_bench.h: bench-only entry points (irbaboon_b200/csrc/irb_benchaids.cu)
_BENCH_SIGS = {
    "irbx_set_tuning": (ctypes.c_int, [ctypes.c_char_p, ctypes.c_int]),
    "irbx_get_tuning": (ctypes.c_int, [ctypes.c_char_p]),
    "irbx_engine_mac_only_device": (ctypes.c_int, [_vp, _vp]),
    "irbx_engine_set_stamps": (ctypes.c_int, [_vp, _vp]),
    "irbx_engine_ir_copies": (ctypes.c_int, [_vp]),
    "irbx_hbm_read_probe": (ctypes.c_int, [ctypes.c_size_t, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_double)]),
    "irbx_copy_probe_create": (ctypes.c_int, [ctypes.POINTER(_vp), ctypes.c_int, ctypes.c_size_t, ctypes.c_int]),
    "irbx_copy_probe_run": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_size_t, ctypes.POINTER(ctypes.c_double)]),
    "irbx_copy_probe_destroy": (ctypes.c_int, [_vp]),
}


def lib():
    """Load libirb_b200.so; raises if it has not been built (python -m irbaboon_b200.build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise FileNotFoundError(LIB_PATH + " is missing: run `python -m irbaboon_b200.build` (there is no CPU fallback)")
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in list(_SIGS.items()) + list(_BENCH_SIGS.items()):
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def _ck(rc):
    if rc < 0:
        raise IrbError(rc, lib().irb_last_error().decode("utf-8", "replace"))
    return rc


def _ptr(a):
    return a.ctypes.data_as(_vp)


# irb_sample_format (include/irb_b200.h): the streaming engine's block arrays in float32, int16 or packed little-endian 24-bit PCM
IRB_SAMPLE_F32, IRB_SAMPLE_S16, IRB_SAMPLE_S24 = 0, 1, 2
SAMPLE_FORMATS = {"f32": IRB_SAMPLE_F32, "s16": IRB_SAMPLE_S16, "s24": IRB_SAMPLE_S24}
_FORMAT_DTYPE = {IRB_SAMPLE_F32: np.float32, IRB_SAMPLE_S16: np.int16, IRB_SAMPLE_S24: np.uint8}


def sample_format(name):
    """"f32" | "s16" | "s24" -> irb_sample_format code."""
    f = SAMPLE_FORMATS.get(name)
    if f is None:
        raise ValueError("sample format %r: expected one of %s" % (name, ", ".join(SAMPLE_FORMATS)))
    return f


def _process_call(h, x, fin, out, fout, nb, group=False):
    """irb_engine_process_pcm / irb_group_process_pcm.  On the one-block latency path the binding's own microseconds show:
    float in and out take the float entry point (two ctypes arguments fewer), and the addresses go over as plain integers
    (a.ctypes.data costs half of a.ctypes.data_as)."""
    L = lib()
    if fin == IRB_SAMPLE_F32 and fout == IRB_SAMPLE_F32:
        return _ck((L.irb_group_process if group else L.irb_engine_process)(h, x.ctypes.data, out.ctypes.data, nb))
    return _ck((L.irb_group_process_pcm if group else L.irb_engine_process_pcm)(h, x.ctypes.data, fin, out.ctypes.data, fout, nb))


def _pcm_input(x, block_size):
    """A block array and its sample format, taken from its dtype: int16 is 16-bit PCM, uint8 with a last axis of 3*block_size
    bytes is packed 24-bit PCM, anything else is converted to float32.  -> (C-contiguous array, format, shape in samples)"""
    x = np.asarray(x)
    c = x.dtype.char
    if c == "h":
        x = np.ascontiguousarray(x)
        return x, IRB_SAMPLE_S16, x.shape
    if c == "B":
        if x.ndim < 1 or x.shape[-1] != 3 * block_size:
            raise ValueError("a uint8 (packed 24-bit) block array needs a last axis of 3*B = %d bytes, got shape %r" % (3 * block_size, x.shape))
        x = np.ascontiguousarray(x)
        return x, IRB_SAMPLE_S24, x.shape[:-1] + (block_size,)
    x = np.ascontiguousarray(x, np.float32)
    return x, IRB_SAMPLE_F32, x.shape


def _pcm_output(shape, fmt, out):
    """The output array for `shape` samples ([..][B]) in format fmt: a new one, or `out` once it is checked (its raw pointer goes
    to the library).  Packed 24-bit arrays are uint8 with a last axis of 3*B."""
    dt = _FORMAT_DTYPE[fmt]
    shp = tuple(shape[:-1]) + (3 * shape[-1],) if fmt == IRB_SAMPLE_S24 else shape
    if out is None:
        return np.empty(shp, dt)
    if not (isinstance(out, np.ndarray) and out.dtype == dt and out.shape == shp and out.flags.c_contiguous and out.flags.writeable):
        raise ValueError("out must be a writable C-contiguous %s array of shape %r" % (np.dtype(dt).name, shp))
    return out


def _planar(a):
    a = np.ascontiguousarray(a, dtype=np.float32)
    return a[None, :] if a.ndim == 1 else a


def _ir_rows(ir_ids, taps, n_taps, right, ld, allow_ptr=True):
    """The arguments of irb_*_set_irs / _stage_irs: -> (n, ids, taps, right, ld, n_taps, arrays to keep alive).  taps / right are
    host arrays [n][ld] (a 1-D array is one row), or raw device pointers (ints, e.g. tensor.data_ptr()) with ld given."""
    ids = np.ascontiguousarray(np.asarray(ir_ids, dtype=np.int64).reshape(-1), np.int32)
    if not np.array_equal(ids, np.asarray(ir_ids, dtype=np.int64).reshape(-1)):
        raise ValueError("ir_ids do not fit int32")
    n = ids.size
    if n < 1:
        raise ValueError("ir_ids is empty: a load takes at least one row")
    keep = [ids]
    if isinstance(taps, (int, np.integer)):
        if not allow_ptr:
            raise ValueError("a group loads from host arrays only, not from a pointer")
        if ld is None:
            raise ValueError("ld is needed with a pointer taps")
        if right is not None and not isinstance(right, (int, np.integer)):
            raise ValueError("right must be a pointer too when taps is one")
        if not taps or (right is not None and not right):
            raise ValueError("null taps or right pointer")
        tp, rp, ld = _vp(int(taps)), (_vp(int(right)) if right is not None else None), int(ld)
    else:
        t = np.ascontiguousarray(taps, np.float32)
        t = t[None, :] if t.ndim == 1 else t
        if t.ndim != 2 or t.shape[0] != n:
            raise ValueError("taps must be [n][ld] with one row per IR id (%d), got shape %r" % (n, np.shape(taps)))
        if ld is not None and int(ld) != t.shape[1]:
            raise ValueError("ld=%r contradicts taps of shape %r" % (ld, t.shape))
        ld = t.shape[1]
        keep.append(t)
        tp, rp = _ptr(t), None
        if right is not None:
            if isinstance(right, (int, np.integer)):
                raise ValueError("right must be a host array when taps is one")
            r = np.ascontiguousarray(right, np.float32)
            r = r[None, :] if r.ndim == 1 else r
            if r.shape != t.shape:
                raise ValueError("right must have the shape of taps %r, got %r" % (t.shape, r.shape))
            keep.append(r)
            rp = _ptr(r)
    nt = None
    if n_taps is not None:
        nt = np.ascontiguousarray(np.asarray(n_taps, dtype=np.int64).reshape(-1), np.int64)
        if nt.size != n:
            raise ValueError("n_taps needs one entry per row (%d), got %d" % (n, nt.size))
        if nt.min() < -2**31 or nt.max() >= 2**31:
            raise ValueError("n_taps do not fit int32")
        nt = nt.astype(np.int32)
        keep.append(nt)
    return n, _ptr(ids), tp, rp, ld, (_ptr(nt) if nt is not None else None), keep


def device_count():
    return _ck(lib().irb_device_count())


def set_device(device):
    _ck(lib().irb_set_device(int(device)))


def launch_count():
    return lib().irb_launch_count()


def release_workspace():
    """Return the offline functions' recycled device scratch buffers to the driver; -> bytes released."""
    return lib().irb_release_workspace()


def last_compute_ms():
    return lib().irb_last_compute_ms()


def hbm_read_probe(nbytes, iters=5, write_every=0, store_kind=0):
    """GB/s of a read-only streaming kernel over nbytes of device memory (measurement aid, irb_b200_bench.h)."""
    g = ctypes.c_double(0.0)
    _ck(lib().irbx_hbm_read_probe(int(nbytes), int(iters), int(write_every), int(store_kind), ctypes.byref(g)))
    return g.value


def set_tuning(name, value):
    """Launch-policy knob of the library by name (irb_b200_bench.h; A/B measurements and tests only)."""
    _ck(lib().irbx_set_tuning(name.encode(), int(value)))


def get_tuning(name):
    return _ck(lib().irbx_get_tuning(name.encode()))


class CopyProbe:
    """Copy-only host<->device ceiling (irb_b200_bench.h): `nbytes` per direction, no kernels."""

    def __init__(self, nbytes, host_mode=0, device=0):
        self._h = _vp()
        _ck(lib().irbx_copy_probe_create(ctypes.byref(self._h), int(device), int(nbytes), int(host_mode)))
        self.nbytes = int(nbytes)

    def run(self, iters=8, direction=3, chunk_bytes=0):
        """-> wall seconds of `iters` rounds (direction 1: H2D, 2: D2H, 3: both at once)."""
        s = ctypes.c_double(0.0)
        _ck(lib().irbx_copy_probe_run(self._h, int(iters), int(direction), int(chunk_bytes), ctypes.byref(s)))
        return s.value

    def close(self):
        if self._h:
            lib().irbx_copy_probe_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class _PinnedOwner:
    """Owns one cudaMallocHost block: the block is released when the last numpy view of it is collected, or by pinned_free."""

    def __init__(self, ptr):
        self.ptr = ptr
        self._fin = weakref.finalize(self, lib().irb_host_free, ptr)

    def free(self):
        self._fin()


def pinned_empty(shape, dtype=np.float32, write_combined=False):
    """numpy array over cudaMallocHost memory (write_combined: for input the host only writes; never read it back from the CPU).
    The memory goes back when the array (and every view of it) is collected; pinned_free(arr) releases it at once (the array
    must not be touched afterwards)."""
    n = int(np.prod(shape)) * np.dtype(dtype).itemsize
    p = lib().irb_host_alloc_write_combined(n) if write_combined else lib().irb_host_alloc(n)
    if not p:
        raise IrbError(IRB_ERR_CUDA, lib().irb_last_error().decode())
    owner = _PinnedOwner(p)
    buf = (ctypes.c_char * max(n, 1)).from_address(p)
    buf._irb_owner = owner                      # the ctypes buffer is the base of every numpy view: it keeps the owner alive
    arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
    _PINNED[p] = weakref.ref(owner)
    return arr


_PINNED = {}


def pinned_free(arr):
    ref = _PINNED.pop(arr.__array_interface__["data"][0], None)
    owner = ref() if ref else None
    if owner is not None:
        owner.free()


def convolve_periodic(x, h, block_size=256):
    """fp::convolution::convolvePeriodic (fp/convolution.cpp:14-242): planar [ch][n] float32 in and out."""
    x, h = _planar(x), _planar(h)
    out = np.zeros((x.shape[0], x.shape[1] + h.shape[1] - 1), np.float32)
    rc = lib().irb_convolve_periodic(_ptr(x), x.shape[0], x.shape[1], _ptr(h), h.shape[0], h.shape[1], int(block_size), _ptr(out))
    if rc == IRB_ERR_LAYOUT:
        return out                      # the reference prints a DBG line and returns the cleared buffer
    _ck(rc)
    return out


def next_pow2(x):
    """tools::nextPowerOfTwo (fp/tools.cpp:189-196): x itself when already a power of two."""
    if x > 0 and (x & (x - 1)) == 0:
        return x
    r = 1
    while r <= x:
        r *= 2
    return r


def convolve_nonperiodic(x, h):
    """fp::convolution::convolveNonPeriodic (fp/convolution.cpp:246-347)."""
    x, h = _planar(x), _planar(h)
    out = np.zeros((x.shape[0], x.shape[1] + h.shape[1] - 1), np.float32)
    rc = lib().irb_convolve_nonperiodic(_ptr(x), x.shape[0], x.shape[1], _ptr(h), h.shape[0], h.shape[1], _ptr(out))
    if rc == IRB_ERR_LAYOUT:
        return np.zeros_like(x)         # the reference returns a cleared copy of the input (fp/convolution.cpp:271-275)
    _ck(rc)
    return out


def _window(len_x, len_h, out_offset, out_len):
    """(out_offset, out_len) of a batched convolution's window; out_len None: the rest of the len_x + len_h - 1 samples"""
    full = int(len_x) + int(len_h) - 1
    return int(out_offset), full - int(out_offset) if out_len is None else int(out_len)


def convolve_batch(x, h, out_offset=0, out_len=None, out=None):
    """irb_convolve_batch: signals x[batch][len_x], each convolved with h[len_h] (shared) or h[1 | batch][len_h] (h[b] for signal
    b) -> out[batch][out_len], the window [out_offset, out_offset + out_len) of every len_x + len_h - 1 sample result (default: all
    of it).  `out` may be a C-contiguous float32 array of that shape (pinned memory: eng.pinned_empty)."""
    x = np.ascontiguousarray(x, np.float32)
    x = x[None, :] if x.ndim == 1 else x
    h = np.ascontiguousarray(h, np.float32)
    h = h[None, :] if h.ndim == 1 else h
    if x.ndim != 2 or h.ndim != 2:
        raise ValueError("x must be [batch][len_x] and h [len_h] or [1 | batch][len_h], got %r and %r" % (x.shape, h.shape))
    off, n = _window(x.shape[1], h.shape[1], out_offset, out_len)
    if out is None:
        out = np.empty((x.shape[0], max(n, 0)), np.float32)
    elif not (isinstance(out, np.ndarray) and out.dtype == np.float32 and out.shape == (x.shape[0], n) and out.flags.c_contiguous and out.flags.writeable):
        raise ValueError("out must be a writable C-contiguous float32 array of shape %r" % ((x.shape[0], n),))
    _ck(lib().irb_convolve_batch(_ptr(x), x.shape[0], x.shape[1], _ptr(h), h.shape[0], h.shape[1], off, n, _ptr(out)))
    return out


def convolve_batch_device(x_ptr, batch, len_x, h, out_ptr, len_h=None, h_batch=None, out_offset=0, out_len=None):
    """irb_convolve_batch_device: x and the result are raw DEVICE pointers ([batch][len_x] / [batch][out_len] float32).  h is either
    a raw pointer (an int, e.g. tensor.data_ptr(), to device or host memory) with len_h given and h_batch 1 (the default) or batch,
    or a host array-like ([len_h] or [h_batch][len_h]) whose shape gives both; len_h / h_batch that contradict it are an error."""
    if isinstance(h, (int, np.integer)):
        if len_h is None:
            raise ValueError("len_h is needed with a pointer h")
        hp = _vp(int(h))
        h_batch = 1 if h_batch is None else h_batch
    else:
        ha = np.asarray(h)
        if ha.ndim not in (1, 2):
            raise ValueError("h must be [len_h] or [h_batch][len_h], got shape %r" % (ha.shape,))
        ha = np.ascontiguousarray(ha[None, :] if ha.ndim == 1 else ha, np.float32)
        if (len_h is not None and int(len_h) != ha.shape[1]) or (h_batch is not None and int(h_batch) != ha.shape[0]):
            raise ValueError("len_h=%r, h_batch=%r contradict h of shape %r" % (len_h, h_batch, ha.shape))
        h_batch, len_h, hp = ha.shape[0], ha.shape[1], _ptr(ha)
    off, n = _window(len_x, len_h, out_offset, out_len)
    _ck(lib().irb_convolve_batch_device(_vp(int(x_ptr)), int(batch), int(len_x), hp, int(h_batch), int(len_h), off, n, _vp(int(out_ptr))))


def deconvolve(num, den, sample_rate=48000.0, smoothing=True, include_phase=True, include_amplitude=True):
    """fp::convolution::deconvolve (fp/convolution.cpp:351-403); channel 0 of each input is used.  -> [1][N]"""
    num, den = np.ascontiguousarray(_planar(num)[0]), np.ascontiguousarray(_planar(den)[0])
    N = next_pow2(max(len(num), len(den)))
    out = np.zeros((1, N), np.float32)
    _ck(lib().irb_deconvolve(_ptr(num), len(num), _ptr(den), len(den), float(sample_rate), int(smoothing), int(include_phase), int(include_amplitude), _ptr(out)))
    return out


def deconvolve_batch(nums, den, sample_rate=48000.0, smoothing=False, include_phase=True, include_amplitude=True, out=None):
    """`batch` captures nums[batch][len] divided by one sweep den[len_den] -> [batch][N]."""
    nums = np.ascontiguousarray(nums, np.float32)
    den = np.ascontiguousarray(den, np.float32).reshape(-1)
    N = next_pow2(max(nums.shape[1], len(den)))
    if out is None:
        out = np.zeros((nums.shape[0], N), np.float32)
    assert out.shape == (nums.shape[0], N) and out.dtype == np.float32 and out.flags.c_contiguous
    _ck(lib().irb_deconvolve_batch(_ptr(nums), nums.shape[0], nums.shape[1], _ptr(den), len(den), float(sample_rate), int(smoothing), int(include_phase),
                                   int(include_amplitude), _ptr(out)))
    return out


def deconvolve_batch_device(nums_ptr, batch, len_num, den, out_ptr, sample_rate=48000.0, smoothing=False, include_phase=True, include_amplitude=True):
    """irb_deconvolve_batch_device: captures and results are raw DEVICE pointers ([batch][len_num] / [batch][N] float32)."""
    den = np.ascontiguousarray(den, np.float32).reshape(-1)
    _ck(lib().irb_deconvolve_batch_device(_vp(int(nums_ptr)), int(batch), int(len_num), _ptr(den), len(den), float(sample_rate), int(smoothing), int(include_phase),
                                          int(include_amplitude), _vp(int(out_ptr))))


def _check_chop(batch, length, ir_length):
    if int(batch) < 1 or int(length) < 1:
        raise ValueError("batch %r and row length %r must be at least 1" % (batch, length))
    if not 1 <= int(ir_length) <= int(length):
        raise ValueError("ir_length %r outside [1, %d]: the IR is cut from rows of %d samples" % (ir_length, int(length), int(length)))


def ir_chop_batch_device(x_ptr, batch, len, ir_length, out_ptr, threshold_db=-60.0, consecutive=50, normalize=True, goal_db=0.0, positions_ptr=None):
    """irb_ir_chop_batch_device: fp::ir::IRchop (+ fp::tools::normalize(goal_db)) of every row of x[batch][len] -> out[batch][ir_length];
    x_ptr, out_ptr and positions_ptr ([batch][2] int32 {peak index, start}, optional) are raw DEVICE pointers (ints)."""
    _check_chop(batch, len, ir_length)
    if not x_ptr or not out_ptr:
        raise ValueError("x_ptr and out_ptr must be device pointers")
    _ck(lib().irb_ir_chop_batch_device(_vp(int(x_ptr)), int(batch), int(len), int(ir_length), float(threshold_db), int(consecutive), int(bool(normalize)),
                                       float(goal_db), _vp(int(out_ptr)), _vp(int(positions_ptr)) if positions_ptr else None))


def deconvolve_chop_batch(nums, den, ir_length, sample_rate=48000.0, smoothing=False, include_phase=True, include_amplitude=True, threshold_db=-60.0,
                          consecutive=50, normalize=True, goal_db=0.0, out=None, return_positions=False):
    """irb_deconvolve_chop_batch: deconvolve_batch(nums, den, ...) with every row cut by ir_chop_batch_device on the device
    -> out[batch][ir_length] (and, with return_positions, int32 [batch][2] {peak index, start})."""
    nums = np.ascontiguousarray(nums, np.float32)
    nums = nums[None, :] if nums.ndim == 1 else nums
    den = np.ascontiguousarray(den, np.float32).reshape(-1)
    if nums.ndim != 2 or len(den) < 1:
        raise ValueError("nums must be [batch][len_num] and den a non-empty [len_den], got %r and %r" % (nums.shape, den.shape))
    N = next_pow2(max(nums.shape[1], len(den)))
    _check_chop(nums.shape[0], N, ir_length)
    if out is None:
        out = np.empty((nums.shape[0], int(ir_length)), np.float32)
    elif not (isinstance(out, np.ndarray) and out.dtype == np.float32 and out.shape == (nums.shape[0], int(ir_length)) and out.flags.c_contiguous and out.flags.writeable):
        raise ValueError("out must be a writable C-contiguous float32 array of shape %r" % ((nums.shape[0], int(ir_length)),))
    pos = np.empty((nums.shape[0], 2), np.int32) if return_positions else None
    _ck(lib().irb_deconvolve_chop_batch(_ptr(nums), nums.shape[0], nums.shape[1], _ptr(den), len(den), float(sample_rate), int(smoothing), int(include_phase),
                                        int(include_amplitude), int(ir_length), float(threshold_db), int(consecutive), int(bool(normalize)), float(goal_db),
                                        _ptr(out), _ptr(pos) if pos is not None else None))
    return (out, pos) if return_positions else out


def invert_filter(x, sample_rate=48000):
    x = np.ascontiguousarray(_planar(x)[0])
    out = np.zeros((1, next_pow2(len(x))), np.float32)
    _ck(lib().irb_invert_filter(_ptr(x), len(x), int(sample_rate), _ptr(out)))
    return out


def averaging_filter(spec, octave_fraction, sample_rate, log_avg=True, include_phase=True, include_amplitude=True):
    s = _planar(spec).copy()
    _ck(lib().irb_averaging_filter(_ptr(s), s.shape[0], s.shape[1], float(octave_fraction), float(sample_rate), int(log_avg), int(include_phase), int(include_amplitude)))
    return s


def fft_transform(x, format_ampl_phase=False):
    x = _planar(x)
    N = next_pow2(x.shape[1])
    out = np.zeros((x.shape[0], 2 * N), np.float32)
    _ck(lib().irb_fft_transform(_ptr(x), x.shape[0], x.shape[1], int(format_ampl_phase), _ptr(out)))
    return out


def fft_inv_transform(spec):
    s = _planar(spec)
    out = np.zeros((s.shape[0], s.shape[1] // 2), np.float32)
    _ck(lib().irb_fft_inv_transform(_ptr(s), s.shape[0], s.shape[1], _ptr(out)))
    return out


def ir_to_real_fft_raw(x, part_size):
    """fp::ir::IRtoRealFFTRaw (fp/ir.cpp:106-147): packed partition spectra, (len/part + 1) * 2*part floats."""
    x = np.ascontiguousarray(_planar(x)[0])
    out = np.zeros((len(x) // part_size + 1) * 2 * part_size, np.float32)
    _ck(lib().irb_ir_to_real_fft_raw(_ptr(x), len(x), int(part_size), _ptr(out)))
    return out


def ess(duration_s, sample_rate, f1, f2, gain_db=0.0, inverse=False):
    """fp::ExpSineSweep::generate / generateInv in FP64 on the device -> float64 array."""
    n = _ck(lib().irb_ess_generate(duration_s, sample_rate, f1, f2, gain_db, int(inverse), None, 0))
    out = np.zeros(n, np.float64)
    _ck(lib().irb_ess_generate(duration_s, sample_rate, f1, f2, gain_db, int(inverse), _ptr(out), n))
    return out


class Engine:
    """Streaming UPOLA engine over n_channels independent stream-channels on one GPU."""

    def __init__(self, block_size, max_partitions, n_channels, n_irs=1, device=0):
        self._h = _vp()
        _ck(lib().irb_engine_create(ctypes.byref(self._h), int(device), int(block_size), int(max_partitions), int(n_channels), int(n_irs)))
        self.block_size, self.max_partitions, self.n_channels, self.n_irs, self.device = block_size, max_partitions, n_channels, n_irs, device
        self.fft_size = lib().irb_engine_fft_size(self._h)
        self.active_channels = n_channels

    def close(self):
        if self._h:
            lib().irb_engine_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def set_stream(self, cuda_stream):
        """cuda_stream: a cudaStream_t handle as int (0 = legacy default stream); None = the engine's own stream."""
        h = _vp(ctypes.c_size_t(-1).value) if cuda_stream is None else _vp(int(cuda_stream))
        _ck(lib().irb_engine_set_stream(self._h, h))

    def set_ir(self, ir_id, taps):
        """taps: [n] mono, or [2][n] stereo folded to (L+R)/2."""
        t = _planar(taps)
        if t.shape[0] == 1:
            _ck(lib().irb_engine_set_ir(self._h, int(ir_id), _ptr(t), None, t.shape[1]))
        elif t.shape[0] == 2:
            l, r = np.ascontiguousarray(t[0]), np.ascontiguousarray(t[1])
            _ck(lib().irb_engine_set_ir(self._h, int(ir_id), _ptr(l), _ptr(r), t.shape[1]))
        else:
            raise ValueError("IR must be mono or stereo")

    def stage_ir(self, ir_id, taps, n_partitions=0):
        """Round-robin IR switch (PluginProcessor.cpp:411-414,455-461): one partition re-transformed per block step."""
        t = _planar(taps)
        if t.shape[0] == 1:
            _ck(lib().irb_engine_stage_ir(self._h, int(ir_id), _ptr(t), None, t.shape[1], int(n_partitions)))
        elif t.shape[0] == 2:
            l, r = np.ascontiguousarray(t[0]), np.ascontiguousarray(t[1])
            _ck(lib().irb_engine_stage_ir(self._h, int(ir_id), _ptr(l), _ptr(r), t.shape[1], int(n_partitions)))
        else:
            raise ValueError("IR must be mono or stereo")

    def set_irs(self, ir_ids, taps, n_taps=None, right=None, ld=None):
        """Load n IRs in one call (irb_engine_set_irs): row j of taps ([n][ld] host float32, or a raw device pointer with ld
        given) holds n_taps[j] taps (default: ld) of IR ir_ids[j]; right (same kind) folds a stereo IR to (L+R)/2.  Row j's
        spectra are exactly those of set_ir on that row."""
        n, ids, tp, rp, ld, nt, _keep = _ir_rows(ir_ids, taps, n_taps, right, ld)
        _ck(lib().irb_engine_set_irs(self._h, n, ids, tp, rp, ld, nt))

    def stage_irs(self, ir_ids, taps, n_taps=None, right=None, ld=None, n_partitions=0):
        """stage_ir for n IRs in one call (irb_engine_stage_irs); arguments as set_irs."""
        n, ids, tp, rp, ld, nt, _keep = _ir_rows(ir_ids, taps, n_taps, right, ld)
        _ck(lib().irb_engine_stage_irs(self._h, n, ids, tp, rp, ld, nt, int(n_partitions)))

    def mac_plan(self):
        """(slots_kernel, split_in, cluster) of the next block step's MAC launch."""
        a, b, c = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
        _ck(lib().irb_engine_mac_plan(self._h, ctypes.byref(a), ctypes.byref(b), ctypes.byref(c)))
        return bool(a.value), b.value, c.value

    def set_mac_split(self, split_in=0, cluster=0):
        """Force how few-row launches split a row's partitions (0, 0 = automatic)."""
        _ck(lib().irb_engine_set_mac_split(self._h, int(split_in), int(cluster)))

    def set_fused_step(self, enable=True):
        """One launch per block step (forward transform inside the MAC kernel) or the two-launch form."""
        _ck(lib().irb_engine_set_fused_step(self._h, int(bool(enable))))

    def bind(self, chan_begin, chan_end, ir_id):
        _ck(lib().irb_engine_bind(self._h, int(chan_begin), int(chan_end), int(ir_id)))

    @property
    def tile_channels(self):
        return lib().irb_engine_tile_channels(self._h)

    def reset(self):
        _ck(lib().irb_engine_reset(self._h))

    def process(self, x, out=None, out_format="f32"):
        """x: host [n_blocks][n_channels][B] (or [n_channels][B]); returns the same shape.  The input format follows x's dtype
        (float32; int16 = 16-bit PCM; uint8 with a last axis of 3*B = packed 24-bit PCM), the output's is out_format
        ("f32", "s16" or "s24"); integer PCM is converted on the device (include/irb_b200.h, irb_sample_format)."""
        x, fin, shp = _pcm_input(x, self.block_size)
        nb = 1 if len(shp) == 2 else shp[0]
        if len(shp) not in (2, 3) or shp[-2:] != (self.active_channels, self.block_size):
            raise ValueError("input shape %r, expected [n_blocks][%d][%d]" % (x.shape, self.active_channels, self.block_size))
        fout = sample_format(out_format)
        out = _pcm_output(shp, fout, out)
        _process_call(self._h, x, fin, out, fout, nb)
        return out

    def process_callback(self, x):
        """Blocks of one plug-in callback, reference order (all forward FFTs first): host [n_blocks][n_channels][B]."""
        x = np.ascontiguousarray(x, np.float32)
        assert x.ndim == 3 and x.shape[1:] == (self.active_channels, self.block_size), x.shape
        out = np.empty(x.shape, np.float32)
        _ck(lib().irb_engine_process_callback(self._h, _ptr(x), _ptr(out), x.shape[0]))
        return out

    def submit(self, x, out, out_format="f32"):
        """Asynchronous multi-block call on pinned host arrays [n_blocks >= 2][n_channels][B]; pair with wait().  Formats as in
        process(); both arrays are used in place."""
        assert isinstance(x, np.ndarray) and x.flags.c_contiguous, "x must be a C-contiguous (pinned) array"
        x2, fin, shp = _pcm_input(x, self.block_size)
        assert x2 is x, "x must be float32, int16 or uint8: it is used in place"
        assert len(shp) == 3 and shp[1:] == (self.active_channels, self.block_size), x.shape
        fout = sample_format(out_format)
        _pcm_output(shp, fout, out)
        _ck(lib().irb_engine_submit_pcm(self._h, _ptr(x), fin, _ptr(out), fout, shp[0]))

    def wait(self):
        _ck(lib().irb_engine_wait(self._h))

    def process_device(self, in_ptr, out_ptr, n_blocks=1, in_format="f32", out_format="f32"):
        """Raw DEVICE pointers to [n_blocks][channels][B] elements of the given formats ("f32", "s16", "s24"); asynchronous."""
        _ck(lib().irb_engine_process_device_pcm(self._h, _vp(int(in_ptr)), sample_format(in_format), _vp(int(out_ptr)), sample_format(out_format), int(n_blocks)))

    def mac_only_device(self, acc_ptr):
        """bench-only (irb_b200_bench.h): the bare FDL multiply-accumulate into a device buffer"""
        _ck(lib().irbx_engine_mac_only_device(self._h, _vp(int(acc_ptr))))

    def set_stamps(self, dev_ptr):
        """bench-only: device array of 16 uint64 for the phase time stamps of the latency-path kernel (0 / None: off)"""
        _ck(lib().irbx_engine_set_stamps(self._h, _vp(int(dev_ptr or 0))))

    @property
    def ir_copies(self):
        """bench-only: identical copies of the IR spectra the engine keeps (every load writes all of them)"""
        return _ck(lib().irbx_engine_ir_copies(self._h))

    def set_active_channels(self, n_active):
        """Only channels [0, n_active) take part in the following block steps; I/O arrays are then [n_blocks][n_active][B]."""
        _ck(lib().irb_engine_set_active_channels(self._h, int(n_active)))
        self.active_channels = int(n_active)

    def set_timing(self, enable=True):
        _ck(lib().irb_engine_set_timing(self._h, int(bool(enable))))

    def timings(self, max_steps=16384):
        """(step_ms, mac_ms) device times of the steps recorded since set_timing(True)."""
        a = np.zeros(max_steps, np.float32)
        b = np.zeros(max_steps, np.float32)
        n = _ck(lib().irb_engine_get_timings(self._h, _ptr(a), _ptr(b), max_steps))
        return a[:n].copy(), b[:n].copy()

    def synchronize(self):
        _ck(lib().irb_engine_synchronize(self._h))

    def process_stream(self, x):
        """Convenience for tests: planar audio x[n_channels][n] -> y[n_channels][n] block by block
        (n is padded up to whole blocks with zeros and cut back)."""
        x = _planar(x)
        B = self.block_size
        n = x.shape[1]
        nb = (n + B - 1) // B
        xp = np.zeros((self.n_channels, nb * B), np.float32)
        xp[:, :n] = x
        blocks = np.ascontiguousarray(xp.reshape(self.n_channels, nb, B).transpose(1, 0, 2))
        y = self.process(blocks)
        return np.ascontiguousarray(y.transpose(1, 0, 2)).reshape(self.n_channels, nb * B)[:, :n]

    @property
    def state_bytes(self):
        return lib().irb_engine_state_bytes(self._h)

    def partitions(self, ir_id=0):
        return _ck(lib().irb_engine_partitions(self._h, int(ir_id)))

    @property
    def launches(self):
        return lib().irb_engine_launch_count(self._h)

    def ir_spectrum(self, ir_id, part):
        out = np.zeros(self.fft_size, np.float32)
        _ck(lib().irb_engine_read_ir_spectrum(self._h, int(ir_id), int(part), _ptr(out)))
        return out

    def fdl_spectrum(self, chan, age=0):
        out = np.zeros(self.fft_size, np.float32)
        _ck(lib().irb_engine_read_fdl_spectrum(self._h, int(chan), int(age), _ptr(out)))
        return out


class MatrixEngine(Engine):
    """IR-matrix streaming engine (irb_engine_create_matrix): n_groups groups of `ins` input channels, each producing `outs`
    output channels, out[g*outs + o] = sum_i conv(in[g*ins + i], IR ir_ids[i*outs + o]).  (ins, outs) = (1, 2) is mono -> stereo,
    (2, 2) true stereo with the IRs in the order LL, LR, RL, RR.  Every input keeps one delay line, read once per block step for
    all the IRs it feeds.  I/O arrays: in [n_blocks][n_groups*ins][B], out [n_blocks][n_groups*outs][B]."""

    def __init__(self, block_size, max_partitions, n_groups, ins, outs, n_irs=None, device=0):
        self._h = _vp()
        n_irs = ins * outs if n_irs is None else n_irs
        _ck(lib().irb_engine_create_matrix(ctypes.byref(self._h), int(device), int(block_size), int(max_partitions), int(n_groups), int(ins), int(outs), int(n_irs)))
        self.block_size, self.max_partitions, self.n_irs, self.device = block_size, max_partitions, n_irs, device
        self.n_groups, self.ins, self.outs = n_groups, ins, outs
        self.n_channels = self.active_channels = n_groups * ins         # input channels (FDL rows)
        self.n_outputs = n_groups * outs
        self.fft_size = lib().irb_engine_fft_size(self._h)

    def bind_matrix(self, group_begin, group_end, ir_ids):
        """groups [group_begin, group_end) convolve with the IRs ir_ids[i*outs + o] (input i -> output o)."""
        ids = [int(v) for v in ir_ids]
        if len(ids) != self.ins * self.outs:
            raise ValueError("ir_ids needs %d entries (ins*outs)" % (self.ins * self.outs))
        arr = (ctypes.c_int * len(ids))(*ids)
        _ck(lib().irb_engine_bind_matrix(self._h, int(group_begin), int(group_end), arr))

    def _out_shape(self, shape):
        return tuple(shape[:-2]) + (self.n_outputs, self.block_size)

    def process(self, x, out=None, out_format="f32"):
        """x: host [n_blocks][n_groups*ins][B] (or [n_groups*ins][B]) -> [n_blocks][n_groups*outs][B].  Formats as in
        Engine.process."""
        x, fin, ishp = _pcm_input(x, self.block_size)
        if len(ishp) not in (2, 3) or ishp[-2:] != (self.n_channels, self.block_size):
            raise ValueError("input shape %r, expected [n_blocks][%d][%d]" % (x.shape, self.n_channels, self.block_size))
        nb = 1 if len(ishp) == 2 else ishp[0]
        fout = sample_format(out_format)
        out = _pcm_output(self._out_shape(ishp), fout, out)
        _process_call(self._h, x, fin, out, fout, nb)
        return out

    def submit(self, x, out, out_format="f32"):
        """Asynchronous multi-block call on pinned host arrays (in [n_blocks >= 2][n_groups*ins][B], out [..][n_groups*outs][B]).
        Formats as in Engine.process."""
        assert isinstance(x, np.ndarray) and x.flags.c_contiguous, "x must be a C-contiguous (pinned) array"
        x2, fin, ishp = _pcm_input(x, self.block_size)
        assert x2 is x, "x must be float32, int16 or uint8: it is used in place"
        assert len(ishp) == 3 and ishp[1:] == (self.n_channels, self.block_size), x.shape
        fout = sample_format(out_format)
        _pcm_output(self._out_shape(ishp), fout, out)
        _ck(lib().irb_engine_submit_pcm(self._h, _ptr(x), fin, _ptr(out), fout, ishp[0]))

    def process_stream(self, x):
        """Planar inputs x[n_groups*ins][n] -> outputs y[n_groups*outs][n], block by block (zero-padded to whole blocks)."""
        x = _planar(x)
        B, n = self.block_size, x.shape[1]
        nb = (n + B - 1) // B
        xp = np.zeros((self.n_channels, nb * B), np.float32)
        xp[:, :n] = x
        y = self.process(np.ascontiguousarray(xp.reshape(self.n_channels, nb, B).transpose(1, 0, 2)))
        return np.ascontiguousarray(y.transpose(1, 0, 2)).reshape(self.n_outputs, nb * B)[:, :n]


class Group:
    """Several GPUs driven from one process: channels sharded by contiguous tile-aligned ranges (irb_group_*).
    n_irs > 0: shared IRs replicated on every device; n_irs == 0: one private IR per channel, living on its device."""

    def __init__(self, devices, block_size, max_partitions, n_channels, n_irs=1):
        self._h = _vp()
        devs = (ctypes.c_int * len(devices))(*[int(d) for d in devices])
        _ck(lib().irb_group_create(ctypes.byref(self._h), devs, len(devices), int(block_size), int(max_partitions), int(n_channels), int(n_irs)))
        self.block_size, self.n_channels, self.n_irs = block_size, n_channels, n_irs

    def close(self):
        if self._h:
            lib().irb_group_destroy(self._h)
            self._h = _vp()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def ranges(self):
        out = []
        for i in range(_ck(lib().irb_group_device_count(self._h))):
            b, e = ctypes.c_int(), ctypes.c_int()
            _ck(lib().irb_group_channel_range(self._h, i, ctypes.byref(b), ctypes.byref(e)))
            out.append((b.value, e.value))
        return out

    def set_ir(self, ir_id, taps):
        t = np.ascontiguousarray(_planar(taps)[0])
        _ck(lib().irb_group_set_ir(self._h, int(ir_id), _ptr(t), None, len(t)))

    def stage_ir(self, ir_id, taps, n_partitions=0):
        t = np.ascontiguousarray(_planar(taps)[0])
        _ck(lib().irb_group_stage_ir(self._h, int(ir_id), _ptr(t), None, len(t), int(n_partitions)))

    def set_irs(self, ir_ids, taps, n_taps=None, right=None):
        """irb_group_set_irs: host arrays only (taps / right [n][ld] float32); private-IR groups: ir_ids are channels."""
        n, ids, tp, rp, ld, nt, _keep = _ir_rows(ir_ids, taps, n_taps, right, None, allow_ptr=False)
        _ck(lib().irb_group_set_irs(self._h, n, ids, tp, rp, ld, nt))

    def stage_irs(self, ir_ids, taps, n_taps=None, right=None, n_partitions=0):
        """irb_group_stage_irs: host arrays only, as set_irs."""
        n, ids, tp, rp, ld, nt, _keep = _ir_rows(ir_ids, taps, n_taps, right, None, allow_ptr=False)
        _ck(lib().irb_group_stage_irs(self._h, n, ids, tp, rp, ld, nt, int(n_partitions)))

    def bind(self, chan_begin, chan_end, ir_id):
        _ck(lib().irb_group_bind(self._h, int(chan_begin), int(chan_end), int(ir_id)))

    def reset(self):
        _ck(lib().irb_group_reset(self._h))

    def process(self, x, out=None, out_format="f32"):
        """Host [n_blocks][n_channels][B] for all channels; formats as in Engine.process."""
        x, fin, shp = _pcm_input(x, self.block_size)
        nb = 1 if len(shp) == 2 else shp[0]
        assert shp[-2:] == (self.n_channels, self.block_size), x.shape
        fout = sample_format(out_format)
        out = _pcm_output(shp, fout, out)
        _process_call(self._h, x, fin, out, fout, nb, group=True)
        return out

    @property
    def state_bytes(self):
        return lib().irb_group_state_bytes(self._h)


def unpack_spectrum(packed):
    """packed M complex (bin 0 = {Re X[0], Re X[M]}) -> M+1 complex bins."""
    p = np.asarray(packed, np.float32)
    M = p.size // 2
    z = (p[0::2] + 1j * p[1::2]).astype(np.complex64)
    out = np.zeros(M + 1, np.complex64)
    out[1:M] = z[1:]
    out[0] = z[0].real
    out[M] = z[0].imag
    return out
