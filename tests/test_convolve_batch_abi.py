"""CPU: the batched linear convolution (irb_convolve_batch, irb_convolve_batch_device) rejects every bad argument with
IRB_ERR_ARG before it touches a device, and the inverse line-FFT kernels keep their registers and spill no more than before the
windowed copy (k_line_fft_win) existed, which itself keeps the same budget."""
import ctypes
import re
import subprocess

import numpy as np
import pytest

_FNS = ("irb_convolve_batch", "irb_convolve_batch_device")
_BUF = ctypes.create_string_buffer(4096)
_P = ctypes.cast(_BUF, ctypes.c_void_p)

# (x, batch, len_x, h, h_batch, len_h, out_offset, out_len, out) -> the word irb_last_error() carries
_BAD = [
    ((None, 1, 10, _P, 1, 5, 0, 14, _P), b"null"),
    ((_P, 1, 10, None, 1, 5, 0, 14, _P), b"null"),
    ((_P, 1, 10, _P, 1, 5, 0, 14, None), b"null"),
    ((_P, 0, 10, _P, 1, 5, 0, 14, _P), b"empty"),
    ((_P, -3, 10, _P, 1, 5, 0, 14, _P), b"empty"),
    ((_P, 1, 0, _P, 1, 5, 0, 4, _P), b"empty"),
    ((_P, 1, 10, _P, 1, 0, 0, 9, _P), b"empty"),
    ((_P, 2, 10, _P, 3, 5, 0, 14, _P), b"h_batch"),
    ((_P, 2, 10, _P, 0, 5, 0, 14, _P), b"h_batch"),
    ((_P, 3, 10, _P, 2, 5, 0, 14, _P), b"h_batch"),
    ((_P, 1, 10, _P, 1, 5, -1, 14, _P), b"window"),
    ((_P, 1, 10, _P, 1, 5, 0, 15, _P), b"window"),
    ((_P, 1, 10, _P, 1, 5, 13, 2, _P), b"window"),
    ((_P, 1, 10, _P, 1, 5, 14, 1, _P), b"window"),
    ((_P, 1, 10, _P, 1, 5, 3, 0, _P), b"window"),
    ((_P, 1, 10, _P, 1, 5, 3, -2, _P), b"window"),
    ((_P, 1, 10, _P, 1, 5, 2147483647, 2147483647, _P), b"window"),
    ((_P, 1, 1 << 22, _P, 1, 2, 0, 1, _P), b"2^22"),
    ((_P, 4, 3 << 21, _P, 4, 3 << 21, 0, 1, _P), b"2^22"),
]


@pytest.mark.parametrize("fn", _FNS)
@pytest.mark.parametrize("args,word", _BAD, ids=[str(i) for i in range(len(_BAD))])
def test_bad_arguments_are_rejected_without_a_device(eng, fn, args, word):
    L = eng.lib()
    assert getattr(L, fn)(*args) == eng.IRB_ERR_ARG
    assert word in L.irb_last_error()


@pytest.mark.parametrize("fn", _FNS)
def test_the_largest_result_is_accepted(eng, fn):
    """2^22 samples exactly is the top of the range: the call gets past the checks (and fails only for want of a GPU)."""
    try:
        if eng.device_count() > 0:
            pytest.skip("a GPU is visible")
    except eng.IrbError:
        pass
    L = eng.lib()
    rc = getattr(L, fn)(_P, 1, (1 << 22) - 1, _P, 1, 2, (1 << 22) - 1, 1, _P)
    assert rc == eng.IRB_ERR_CUDA, (rc, L.irb_last_error())


def test_python_window_and_shapes(eng):
    assert eng._window(10, 5, 0, None) == (0, 14)
    assert eng._window(10, 5, 3, None) == (3, 11)
    assert eng._window(10, 5, 3, 1) == (3, 1)
    with pytest.raises(ValueError):
        eng.convolve_batch(np.zeros((2, 10), np.float32), np.zeros((2, 3, 4), np.float32))
    with pytest.raises(ValueError):
        eng.convolve_batch(np.zeros((2, 10), np.float32), np.zeros(5, np.float32), out=np.zeros((2, 13), np.float32))
    with pytest.raises(ValueError):
        eng.convolve_batch_device(1, 1, 10, 2, 3)                          # a device pointer h needs len_h
    h2 = np.zeros((2, 5), np.float32)
    for kw in ({"len_h": 4}, {"h_batch": 1}, {"h_batch": 3}):             # arguments that contradict a host array's shape
        with pytest.raises(ValueError):
            eng.convolve_batch_device(1, 2, 10, h2, 3, **kw)
    with pytest.raises(ValueError):
        eng.convolve_batch_device(1, 2, 10, np.zeros((2, 2, 5), np.float32), 3)
    with pytest.raises(eng.IrbError) as e:                                  # the library's own check, no device needed
        eng.convolve_batch(np.zeros((2, 10), np.float32), np.zeros((3, 5), np.float32))
    assert e.value.code == eng.IRB_ERR_ARG
    with pytest.raises(eng.IrbError) as e:
        eng.convolve_batch(np.zeros((1, 10), np.float32), np.zeros(5, np.float32), out_offset=14)
    assert e.value.code == eng.IRB_ERR_ARG


# ---- the inverse line-FFT kernels -------------------------------------------------------------------------------------------------
# registers and spill instructions (STL, LDL) of every k_line_fft<L, true> before the window existed; the windowed copy
# k_line_fft_win<L> has the same budget.  The launch bounds ask for 4 CTAs per SM (2 at L >= 1024).
_LINE_INV = {8: (48, 0, 0), 16: (64, 0, 0), 32: (64, 0, 0), 64: (64, 0, 0), 128: (64, 0, 0), 256: (64, 0, 0), 512: (64, 17, 17),
             1024: (128, 0, 0), 2048: (128, 0, 0)}
_NAMES = ("_ZN3irb10k_line_fftILi%dELb1EEEvNS_8LineArgsE", "_ZN3irb14k_line_fft_winILi%dEEEvNS_8LineArgsENS_10LineWindowE")


@pytest.mark.parametrize("name", _NAMES, ids=["plain", "windowed"])
def test_inverse_line_kernels_keep_their_registers(eng, name):
    out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-res-usage", eng.LIB_PATH], capture_output=True, text=True).stdout
    res = dict(re.findall(r"Function (\w+):\s*\n\s*REG:(\d+)", out))
    for L, (reg, _, _) in _LINE_INV.items():
        assert int(res[name % L]) == reg, (L, res.get(name % L))


@pytest.mark.parametrize("name", _NAMES, ids=["plain", "windowed"])
def test_inverse_line_kernels_spill_no_more_than_before(eng, name):
    for L, (_, stl, ldl) in _LINE_INV.items():
        sass = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", "-fun", name % L, eng.LIB_PATH], capture_output=True, text=True).stdout
        assert "Function : " + name % L in sass, L
        n_stl, n_ldl = len(re.findall(r"\bSTL\b", sass)), len(re.findall(r"\bLDL\b", sass))
        assert n_stl <= stl and n_ldl <= ldl, (L, n_stl, n_ldl)
