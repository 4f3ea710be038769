"""CPU: the batched IR chop (irb_ir_chop_batch_device, irb_deconvolve_chop_batch) rejects every bad argument with IRB_ERR_ARG
before it touches a device, and so do the Python wrappers; its kernels keep their register budget and spill nothing; the
flags-and-run-scan statement of the walk the device computes (tests/chop_rule.py) is the facade's sequential fp::ir::IRchop,
bit for bit, on rows with wrap at both ends, ties, NaN / Inf and every consecutive / ir_length corner; and the level rule's log,
(float) log((double) v), is the correctly rounded float log on every positive float but five hard cases."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

import chop_rule

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_f32p = ctypes.POINTER(ctypes.c_float)
_BUF = ctypes.create_string_buffer(4096)
_P = ctypes.cast(_BUF, ctypes.c_void_p)
_I = ctypes.cast(ctypes.create_string_buffer(64), ctypes.c_void_p)

# irb_ir_chop_batch_device(x, batch, len, ir_length, thr, consecutive, normalize, goal_db, out, positions) -> the word of irb_last_error()
_BAD_CHOP = [
    ((None, 1, 100, 10, -60.0, 50, 1, 0.0, _P, _I), b"null"),
    ((_P, 1, 100, 10, -60.0, 50, 1, 0.0, None, _I), b"null"),
    ((_P, 0, 100, 10, -60.0, 50, 1, 0.0, _P, _I), b"empty"),
    ((_P, -5, 100, 10, -60.0, 50, 1, 0.0, _P, None), b"empty"),
    ((_P, 1, 0, 1, -60.0, 50, 1, 0.0, _P, _I), b"empty"),
    ((_P, 1, -1, 1, -60.0, 50, 1, 0.0, _P, _I), b"empty"),
    ((_P, 1, 100, 0, -60.0, 50, 1, 0.0, _P, _I), b"ir_length"),
    ((_P, 1, 100, -3, -60.0, 50, 0, 0.0, _P, _I), b"ir_length"),
    ((_P, 2, 100, 101, -60.0, 50, 1, 0.0, _P, _I), b"ir_length"),
]
# irb_deconvolve_chop_batch(nums, batch, len_num, den, len_den, sr, smoothing, phase, ampl, ir_length, thr, cons, normalize, goal_db, out, pos)
_BAD_DECONV = [
    ((None, 1, 100, _P, 50, 48000.0, 0, 1, 1, 10, -60.0, 50, 1, 0.0, _P, _I), b"null"),
    ((_P, 1, 100, None, 50, 48000.0, 0, 1, 1, 10, -60.0, 50, 1, 0.0, _P, _I), b"null"),
    ((_P, 1, 100, _P, 50, 48000.0, 0, 1, 1, 10, -60.0, 50, 1, 0.0, None, _I), b"null"),
    ((_P, 0, 100, _P, 50, 48000.0, 0, 1, 1, 10, -60.0, 50, 1, 0.0, _P, _I), b"empty"),
    ((_P, 1, 0, _P, 50, 48000.0, 0, 1, 1, 10, -60.0, 50, 1, 0.0, _P, _I), b"empty"),
    ((_P, 1, 100, _P, 0, 48000.0, 0, 1, 1, 10, -60.0, 50, 1, 0.0, _P, _I), b"empty"),
    ((_P, 1, 1 << 23, _P, 50, 48000.0, 0, 1, 1, 10, -60.0, 50, 1, 0.0, _P, _I), b"2^22"),
    ((_P, 1, 4, _P, 4, 48000.0, 0, 1, 1, 4, -60.0, 50, 1, 0.0, _P, _I), b"FFT of 4"),
    ((_P, 1, 100, _P, 50, 48000.0, 0, 1, 1, 0, -60.0, 50, 1, 0.0, _P, _I), b"ir_length"),
    ((_P, 1, 100, _P, 50, 48000.0, 1, 0, 1, 129, -60.0, 50, 1, 0.0, _P, None), b"ir_length"),     # N = 128
    ((_P, 3, 128, _P, 200, 48000.0, 0, 1, 1, 257, -60.0, 50, 1, 0.0, _P, _I), b"ir_length"),      # N = 256
]


@pytest.mark.parametrize("args,word", _BAD_CHOP, ids=[str(i) for i in range(len(_BAD_CHOP))])
def test_chop_bad_arguments_are_rejected_without_a_device(eng, args, word):
    L = eng.lib()
    assert L.irb_ir_chop_batch_device(*args) == eng.IRB_ERR_ARG
    assert word in L.irb_last_error()


@pytest.mark.parametrize("args,word", _BAD_DECONV, ids=[str(i) for i in range(len(_BAD_DECONV))])
def test_capture_batch_bad_arguments_are_rejected_without_a_device(eng, args, word):
    L = eng.lib()
    assert L.irb_deconvolve_chop_batch(*args) == eng.IRB_ERR_ARG
    assert word in L.irb_last_error()


def test_the_longest_ir_is_accepted(eng):
    """ir_length == len (== N for the capture batch) gets past the checks, and fails only for want of a GPU"""
    try:
        if eng.device_count() > 0:
            pytest.skip("a GPU is visible")
    except eng.IrbError:
        pass
    L = eng.lib()
    assert L.irb_ir_chop_batch_device(_P, 1, 100, 100, -60.0, 50, 1, 0.0, _P, None) == eng.IRB_ERR_CUDA
    assert L.irb_deconvolve_chop_batch(_P, 1, 100, _P, 50, 48000.0, 0, 1, 1, 128, -60.0, 50, 1, 0.0, _P, None) == eng.IRB_ERR_CUDA


def test_python_argument_checks(eng):
    for kw in ({"batch": 0}, {"len": 0}, {"ir_length": 0}, {"ir_length": 101}, {"x_ptr": 0}, {"out_ptr": 0}):
        a = dict(x_ptr=1, batch=2, len=100, ir_length=10, out_ptr=2)
        a.update(kw)
        with pytest.raises(ValueError):
            eng.ir_chop_batch_device(**a)
    nums, den = np.zeros((2, 100), np.float32), np.ones(50, np.float32)
    for L in (0, -1, 129):
        with pytest.raises(ValueError):
            eng.deconvolve_chop_batch(nums, den, L)
    with pytest.raises(ValueError):
        eng.deconvolve_chop_batch(nums, den, 16, out=np.zeros((2, 15), np.float32))
    with pytest.raises(ValueError):
        eng.deconvolve_chop_batch(nums, den, 16, out=np.zeros((2, 16), np.float64))
    with pytest.raises(ValueError):
        eng.deconvolve_chop_batch(np.zeros((2, 3, 4), np.float32), den, 4)
    with pytest.raises(ValueError):
        eng.deconvolve_chop_batch(nums, np.zeros(0, np.float32), 4)
    with pytest.raises(eng.IrbError) as e:                                  # the library's own check (N = 8 is below the transforms)
        eng.deconvolve_chop_batch(np.zeros((1, 5), np.float32), np.ones(3, np.float32), 4)
    assert e.value.code == eng.IRB_ERR_ARG


# ---- the kernels ------------------------------------------------------------------------------------------------------------------
# registers of the chop kernels (launch bounds: 256 threads for the peak pass, 512 for the cut); none spills
_KERNELS = {"_ZN3irb11k_chop_peakILb0EEEvPKfxixPfPx": 32, "_ZN3irb11k_chop_peakILb1EEEvPKfxixPfPx": 34, "_ZN3irb10k_chop_cutENS_8ChopArgsE": 32}


def test_chop_kernels_keep_their_registers_and_do_not_spill(eng):
    out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-res-usage", eng.LIB_PATH], capture_output=True, text=True).stdout
    res = dict(re.findall(r"Function (\w+):\s*\n\s*REG:(\d+)", out))
    for name, reg in _KERNELS.items():
        assert int(res[name]) == reg, (name, res.get(name))
        sass = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", "-fun", name, eng.LIB_PATH], capture_output=True, text=True).stdout
        assert "Function : " + name in sass
        assert not re.findall(r"\b(STL|LDL)\b", sass), name


# ---- the rule ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def fac(built):
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "tests", "cpp")])
    h = ctypes.CDLL(os.path.join(ROOT, "tests", "cpp", "libfacade_capi.so"))
    h.fac_ir_chop.argtypes = [_f32p, ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_int, _f32p]
    return h


@pytest.fixture(scope="module")
def helper(built, tmp_path_factory):
    return chop_rule.build_helper(tmp_path_factory.mktemp("chop_rule"))


def _fac_chop(fac, x, L, thr, c):
    x = np.ascontiguousarray(x, np.float32)
    out = np.empty(L, np.float32)
    assert fac.fac_ir_chop(x.ctypes.data_as(_f32p), len(x), L, thr, c, out.ctypes.data_as(_f32p)) == L
    return out


def _same(a, b):
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def test_the_run_scan_is_the_facades_sequential_walk(fac, helper):
    """with the facade's own levels, the statement of the walk the device computes gives the facade's IR bit for bit (NaN payloads too)"""
    n_cases = 0
    for seed in range(6):
        for name, x, L, thr, c in chop_rule.cases(seed):
            got, q, start = chop_rule.chop(helper, x, L, thr, c, rule=False)
            want = _fac_chop(fac, x, L, thr, c)
            assert _same(got, want), (seed, name, q, start)
            n_cases += 1
    assert n_cases >= 6 * 60


def test_a_wrapped_cut_and_a_capped_walk(helper):
    """the corners the statement is built for, checked by hand: the walk wraps below index 0, the cut wraps past n - 1"""
    x = np.full(100, 1e-6, np.float32)
    x[2] = 1.0
    x[95:100] = 0.5                                       # loud: the walk from q = 2 meets 99 .. 95 after the wrap below index 0
    out, q, start = chop_rule.chop(helper, x, 40, -60.0, 10, rule=True)
    assert q == 2 and start == 100 + 2 - 18               # walk positions 0 (the peak) and 3..7 (99..95) loud, 8..17 quiet: walked = 18
    assert out[18] == np.float32(1.0)                     # the peak lands at offset walked; no fade touches it (18/4 = 4, 40 - 1 - 10 = 29)
    x2 = np.full(100, 0.5, np.float32)
    x2[50] = 1.0
    assert chop_rule.chop(helper, x2, 30, -60.0, 5, rule=True)[2] == 20        # never quiet: walked = ir_length
    assert chop_rule.chop(helper, x2, 30, -60.0, 31, rule=True)[2] == 20       # consecutive > ir_length: the same cap
    assert chop_rule.chop(helper, x2, 30, -60.0, 0, rule=True)[2] == 50        # consecutive 0: the cut starts at the peak


def test_ln10_is_the_correctly_rounded_constant(helper):
    assert helper.chop_ln10f() == np.float32(np.log(10.0)) == helper.chop_glibc_ln10f()


# the five positive floats whose ln lies so close to a float rounding boundary that rounding the double-precision log to float
# misses the nearest float (hard cases of the float log): the rule is (float) log((double) v) there too, as on the device
_HARD_CASES = ["0x3c413d3a", "0x41178feb", "0x4c5d65a5", "0x65d890d3", "0x6f31a8ec"]


def test_the_level_log_is_correctly_rounded_on_every_positive_float(helper):
    """(float) log((double) v) against ln(v) in 64-bit-significand precision, over all 2 139 095 039 positive finite floats (OpenMP):
    the nearest float everywhere but the five hard cases; also counts where glibc's logf, and the facade's linTodB, differ from the
    rule (the inputs on which a cut can move)"""
    counts = (ctypes.c_longlong * 4)()
    bad = (ctypes.c_uint32 * 16)()
    helper.chop_log_sweep(counts, bad, 16)
    n, miss, dlog, ddb = list(counts)
    print("positive floats %d, rule not nearest %d, glibc logf != rule %d, linTodB != rule %d" % (n, miss, dlog, ddb))
    assert n == 0x7f800000 - 1
    assert sorted(hex(b) for b in list(bad)[:min(miss, 16)]) == _HARD_CASES
    assert dlog > ddb > 0                                 # glibc's logf is not correctly rounded: the rule is a choice, and a documented one


def test_a_level_flip_exists_where_the_gpu_test_looks(helper):
    """the constructed flip row of tests/test_gpu_ir_chop.py needs a v near 1e-3 whose facade level is below the rule's"""
    v = (ctypes.c_float * 4)()
    assert helper.chop_find_level_flips(np.float32(1e-3).view(np.uint32).item(), v, 4) == 4
    x = np.array(list(v), np.float32)
    assert np.all(chop_rule.levels(helper, x, False) < chop_rule.levels(helper, x, True))
