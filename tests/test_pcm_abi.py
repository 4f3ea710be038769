"""CPU: the PCM entry points of the streaming engine (irb_engine_*_pcm, irb_group_process_pcm) reject bad formats, null
pointers and one-block submits without touching a device; the numpy quantiser the GPU tests use (tests/pcm_rule.py) is the
facade's formats::writeWav rule, byte for byte; and the block-step kernels keep their register budget with the conversions in
their prologue and epilogue."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

import pcm_rule

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_f32p = ctypes.POINTER(ctypes.c_float)
_PCM = ("irb_engine_process_pcm", "irb_engine_submit_pcm", "irb_engine_process_device_pcm", "irb_group_process_pcm")


@pytest.mark.parametrize("fn", _PCM)
@pytest.mark.parametrize("fin,fout", [(3, 0), (0, 3), (-1, 1), (2, -1), (1 << 30, 0)])
def test_formats_outside_the_enum_are_rejected_without_a_device(eng, fn, fin, fout):
    buf = ctypes.create_string_buffer(64)
    rc = getattr(eng.lib(), fn)(None, buf, fin, buf, fout, 2)
    assert rc == eng.IRB_ERR_ARG
    assert b"sample format" in eng.lib().irb_last_error()


@pytest.mark.parametrize("fn", _PCM)
def test_null_pointers_are_rejected(eng, fn):
    L, buf = eng.lib(), ctypes.create_string_buffer(64)
    for args in [(None, buf, 1, buf, 2, 2), (ctypes.c_void_p(1), None, 1, buf, 2, 2), (ctypes.c_void_p(1), buf, 1, None, 2, 2)]:
        assert getattr(L, fn)(*args) == eng.IRB_ERR_ARG
        assert b"null" in L.irb_last_error()


@pytest.mark.parametrize("fin,fout", [(0, 0), (1, 1), (2, 2), (1, 0)])
def test_one_block_submit_pcm_is_rejected_like_submit(eng, fin, fout):
    L, buf = eng.lib(), ctypes.create_string_buffer(64)
    assert L.irb_engine_submit_pcm(ctypes.c_void_p(1), buf, fin, buf, fout, 1) == eng.IRB_ERR_ARG
    msg = L.irb_last_error()
    assert L.irb_engine_submit(None, ctypes.cast(buf, _f32p), ctypes.cast(buf, _f32p), 1) == eng.IRB_ERR_ARG
    assert b"at least two blocks" in msg


def test_python_formats_are_checked_before_the_library(eng):
    with pytest.raises(ValueError):
        eng.sample_format("s32")
    with pytest.raises(ValueError):
        eng._pcm_input(np.zeros((2, 4, 10), np.uint8), 4)                 # a packed 24-bit array needs 3*B bytes per row
    x, f, shp = eng._pcm_input(np.zeros((2, 4, 12), np.uint8), 4)
    assert f == eng.IRB_SAMPLE_S24 and shp == (2, 4, 4)
    assert eng._pcm_input(np.zeros((3, 5), np.int16), 5)[1] == eng.IRB_SAMPLE_S16
    assert eng._pcm_input(np.zeros((3, 5), np.float64), 5)[1] == eng.IRB_SAMPLE_F32
    assert eng._pcm_output((2, 4, 4), eng.IRB_SAMPLE_S24, None).shape == (2, 4, 12)
    with pytest.raises(ValueError):
        eng._pcm_output((2, 4, 4), eng.IRB_SAMPLE_S16, np.zeros((2, 4, 4), np.float32))


# ---- the quantiser of the GPU tests is the repository's writeWav rule ------------------------------------------------------------
@pytest.fixture(scope="module")
def fac(built):
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "tests", "cpp")])
    return ctypes.CDLL(os.path.join(ROOT, "tests", "cpp", "libfacade_capi.so"))


def _write_wav_codes(fac, tmp_path, x, bits):
    path = str(tmp_path / ("q%d.wav" % bits))
    x = np.ascontiguousarray(x, np.float32).reshape(1, -1)
    assert fac.fac_write_wav(path.encode(), x.ctypes.data_as(_f32p), 1, x.shape[1], 48000, bits) == 0
    raw = np.frombuffer(open(path, "rb").read()[44:44 + x.shape[1] * bits // 8], np.uint8)
    return raw


def _edge_vector():
    f = np.float32
    vec = [0.0, -0.0, 1.0, -1.0, 1.5, -1.5, 3.4e38, -3.4e38, np.inf, -np.inf, np.nan, 2.0 ** -31, -2.0 ** -31, 2.0 ** -32, -2.0 ** -33, 1e-45, -1e-45,
           np.finfo(f).tiny, 0.5, -0.5, 1.0 / 3.0, -2.0 / 3.0]
    vec += [np.nextafter(f(1), f(0)), np.nextafter(f(-1), f(0)), np.nextafter(f(1), f(2)), np.nextafter(f(-1), f(-2))]
    for bits in (16, 24):
        step = 2.0 ** -(bits - 1)
        for k in (1, 2, 3, 12345, (1 << (bits - 1)) - 1):
            for d in (0.0, 0.5, -0.5, 0.25):
                vec += [(k + d) * step, -(k + d) * step]
        vec += [np.nextafter(f(step / 2), f(1)), np.nextafter(f(-step / 2), f(-1))]
    return np.array(vec, np.float32)


@pytest.mark.parametrize("bits", [16, 24])
def test_numpy_quantiser_is_write_wav_on_edge_vectors(fac, tmp_path, bits):
    """Full scale, one ulp either side of it, infinities, NaN, signed zeros, denormals, the codes' half-way points."""
    x = _edge_vector()
    raw = _write_wav_codes(fac, tmp_path, x, bits)
    fmt = "s%d" % bits
    want = pcm_rule.encode(x, fmt)
    assert np.array_equal(raw, want.view(np.uint8).reshape(-1)), bits
    nan = int(np.flatnonzero(np.isnan(x))[0])
    assert pcm_rule.quantise(x, bits)[nan] == 0
    assert np.array_equal(pcm_rule.decode(want, fmt), pcm_rule.quantise(x, bits) / float(1 << (bits - 1)))


@pytest.mark.parametrize("bits", [16, 24])
def test_numpy_quantiser_is_write_wav_on_a_million_random_floats(fac, tmp_path, bits):
    """1.2e6 floats: uniform over +-1.1 of full scale, and log-uniform magnitudes down to 2^-40 (rounding of small values)."""
    rng = np.random.default_rng(bits)
    x = np.concatenate([(rng.random(600_000) * 2.2 - 1.1), rng.choice([-1.0, 1.0], 600_000) * 2.0 ** rng.uniform(-40, 0, 600_000)]).astype(np.float32)
    raw = _write_wav_codes(fac, tmp_path, x, bits)
    assert np.array_equal(raw, pcm_rule.encode(x, "s%d" % bits).view(np.uint8).reshape(-1))


def test_pack24_round_trip():
    q = np.array([[-(1 << 23), -1, 0, 1, (1 << 23) - 1, 12345]], np.int64)
    b = pcm_rule.pack24(q)
    assert b.shape == (1, 18) and b.dtype == np.uint8 and list(b[0, :3]) == [0, 0, 0x80]
    assert np.array_equal(pcm_rule.unpack24(b), q)


# ---- register budget of the block-step kernels with the conversions ---------------------------------------------------------------
_KERNELS = {  # kernel -> registers it uses (the launch bounds allow 2 CTAs per SM for k_mac_p / k_mac_mx)
    "_ZN3irb7k_mac_pILi512ELb0EEEvNS_7MacArgsE": 96,
    "_ZN3irb7k_mac_pILi1024ELb1EEEvNS_7MacArgsE": 96,
    "_ZN3irb8k_mac_mxILi512ELi1ELi2ELb0EEEvNS_7MacArgsE": 96,
    "_ZN3irb8k_mac_mxILi512ELi2ELi2ELb1EEEvNS_7MacArgsE": 96,
    "_ZN3irb11k_mac_slotsILi256ELb1ELb1EEEvNS_7MacArgsE": 127,
}


def test_block_step_kernels_keep_their_registers(eng):
    out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-res-usage", eng.LIB_PATH], capture_output=True, text=True).stdout
    res = dict(re.findall(r"Function (\w+):\s*\n\s*REG:(\d+)", out))
    for k, reg in _KERNELS.items():
        assert int(res[k]) == reg, (k, res.get(k))


# local-memory instructions (spill stores, spill loads) the block steps may have: none, except k_mac_p<512, shared>, which
# before the PCM conversions had 4 spill stores and 7 spill loads at the same 96 registers
_SPILLS = {k: (0, 0) for k in _KERNELS}
_SPILLS["_ZN3irb7k_mac_pILi512ELb0EEEvNS_7MacArgsE"] = (1, 1)
_SPILLS["_ZN3irb8k_mac_mxILi512ELi1ELi2ELb1EEEvNS_7MacArgsE"] = (0, 0)
_SPILLS["_ZN3irb8k_mac_mxILi512ELi2ELi2ELb0EEEvNS_7MacArgsE"] = (0, 0)


def test_block_step_kernels_spill_no_more_than_before(eng):
    for k, (stl, ldl) in _SPILLS.items():
        sass = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", "-fun", k, eng.LIB_PATH], capture_output=True, text=True).stdout
        assert "Function : " + k in sass, k
        assert len(re.findall(r"\bSTL\b", sass)) <= stl and len(re.findall(r"\bLDL\b", sass)) <= ldl, k


def test_pcm_conversions_are_in_the_kernels(eng):
    """The epilogue converts in double (DMUL, F2I.F64); the prologue reads integers one element at a time."""
    sass = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", "-fun", "_ZN3irb7k_mac_pILi512ELb0EEEvNS_7MacArgsE", eng.LIB_PATH], capture_output=True, text=True).stdout
    assert "DMUL" in sass and re.search(r"F2I\.F64", sass)
    assert re.search(r"LDG\.E\.[SU]16", sass) and re.search(r"LDG\.E\.U8", sass)
    assert re.search(r"STG\.E\.U8", sass) and re.search(r"STG\.E\.U?16", sass)
