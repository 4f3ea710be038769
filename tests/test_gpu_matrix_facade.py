"""GPU: fp::b200::MatrixConvolver (the C++ facade of the IR-matrix engine) through the flat C view in tests/cpp/matrix_capi.cpp,
bit for bit against the Python MatrixEngine on the same IR files and inputs."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from irbaboon_b200 import synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_f32p = ctypes.POINTER(ctypes.c_float)


@pytest.fixture(scope="module")
def fac(built, tmp_path_factory):
    """tests/cpp/matrix_capi.cpp compiled against the facade library (irbaboon_b200/fp/libfp_b200.so, made by build()) into a
    temporary directory: the source tree is not written to."""
    fp_dir, lib_dir = os.path.join(ROOT, "irbaboon_b200", "fp"), os.path.join(ROOT, "irbaboon_b200")
    so = str(tmp_path_factory.mktemp("matrix_capi") / "libmatrix_capi.so")
    subprocess.check_call(["g++", "-std=c++14", "-O2", "-fPIC", "-shared", "-Wl,-Bsymbolic", "-o", so, os.path.join(ROOT, "tests", "cpp", "matrix_capi.cpp"),
                           "-L" + fp_dir, "-lfp_b200", "-L" + lib_dir, "-lirb_b200", "-Wl,-rpath," + fp_dir, "-Wl,-rpath," + lib_dir])
    L = ctypes.CDLL(so)
    L.mx_create.restype = ctypes.c_void_p
    L.mx_create.argtypes = [ctypes.c_int] * 6
    L.mx_destroy.argtypes = [ctypes.c_void_p]
    L.mx_set_ir.argtypes = [ctypes.c_void_p, ctypes.c_int, _f32p, ctypes.c_int, ctypes.c_int]
    L.mx_bind.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_int), ctypes.c_int]
    L.mx_reset.argtypes = [ctypes.c_void_p]
    L.mx_process.argtypes = [ctypes.c_void_p, _f32p, _f32p, ctypes.c_int]
    L.mx_process_block.argtypes = [ctypes.c_void_p, _f32p, _f32p]
    return L


def _fp(a):
    return a.ctypes.data_as(_f32p)


@pytest.mark.parametrize("ins,B,G", [(1, 512, 37), (2, 256, 21), (2, 1024, 9)])
def test_matrix_convolver_matches_python_engine(fac, eng, ins, B, G):
    """A stereo IR file is the (1, 2) matrix {L, R}; a four-channel file the (2, 2) matrix LL, LR, RL, RR.  A second file
    bound to every third group.  process() and processBlock() against MatrixEngine.process, same bits."""
    P, nb, terms = 5, 9, 2 * ins
    files = [np.stack([synth.decaying_ir(4100 + 10 * f + c, (P - f) * B - 5, c) for c in range(terms)]) for f in range(2)]      # the channels of a file share a length
    rng = np.random.default_rng(ins)
    x = (rng.random((nb, G * ins, B), dtype=np.float32) * 2 - 1).astype(np.float32)
    with eng.MatrixEngine(B, P, G, ins, 2, 2 * terms) as m:
        for f in range(2):
            for c in range(terms):
                m.set_ir(f * terms + c, files[f][c])
        for g in range(0, G, 3):
            m.bind_matrix(g, g + 1, list(range(terms, 2 * terms)))
        want = m.process(x)
    h = fac.mx_create(B, P, G, ins, 2, 2 * terms)
    assert h
    try:
        for f in range(2):
            assert fac.mx_set_ir(h, f * terms, _fp(np.ascontiguousarray(files[f])), terms, files[f].shape[1]) == 0
        three = np.zeros((3, 64), np.float32)
        assert fac.mx_set_ir(h, 0, _fp(three), 3, 64) == -1      # neither mono nor one channel per IR of the matrix
        ids = (ctypes.c_int * terms)(*range(terms, 2 * terms))
        for g in range(0, G, 3):
            assert fac.mx_bind(h, g, g + 1, ids, terms) == 0
        got = np.empty_like(want)
        assert fac.mx_process(h, _fp(x), _fp(got), nb) == 0
        assert np.array_equal(got, want)
        assert fac.mx_reset(h) == 0
        for b in range(nb):
            out = np.empty((2 * G, B), np.float32)
            assert fac.mx_process_block(h, _fp(np.ascontiguousarray(x[b])), _fp(out)) == 0
            assert np.array_equal(out, want[b]), b
    finally:
        fac.mx_destroy(h)
