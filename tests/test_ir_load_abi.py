"""CPU: the batched IR loads (irb_engine_set_irs / _stage_irs, irb_group_set_irs / _stage_irs) reject every argument error their
rows carry with IRB_ERR_ARG before they touch a device, and so do the per-IR calls that are their one-row case; the Python wrappers
check shapes and kinds; k_ir_load keeps its register budget and spills nothing.  The errors that need an engine (an id outside
[0, n_irs), more taps or partitions than the ring, device memory) are checked in tests/test_gpu_ir_load.py."""
import ctypes
import re
import subprocess

import numpy as np
import pytest

_vp = ctypes.c_void_p
_BUF = ctypes.create_string_buffer(1 << 16)
_P = ctypes.cast(_BUF, _vp)
_H = ctypes.cast(ctypes.create_string_buffer(64), _vp)          # a stand-in engine / group handle: never reached


def _ints(*v):
    return (ctypes.c_int * len(v))(*v)


# (n, ids, taps, ld, n_taps) -> the word of irb_last_error(); every case is also given a non-null handle, which is never looked at
_BAD = [
    ((2, None, _P, 10, None), b"null"),
    ((2, _ints(0, 1), None, 10, None), b"null"),
    ((0, _ints(0), _P, 10, None), b"n 0"),
    ((-3, _ints(0), _P, 10, None), b"n -3"),
    ((2, _ints(0, 1), _P, 0, None), b"n_taps[0] = 0"),                # n_taps NULL: ld taps each
    ((2, _ints(0, 1), _P, 10, _ints(10, 0)), b"n_taps[1] = 0"),
    ((2, _ints(0, 1), _P, 10, _ints(-5, 3)), b"n_taps[0] = -5"),
    ((2, _ints(0, 1), _P, 10, _ints(10, 11)), b"ld 10 < n_taps[1]"),
    ((3, _ints(0, 1, 2), _P, 4, _ints(4, 4, 5)), b"ld 4 < n_taps[2]"),
    ((3, _ints(4, 1, 4), _P, 10, None), b"repeats"),
    ((4, _ints(0, 7, 3, 7), _P, 10, _ints(1, 2, 3, 4)), b"ir_ids[3] = 7 repeats ir_ids[1]"),
    ((1, _ints(0), _P, 1 << 31, None), b"2^31"),
]


def _full(a):          # (n, ids, taps, ld, n_taps) -> (n, ids, taps, right = NULL, ld, n_taps)
    return a[:3] + (None,) + a[3:]


_CALLS = {
    "engine_set": lambda L, h, a: L.irb_engine_set_irs(h, *_full(a)),
    "engine_stage": lambda L, h, a: L.irb_engine_stage_irs(h, *_full(a), 0),
    "group_set": lambda L, h, a: L.irb_group_set_irs(h, *_full(a)),
    "group_stage": lambda L, h, a: L.irb_group_stage_irs(h, *_full(a), 3),
}


@pytest.mark.parametrize("call", sorted(_CALLS))
@pytest.mark.parametrize("args,word", _BAD, ids=[str(i) for i in range(len(_BAD))])
def test_row_errors_are_rejected_without_a_device(eng, call, args, word):
    L = eng.lib()
    assert _CALLS[call](L, _H, args) == eng.IRB_ERR_ARG
    assert word in L.irb_last_error(), L.irb_last_error()


@pytest.mark.parametrize("call", sorted(_CALLS))
def test_a_null_handle_is_rejected_after_the_rows(eng, call):
    L = eng.lib()
    assert _CALLS[call](L, None, (2, _ints(0, 1), _P, 10, None)) == eng.IRB_ERR_ARG
    assert b"null" in L.irb_last_error()


def test_the_per_ir_calls_are_one_row_loads(eng):
    """irb_engine_set_ir / _stage_ir and the group forms keep their argument errors: they are one-row calls of the batch path"""
    L = eng.lib()
    for rc in (L.irb_engine_set_ir(_H, 0, None, None, 10), L.irb_engine_stage_ir(_H, 0, None, None, 10, 0),
               L.irb_group_set_ir(_H, 0, None, None, 10), L.irb_group_stage_ir(_H, 0, None, None, 10, 0)):
        assert rc == eng.IRB_ERR_ARG
    for rc in (L.irb_engine_set_ir(_H, 0, _P, None, 0), L.irb_engine_stage_ir(_H, 0, _P, None, -1, 0),
               L.irb_group_set_ir(_H, 0, _P, None, 0), L.irb_group_stage_ir(_H, 0, _P, None, 0, 2)):
        assert rc == eng.IRB_ERR_ARG
        assert b"n_taps[0]" in L.irb_last_error()
    assert L.irb_engine_set_ir(None, 0, _P, None, 10) == eng.IRB_ERR_ARG


def test_python_argument_checks(eng):
    """shapes, kinds and counts are checked in Python before the library sees them"""
    e = eng.Engine.__new__(eng.Engine)                  # no device: the checks come before the handle is used
    e._h = _vp()
    t = np.zeros((3, 100), np.float32)
    bad = [
        dict(ir_ids=[], taps=t),                                         # no rows
        dict(ir_ids=[0, 1], taps=t),                                     # one id per row
        dict(ir_ids=[0, 1, 2], taps=np.zeros((3, 4, 5), np.float32)),
        dict(ir_ids=[0, 1, 2], taps=t, ld=99),                           # ld contradicts the array
        dict(ir_ids=[0, 1, 2], taps=t, right=np.zeros((3, 99), np.float32)),
        dict(ir_ids=[0, 1, 2], taps=t, right=12345),                     # a pointer right with a host taps
        dict(ir_ids=[0, 1, 2], taps=t, n_taps=[100, 100]),               # one count per row
        dict(ir_ids=[0, 1, 2], taps=t, n_taps=[100, 100, 2**31]),
        dict(ir_ids=[0, 1], taps=12345),                                 # a pointer needs ld
        dict(ir_ids=[0, 1], taps=12345, ld=10, right=t),                 # a host right with a pointer taps
        dict(ir_ids=[0, 1], taps=0, ld=10),                              # a null pointer
        dict(ir_ids=[2**31], taps=t[:1]),
    ]
    for kw in bad:
        for f in (e.set_irs, e.stage_irs):
            with pytest.raises(ValueError):
                f(**kw)
    g = eng.Group.__new__(eng.Group)
    g._h = _vp()
    for f in (g.set_irs, g.stage_irs):
        with pytest.raises(ValueError):
            f([0, 1], 12345)                                             # a group loads host arrays only
        with pytest.raises(ValueError):
            f([0, 1], t)


# ---- the kernel -------------------------------------------------------------------------------------------------------------------
_KERNELS = {"_ZN3irb9k_ir_loadILi%dEEEvNS_10IrLoadArgsE" % M: 40 for M in (16, 32, 64, 128, 256, 512, 1024, 2048)}


def test_ir_load_kernels_keep_their_registers_and_do_not_spill(eng):
    out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-res-usage", eng.LIB_PATH], capture_output=True, text=True).stdout
    res = dict(re.findall(r"Function (\w+):\s*\n\s*REG:(\d+)", out))
    for name, reg in _KERNELS.items():
        assert int(res[name]) == reg, (name, res.get(name))
        sass = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", "-fun", name, eng.LIB_PATH], capture_output=True, text=True).stdout
        assert "Function : " + name in sass
        assert not re.findall(r"\b(STL|LDL)\b", sass), name
