"""CPU: the IR-matrix engine's C ABI (irb_engine_create_matrix / irb_engine_bind_matrix) rejects bad arguments without touching
a device, and its kernel k_mac_mx has the SASS shape of the persistent block step (bulk TMA only, work counter, fenced and
predicated stage release, 128-bit shared-memory reads, no tensor cores)."""
import ctypes
import re
import subprocess

import pytest


def _create(eng, block_size=512, max_partitions=4, n_groups=8, ins=1, outs=2, n_irs=4):
    h = ctypes.c_void_p()
    rc = eng.lib().irb_engine_create_matrix(ctypes.byref(h), 0, block_size, max_partitions, n_groups, ins, outs, n_irs)
    return rc, h


@pytest.mark.parametrize("kw", [
    dict(ins=2, outs=1), dict(ins=1, outs=1), dict(ins=1, outs=4), dict(ins=4, outs=2), dict(ins=0, outs=2),
    dict(block_size=128), dict(block_size=1025), dict(block_size=2048), dict(block_size=0),
    dict(max_partitions=0), dict(n_groups=0), dict(n_groups=-3),
    dict(n_irs=1), dict(ins=2, outs=2, n_irs=3), dict(n_groups=1 << 30),
])
def test_create_matrix_rejects_bad_arguments_without_a_device(eng, kw):
    rc, h = _create(eng, **kw)
    assert rc == eng.IRB_ERR_ARG and not h.value
    assert eng.lib().irb_last_error()


def test_create_matrix_null_out_and_bind_matrix_null_engine(eng):
    L = eng.lib()
    assert L.irb_engine_create_matrix(None, 0, 512, 4, 8, 1, 2, 2) == eng.IRB_ERR_ARG
    ids = (ctypes.c_int * 2)(0, 1)
    assert L.irb_engine_bind_matrix(None, 0, 1, ids) == eng.IRB_ERR_ARG
    with pytest.raises(eng.IrbError) as ex:
        eng.MatrixEngine(512, 4, 8, 2, 1)
    assert ex.value.code == eng.IRB_ERR_ARG


def test_matrix_kernel_sass(eng):
    """k_mac_mx<512, 1, 2, false> and <512, 2, 2, false>: FDL slots and IR partitions by bulk TMA copies (the FDL ones with an
    L2 cache-policy descriptor), no 16- or 32-byte global load, units from a global atomic counter, the ring stage released behind
    a generic->async proxy fence by one predicated arrive, LDS.128 in the inner loop, no tensor-core instruction."""
    for fun in ("_ZN3irb8k_mac_mxILi512ELi1ELi2ELb0EEEvNS_7MacArgsE", "_ZN3irb8k_mac_mxILi512ELi2ELi2ELb0EEEvNS_7MacArgsE"):
        sass = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", "-fun", fun, eng.LIB_PATH], capture_output=True, text=True).stdout
        assert sass.count("UBLKCP") >= 3 and re.search(r"UBLKCP[^;]*desc\[", sass), fun
        assert not re.search(r"LDG\.E\.[A-Z0-9.]*(128|256)", sass), fun
        assert "ATOMG" in sass and "FENCE.VIEW.ASYNC" in sass and "LDS.128" in sass, fun
        assert re.search(r"@!?P\d SYNCS\.ARRIVE", sass), fun
        assert "HMMA" not in sass and not re.search(r"UTC\w*MMA", sass), fun


def test_every_matrix_instantiation_is_built(eng):
    out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", eng.LIB_PATH], capture_output=True, text=True).stdout
    names = set(re.findall(r"_ZN3irb8k_mac_mxILi(\d+)ELi(\d)ELi(\d)ELb(\d)EEEvNS_7MacArgsE", out))
    want = {(str(m), i, o, p) for m in (256, 512, 1024) for i, o in (("1", "2"), ("2", "2")) for p in ("0", "1")}
    assert names == want
