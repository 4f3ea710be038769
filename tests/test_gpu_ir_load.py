"""GPU: batched IR loads (irb_engine_set_irs / _stage_irs, the group forms, the facade's setIRs) against loops of the per-IR calls
on a second engine, bit for bit: every partition of the spectra (past each IR's end too) at one block size per FFT half size, the
copies of a shared IR through block-step outputs, host (pageable, pinned, several staging chunks) and device sources (a torch
tensor at a 4-byte offset, the output of irb_ir_chop_batch_device), staged IRs over the round-robin refresh, the matrix engine,
private and shared groups; and the argument errors that need an engine, which leave every IR as it was."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from irbaboon_b200 import synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_vp = ctypes.c_void_p
_f32p = ctypes.POINTER(ctypes.c_float)


@pytest.fixture(scope="module")
def torch():
    import torch

    assert torch.cuda.is_available()
    return torch


def _same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def _spectra(e, ids):
    return np.stack([np.stack([e.ir_spectrum(i, p) for p in range(e.max_partitions)]) for i in ids])


def _rows(seed, n, ld, lens, scale=1.0):
    rng = np.random.default_rng(seed)
    t = (rng.standard_normal((n, ld)) * scale).astype(np.float32)
    for j, L in enumerate(lens):
        t[j, L:] = np.float32(np.nan)            # never read: a row past its n_taps would poison the spectra
    return t


def _loop(e, ids, t, lens, right=None, stage=False, n_partitions=0):
    for j, i in enumerate(ids):
        taps = t[j, :lens[j]] if right is None else np.stack([t[j, :lens[j]], right[j, :lens[j]]])
        e.stage_ir(i, taps, n_partitions) if stage else e.set_ir(i, taps)


def _blocks(C, nb, B, seed):
    rng = np.random.default_rng(seed)
    return (rng.random((nb, C, B), dtype=np.float32) * 2 - 1).astype(np.float32)


# one block size per FFT half size 16 .. 2048
@pytest.mark.parametrize("B", [9, 32, 64, 100, 256, 300, 1024, 2048])
def test_spectra_equal_per_ir_loads(eng, torch, B):
    """ragged rows (1 tap, whole partitions, the ring's full length, ld > n_taps), mono and folded stereo, from pageable host
    memory, pinned memory and a device row 4-byte but not 8-byte aligned; loaded over longer IRs, so the partitions past each
    new end must be cleared in place"""
    P, n_irs = 5, 7
    ld = P * B + 3
    lens = [1, B, 3 * B, P * B, 2 * B + 7, B - 1 if B > 1 else 1]
    ids = [5, 0, 3, 6, 1, 2]
    t = _rows(B, len(ids), ld, lens)
    r = _rows(B + 1, len(ids), ld, lens)
    full = _rows(B + 2, n_irs, P * B, [P * B] * n_irs)
    for right in (None, r):
        with eng.Engine(B, P, 4, n_irs) as a, eng.Engine(B, P, 4, n_irs) as b:
            a.set_irs(range(n_irs), full)
            _loop(b, range(n_irs), full, [P * B] * n_irs)
            assert _same(_spectra(a, range(n_irs)), _spectra(b, range(n_irs)))
            a.set_irs(ids, t, n_taps=lens, right=right)
            _loop(b, ids, t, lens, right)
            want = _spectra(b, range(n_irs))
            assert _same(_spectra(a, range(n_irs)), want)
            assert [a.partitions(i) for i in range(n_irs)] == [b.partitions(i) for i in range(n_irs)]
            # pinned host rows
            pt, pr = eng.pinned_empty(t.shape), (eng.pinned_empty(r.shape) if right is not None else None)
            pt[:] = t
            if pr is not None:
                pr[:] = r
            a.set_irs(range(n_irs), full)
            a.set_irs(ids, pt, n_taps=lens, right=pr)
            assert _same(_spectra(a, range(n_irs)), want)
            # device rows at a 4-byte offset
            dt = torch.empty(t.size + 1, dtype=torch.float32, device="cuda")
            dt[1:] = torch.from_numpy(t.reshape(-1))
            dr = torch.empty(r.size + 1, dtype=torch.float32, device="cuda")
            dr[1:] = torch.from_numpy(r.reshape(-1))
            torch.cuda.synchronize()
            assert (dt.data_ptr() + 4) % 8 == 4 and (dr.data_ptr() + 4) % 8 == 4
            a.set_irs(range(n_irs), full)
            a.set_irs(ids, dt.data_ptr() + 4, n_taps=lens, right=(dr.data_ptr() + 4 if right is not None else None), ld=ld)
            assert _same(_spectra(a, range(n_irs)), want)


def test_shared_ir_copies_give_equal_block_steps(eng):
    """one shared IR, kept in many copies (engines created with ir_replicas = 0 keep as many as fit 24 MB; CTA b of the block
    step reads copy b % h_reps): equal outputs over several blocks, and every channel within 1e-5 of the float64 convolution, so
    every copy holds the loaded IR's spectra"""
    B, P, C, nb = 256, 6, 3000, 8
    h = synth.decaying_ir(5100, P * B - 17)
    x = _blocks(C, nb, B, 1)
    old = eng.get_tuning("ir_replicas")
    eng.set_tuning("ir_replicas", 0)
    try:
        a, b = eng.Engine(B, P, C, 1), eng.Engine(B, P, C, 1)
    finally:
        eng.set_tuning("ir_replicas", old)
    with a, b:
        assert a.ir_copies == b.ir_copies == 32
        a.set_ir(0, synth.decaying_ir(5101, P * B))
        b.set_ir(0, synth.decaying_ir(5101, P * B))
        a.set_irs([0], h)
        b.set_ir(0, h)
        ya, yb = a.process(x), b.process(x)
    assert _same(ya, yb)
    xs = x.transpose(1, 0, 2).reshape(C, nb * B).astype(np.float64)
    N = 1 << int(np.ceil(np.log2(nb * B + len(h))))
    want = np.fft.irfft(np.fft.rfft(xs, N) * np.fft.rfft(h.astype(np.float64), N), N)[:, :nb * B]
    got = ya.transpose(1, 0, 2).reshape(C, nb * B)
    err = np.abs(got - want).max(axis=1) / np.maximum(1.0, np.abs(want).max(axis=1))
    assert err.max() <= 1e-5, (int(err.argmax()), float(err.max()))


# the transform of k_ir_load against k_fwd's own: a first staging reaches its spectra through the block steps' refresh rows
@pytest.mark.parametrize("B", [9, 32, 64, 100, 256, 300, 1024, 2048])
def test_set_irs_spectra_equal_the_refresh_rows(eng, B):
    P = 5
    lens = [P * B, 2 * B + 3]
    t, r = _rows(60 + B, 2, P * B, lens), _rows(61 + B, 2, P * B, lens)
    with eng.Engine(B, P, 4, 2) as a, eng.Engine(B, P, 4, 2) as b:
        a.set_irs([0, 1], t, n_taps=lens, right=r)
        b.stage_irs([0, 1], t, n_taps=lens, right=r)                    # cleared spectra, then one partition per block step
        b.process(np.zeros((P, 4, B), np.float32))
        assert [a.partitions(i) for i in range(2)] == [b.partitions(i) for i in range(2)] == [P, 3]
        assert _same(_spectra(a, [0, 1]), _spectra(b, [0, 1]))


def test_a_load_that_runs_out_of_memory_changes_nothing(eng, torch):
    """stage_irs whose round-robin buffers do not fit in free device memory fails as a whole: the partition counts, the staged
    IRs and the block steps (with their refresh rows) are those of an engine that never saw the call; the same call succeeds once
    the memory is back"""
    B, P, C, n = 2048, 512, 16, 1000                  # a round-robin buffer is 4 MB: 4 GB for the call
    nb = 6
    lens = [P * B] * 2
    t = _rows(70, 2, P * B, lens, 0.05)
    one = np.ones((n, 1), np.float32)
    x = _blocks(C, 2 * nb, B, 9)
    with eng.Engine(B, P, C, n) as a, eng.Engine(B, P, C, n) as b:
        for e in (a, b):
            for c in range(C):
                e.bind(c, c + 1, c % 2)
            e.set_irs([0, 1], t)
            e.stage_irs([1], t[1:] * np.float32(0.5))               # one staged IR: the refresh rows run in every block step
        before = [a.partitions(i) for i in range(n)]
        hold, free = [], torch.cuda.mem_get_info()[0]
        try:
            while free > (2 << 30):                                  # leave 1 to 2 GB free
                hold.append(torch.empty(1 << 30, dtype=torch.uint8, device="cuda"))
                free = torch.cuda.mem_get_info()[0]
            with pytest.raises(eng.IrbError) as ex:
                a.stage_irs(range(2, n), one[2:])
            assert ex.value.code == eng.IRB_ERR_CUDA
        finally:
            del hold
            torch.cuda.empty_cache()
        assert [a.partitions(i) for i in range(n)] == before
        assert _same(a.process(x[:nb]), b.process(x[:nb]))
        a.stage_irs(range(2, n), one[2:])
        b.stage_irs(range(2, n), one[2:])
        assert _same(a.process(x[nb:]), b.process(x[nb:]))
        assert [a.partitions(i) for i in range(n)] == [b.partitions(i) for i in range(n)]


def test_many_irs_in_several_staging_chunks(eng):
    """more than one staging chunk of host rows (64 MB per chunk and side): pageable and pinned, mono and folded, set and stage"""
    B, P, n = 1024, 40, 460                           # 460 rows of 160 KB: two chunks
    ld = P * B
    lens = [ld - (j * 37) % B for j in range(n)]
    t, r = _rows(11, n, ld, lens, 0.1), _rows(12, n, ld, lens, 0.1)
    pick = [0, 1, 200, 407, 408, 409, 410, n - 1]        # 409 rows per chunk
    with eng.Engine(B, P, 8, n) as a, eng.Engine(B, P, 8, n) as b:
        _loop(b, range(n), t, lens, r)
        want = _spectra(b, pick)
        a.set_irs(range(n), t, n_taps=lens, right=r)
        assert _same(_spectra(a, pick), want)
        pt = eng.pinned_empty(t.shape)
        pt[:] = t
        a.set_irs(range(n), pt, n_taps=lens)
        _loop(b, range(n), t, lens)
        assert _same(_spectra(a, pick), _spectra(b, pick))
    # staged rows through the chunks: channel c convolves with IR c
    C, nb = 8 * ((n + 7) // 8), P + 2
    x = _blocks(C, nb, B, 2)
    with eng.Engine(B, P, C, n) as a, eng.Engine(B, P, C, n) as b:
        for e in (a, b):
            for c in range(C):
                e.bind(c, c + 1, c % n)
        a.stage_irs(range(n), t, n_taps=lens, right=r)
        _loop(b, range(n), t, lens, r, stage=True)
        assert _same(a.process(x), b.process(x))


def test_device_sources(eng, torch):
    """IRs cut on the device by irb_ir_chop_batch_device, and rows of a torch tensor, load as their host copies do"""
    B, P, n, Lx, L = 512, 8, 12, 1 << 14, 3000
    rng = np.random.default_rng(3)
    x = (rng.standard_normal((n, Lx)) * np.exp(-np.arange(Lx) / 900.0)).astype(np.float32)
    x = np.roll(x, 200, axis=1)
    xd = torch.from_numpy(x).cuda()
    out = torch.empty((n, L), dtype=torch.float32, device="cuda")
    eng.ir_chop_batch_device(xd.data_ptr(), n, Lx, L, out.data_ptr())
    torch.cuda.synchronize()
    host = out.cpu().numpy()
    ids = list(range(n - 1, -1, -1))
    with eng.Engine(B, P, 4, n) as a, eng.Engine(B, P, 4, n) as b:
        a.set_irs(ids, out.data_ptr(), ld=L)
        b.set_irs(ids, host)
        assert _same(_spectra(a, range(n)), _spectra(b, range(n)))
        t = torch.randn((n, P * B), device="cuda")
        torch.cuda.synchronize()                        # written on torch's stream: ordered before the load by the caller
        a.set_irs(range(n), t.data_ptr(), ld=P * B, n_taps=[P * B - j for j in range(n)])
        b.set_irs(range(n), t.cpu().numpy(), n_taps=[P * B - j for j in range(n)])
        assert _same(_spectra(a, range(n)), _spectra(b, range(n)))


def test_staging_equals_per_ir_stage_calls(eng):
    """first staging, restaging with the same and with a new partition count, set_irs on a staged IR: block-step outputs over
    P + 2 blocks after each, equal to per-IR stage_ir / set_ir calls"""
    B, P, C, n = 256, 6, 64, 4
    nb = P + 2
    lens = [P * B, 3 * B + 5, 1, 5 * B]
    t1, t2, t3 = (_rows(20 + k, n, P * B, lens) for k in range(3))
    r1 = _rows(30, n, P * B, lens)
    x = _blocks(C, 5 * nb, B, 4)
    with eng.Engine(B, P, C, n) as a, eng.Engine(B, P, C, n) as b:
        for e in (a, b):
            for c in range(C):
                e.bind(c, c + 1, c % n)
        a.set_irs([3], t3[:1], n_taps=[lens[0]])
        b.set_ir(3, t3[0, :lens[0]])
        steps = [
            (lambda: a.stage_irs([0, 1, 2, 3], t1, n_taps=lens, right=r1), lambda: _loop(b, [0, 1, 2, 3], t1, lens, r1, stage=True)),
            (lambda: a.stage_irs([2, 0, 1, 3], t2, n_taps=lens), lambda: _loop(b, [2, 0, 1, 3], t2, lens, stage=True)),
            (lambda: a.stage_irs([1, 3], t3[:2], n_taps=lens[:2], n_partitions=4), lambda: _loop(b, [1, 3], t3[:2], lens[:2], stage=True, n_partitions=4)),
            (lambda: a.set_irs([0, 1], t1[2:], n_taps=lens[2:]), lambda: _loop(b, [0, 1], t1[2:], lens[2:])),
        ]
        k = 0
        for fa, fb in steps:
            fa()
            fb()
            assert [a.partitions(i) for i in range(n)] == [b.partitions(i) for i in range(n)]
            assert _same(a.process(x[k:k + nb]), b.process(x[k:k + nb])), k
            k += nb
        assert _same(_spectra(a, range(n)), _spectra(b, range(n)))


def test_matrix_engine(eng):
    B, P, G, nb = 512, 5, 40, 7
    irs = np.stack([synth.decaying_ir(5200 + i, P * B - 40) for i in range(4)])
    x = _blocks(2 * G, nb, B, 5)
    with eng.MatrixEngine(B, P, G, 2, 2) as a, eng.MatrixEngine(B, P, G, 2, 2) as b:
        a.set_irs([0, 1, 2, 3], irs)
        for i in range(4):
            b.set_ir(i, irs[i])
        assert _same(a.process(x), b.process(x))


@pytest.mark.parametrize("n_irs", [0, 3])
def test_groups(eng, n_irs):
    """private-IR (ids are channels) and shared-IR groups over the devices the box has (one device serves as two), against
    per-IR group calls; device memory is rejected"""
    B, P, C = 256, 5, 96
    nb = P + 2
    devs = [i % max(1, eng.device_count()) for i in range(2)]
    n = C if n_irs == 0 else n_irs
    lens = [P * B - (7 * j) % B for j in range(n)]
    t = _rows(40, n, P * B, lens)
    ids = list(np.random.default_rng(6).permutation(n))
    x = _blocks(C, 2 * nb, B, 7)
    with eng.Group(devs, B, P, C, n_irs) as a, eng.Group(devs, B, P, C, n_irs) as b:
        if n_irs:
            for g in (a, b):
                for c in range(C):
                    g.bind(c, c + 1, c % n_irs)
        a.set_irs(ids, t[ids], n_taps=[lens[i] for i in ids])
        for i in ids:
            b.set_ir(i, t[i, :lens[i]])
        assert _same(a.process(x[:nb]), b.process(x[:nb]))
        a.stage_irs(ids[::-1], t[ids[::-1]], n_taps=[lens[i] for i in ids[::-1]])
        for i in ids[::-1]:
            b.stage_ir(i, t[i, :lens[i]])
        assert _same(a.process(x[nb:]), b.process(x[nb:]))
        import torch

        d = torch.zeros((n, P * B), device="cuda")
        ids_c = (ctypes.c_int * n)(*range(n))
        assert eng.lib().irb_group_set_irs(a._h, n, ids_c, _vp(d.data_ptr()), None, P * B, None) == eng.IRB_ERR_ARG
        assert b"host memory" in eng.lib().irb_last_error()


def test_engine_errors_leave_every_ir_as_it_was(eng, torch):
    B, P, n = 128, 4, 4                               # IR 3 is never loaded
    L = eng.lib()
    t = _rows(50, 2, P * B, [P * B, P * B])
    with eng.Engine(B, P, 4, n) as e:
        e.set_irs(range(n - 1), _rows(51, n - 1, P * B, [P * B] * (n - 1)))
        before = _spectra(e, range(n))
        parts = [e.partitions(i) for i in range(n)]
        bad = [
            dict(ir_ids=[0, n], taps=t),                                 # an id outside [0, n_irs)
            dict(ir_ids=[0, -1], taps=t),
        ]
        for kw in bad:
            for f in (e.set_irs, e.stage_irs):
                with pytest.raises(eng.IrbError) as ex:
                    f(**kw)
                assert ex.value.code == eng.IRB_ERR_ARG
        big = _rows(52, 2, P * B + 1, [P * B + 1] * 2)
        with pytest.raises(eng.IrbError) as ex:
            e.set_irs([0, 1], big)                                       # more taps than the ring holds
        assert ex.value.code == eng.IRB_ERR_ARG
        with pytest.raises(eng.IrbError) as ex:
            e.stage_irs([0, 1], t, n_partitions=P + 1)                   # more partitions than the ring
        assert ex.value.code == eng.IRB_ERR_ARG
        with pytest.raises(eng.IrbError) as ex:
            e.stage_irs([0, 3], big)                                     # stage_ir's rule for IR 3: ceil(n_taps / B) partitions
        assert ex.value.code == eng.IRB_ERR_ARG
        d = torch.zeros(2 * P * B, device="cuda")
        ids = (ctypes.c_int * 2)(0, 1)
        assert L.irb_engine_set_irs(e._h, 2, ids, t.ctypes.data_as(_vp), _vp(d.data_ptr()), P * B, None) == eng.IRB_ERR_ARG
        assert b"both" in L.irb_last_error()
        if torch.cuda.device_count() > 1:
            d1 = torch.zeros(2 * P * B, device="cuda:1")
            assert L.irb_engine_set_irs(e._h, 2, ids, _vp(d1.data_ptr()), None, P * B, None) == eng.IRB_ERR_ARG
        assert _same(_spectra(e, range(n)), before)
        assert [e.partitions(i) for i in range(n)] == parts


# ---- the facade ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def fac(built, tmp_path_factory):
    """tests/cpp/ir_load_capi.cpp compiled against the facade library into a temporary directory"""
    fp_dir, lib_dir = os.path.join(ROOT, "irbaboon_b200", "fp"), os.path.join(ROOT, "irbaboon_b200")
    so = str(tmp_path_factory.mktemp("ir_load_capi") / "libir_load_capi.so")
    subprocess.check_call(["g++", "-std=c++14", "-O2", "-fPIC", "-shared", "-Wl,-Bsymbolic", "-o", so, os.path.join(ROOT, "tests", "cpp", "ir_load_capi.cpp"),
                           "-L" + fp_dir, "-lfp_b200", "-L" + lib_dir, "-lirb_b200", "-Wl,-rpath," + fp_dir, "-Wl,-rpath," + lib_dir])
    L = ctypes.CDLL(so)
    L.il_create.restype = ctypes.c_void_p
    L.il_create.argtypes = [ctypes.c_int] * 6
    L.il_destroy.argtypes = [ctypes.c_int, ctypes.c_void_p]
    L.il_set.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_int, _f32p, ctypes.c_int, ctypes.c_int, ctypes.c_int]
    L.il_bind.argtypes = [ctypes.c_int, ctypes.c_void_p] + [ctypes.c_int] * 3
    L.il_process.argtypes = [ctypes.c_int, ctypes.c_void_p, _f32p, _f32p, ctypes.c_int]
    return L


@pytest.mark.parametrize("multi", [0, 2])
def test_facade_set_irs_equals_set_ir_loop(fac, eng, multi):
    B, P, C, nb, n = 512, 4, 40, 6, 5
    irs = np.stack([synth.decaying_ir(5300 + i, P * B - 3) for i in range(n)])
    x = _blocks(C, nb, B, 8)
    ys = []
    for loop in (0, 1):
        h = fac.il_create(multi, eng.device_count(), B, P, C, n + 1)
        assert h
        try:
            assert fac.il_set(multi, h, 1, irs.ctypes.data_as(_f32p), n, irs.shape[1], loop) == 0
            for c in range(C):
                assert fac.il_bind(multi, h, c, c + 1, c % (n + 1)) == 0
            y = np.empty_like(x)
            assert fac.il_process(multi, h, x.ctypes.data_as(_f32p), y.ctypes.data_as(_f32p), nb) == 0
            ys.append(y)
        finally:
            fac.il_destroy(multi, h)
    assert _same(ys[0], ys[1])
