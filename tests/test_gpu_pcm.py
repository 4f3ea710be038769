"""GPU: 16- and 24-bit PCM through the streaming engine's block steps (irb_engine_*_pcm, irb_group_process_pcm).

The rule, for every block-step form and every output channel: feeding PCM x and asking for format F gives, bit for bit,
encode(y, F), where y is what the float engine outputs for decode(x) (tests/pcm_rule.py, pinned to formats::writeWav by
tests/test_pcm_abi.py).  Every run takes at least P + 3 blocks, so the delay line wraps.
"""
import ctypes
import itertools
import os
import subprocess

import numpy as np
import pytest

import pcm_rule
from pcm_rule import decode, encode, random_input
from irbaboon_b200 import synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FMTS = ("f32", "s16", "s24")
PAIRS = list(itertools.product(FMTS, FMTS))
PCM_PAIRS = [("s16", "s16"), ("s24", "s24")]


def _same(got, want):
    """bit-for-bit equality of two arrays of one dtype (float32 compared as bits: NaN == NaN, -0 != +0)"""
    assert got.dtype == want.dtype and got.shape == want.shape, (got.dtype, want.dtype, got.shape, want.shape)
    if got.dtype == np.float32:
        return np.array_equal(got.view(np.uint32), want.view(np.uint32))
    return np.array_equal(got, want)


def _ir(seed, n):
    """a decaying IR scaled to sum |h| = 1: outputs of inputs within +-a stay within +-a"""
    h = synth.decaying_ir(seed, n).astype(np.float64)
    return (h / np.abs(h).sum()).astype(np.float32)


def _check_rule(name, run, shape, pairs, seed, level=0.5):
    """run(x, out_format) -> outputs of a freshly reset engine.  For each (fin, fout): PCM-fed output == encode(float output
    of the dequantised input).  -> {(fin, fout): fraction of output samples that are not zero} (the check is not vacuous)"""
    live = {}
    floats = {}
    for fin, fout in pairs:
        x = random_input(shape, fin, seed + FMTS.index(fin), level)
        if fin not in floats:
            floats[fin] = run(decode(x, fin), "f32")
            assert np.isfinite(floats[fin]).all(), name
        y = floats[fin]
        got = run(x, fout)
        want = encode(y, fout)
        if not _same(got, want):
            bad = np.argwhere(got != want) if got.dtype != np.float32 else np.argwhere(got.view(np.uint32) != want.view(np.uint32))
            raise AssertionError("%s (%s -> %s): %d elements differ, first at %s" % (name, fin, fout, len(bad), bad[:5].tolist()))
        live[(fin, fout)] = float(np.count_nonzero(want)) / want.size
        assert live[(fin, fout)] > 0.5, (name, fin, fout, live[(fin, fout)])
    print("%s: %d format pairs bit-exact" % (name, len(pairs)))
    return live


def _engine_run(e, per_block=False):
    def run(x, fout):
        e.reset()
        if per_block:
            return np.stack([e.process(x[k], out_format=fout) for k in range(x.shape[0])])
        return e.process(x, out_format=fout)
    return run


def _runs(pairs):
    """engine runs _check_rule makes: one float run per input format, one run per pair"""
    return len({fin for fin, _ in pairs}) + len(pairs)


def _rows(B):
    """channels per kernel tile at block size B"""
    N = 1
    while N < 2 * B - 1:
        N *= 2
    return 2048 // max(16, N // 2)


# ---- the rule on every block-step form --------------------------------------------------------------------------------------
@pytest.mark.parametrize("B", [129, 300, 512, 1024])
def test_shared_ir_k_mac_p_all_nine_pairs(eng, B):
    P = 4
    C = 75 * _rows(B) + 3                         # enough tiles that no row's partitions are split: the persistent k_mac_p
    with eng.Engine(B, P, C, 1) as e:
        e.set_ir(0, _ir(8001, P * B - 5))
        assert e.mac_plan() == (False, 1, 1)
        _check_rule("shared IR B=%d" % B, _engine_run(e), (P + 3, C, B), PAIRS, 8100 + B)


@pytest.mark.parametrize("B", [129, 300, 512, 1024])
def test_per_row_irs_k_mac_p(eng, B):
    ring = 5
    C = 75 * _rows(B) + 5
    irs = [_ir(8200 + j, max(1, (1 + j % ring) * B - 3 * j)) for j in range(6)]
    bind = (np.arange(C) * 5 + np.arange(C) // 3) % len(irs)
    with eng.Engine(B, ring, C, len(irs)) as e:
        for j, h in enumerate(irs):
            e.set_ir(j, h)
        for c in range(C):
            e.bind(c, c + 1, int(bind[c]))
        assert e.mac_plan() == (True, 1, 1)
        _check_rule("per-row IRs B=%d" % B, _engine_run(e), (ring + 3, C, B), PCM_PAIRS + [("s16", "f32"), ("f32", "s24")], 8300 + B)


@pytest.mark.parametrize("B", [64, 100])
def test_small_block_k_mac_fuse(eng, B):
    """FFT half sizes below 256 take the non-persistent fused step k_mac<FUSE>."""
    P = 6
    C = 75 * _rows(B) + 3
    pairs = PCM_PAIRS + [("s24", "s16")]
    with eng.Engine(B, P, C, 1) as e:
        e.set_ir(0, _ir(8400, P * B - 1))
        assert e.mac_plan() == (False, 1, 1)
        l0 = e.launches
        _check_rule("k_mac<FUSE> B=%d" % B, _engine_run(e), (P + 3, C, B), pairs, 8500 + B)
        assert e.launches - l0 == _runs(pairs) * (P + 3)          # one launch per block step: the forward transform is the MAC's prologue


@pytest.mark.parametrize("B,per_row", [(512, False), (300, False), (512, True)])
def test_two_launch_form(eng, B, per_row):
    """set_fused_step(0): k_fwd reads the new block (its audio rows through load_in), then the MAC kernel."""
    P = 4
    C = 75 * _rows(B) + 1
    irs = [_ir(8600 + j, (j + 1) * B - 2) for j in range(P if per_row else 1)]
    with eng.Engine(B, P, C, len(irs)) as e:
        for j, h in enumerate(irs):
            e.set_ir(j, h)
        if per_row:
            for c in range(C):
                e.bind(c, c + 1, c % P)
        e.set_fused_step(False)
        pairs = PCM_PAIRS + [("s16", "s24")]
        l0 = e.launches
        _check_rule("two-launch B=%d per_row=%d" % (B, per_row), _engine_run(e), (P + 3, C, B), pairs, 8700 + B)
        assert e.launches - l0 == 2 * _runs(pairs) * (P + 3)


def test_cluster_latency_path_stereo_4s_ir(eng):
    """One stereo stream at B = 256 with a 4 s IR (48 kHz): the few-row cluster step k_mac_slots, one block per call (graph
    replays), P + 3 blocks."""
    B, Lh = 256, 4 * 48000
    P = -(-Lh // B)
    with eng.Engine(B, P, 2, 1) as e:
        e.set_ir(0, _ir(8800, Lh))
        slots, split, cluster = e.mac_plan()
        assert slots and split * cluster > 1
        _check_rule("cluster split %d x %d" % (split, cluster), _engine_run(e, per_block=True), (P + 3, 2, B), PCM_PAIRS + [("f32", "s16")], 8900)


@pytest.mark.parametrize("ins,mixed", [(1, False), (1, True), (2, False), (2, True)])
def test_matrix_engine(eng, ins, mixed):
    B, P, G = 512, 4, 301
    irs = [_ir(9000 + j, max(1, (P - j % P) * B - 7 * j)) for j in range(6)]
    with eng.MatrixEngine(B, P, G, ins, 2, len(irs)) as m:
        for j, h in enumerate(irs):
            m.set_ir(j, h)
        if mixed:
            for g in range(0, G, 3):
                m.bind_matrix(g, g + 1, [(g + k) % 6 for k in range(2 * ins)])
        pairs = PAIRS if ins == 2 and not mixed else PCM_PAIRS + [("s16", "f32")]
        _check_rule("matrix (%d, 2) mixed=%d" % (ins, mixed), _engine_run(m), (P + 3, G * ins, B), pairs, 9100 + ins)


def test_group_on_two_devices(eng):
    n = eng.device_count()
    if n < 2:
        pytest.skip("one CUDA device visible: the group spans two")
    B, P, C = 512, 4, 701
    with eng.Group([0, 1], B, P, C, 1) as g:
        g.set_ir(0, _ir(9200, P * B - 3))

        def run(x, fout):
            g.reset()
            return g.process(x, out_format=fout)
        _check_rule("group of 2 devices", run, (P + 3, C, B), PCM_PAIRS + [("s24", "f32")], 9300)


# ---- saturation, NaN taps --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fmt", ["s16", "s24"])
def test_full_scale_inputs_and_a_gain_4_ir_saturate_by_the_rule(eng, fmt):
    B, P, C = 512, 3, 303
    bits = pcm_rule.BITS[fmt]
    top = 1 << (bits - 1)
    rng = np.random.default_rng(bits)
    q = rng.choice(np.array([-top, top - 1, -top + 1, 0, top // 2], np.int64), size=(P + 4, C, B))
    x = q.astype(np.int16) if fmt == "s16" else pcm_rule.pack24(q)
    with eng.Engine(B, P, C, 1) as e:
        e.set_ir(0, (4.0 * synth.decaying_ir(9400, P * B - 1)).astype(np.float32))      # gain 4 (L2 norm): most outputs clip
        e.reset()
        y = e.process(decode(x, fmt))
        assert np.abs(y).max() > 2.0 and (np.abs(y) < 1.0).mean() > 0.05         # well beyond full scale, and inside it
        e.reset()
        got = e.process(x, out_format=fmt)
    assert _same(got, encode(y, fmt))
    codes = got.astype(np.int64) if fmt == "s16" else pcm_rule.unpack24(got)
    assert np.array_equal(codes[y >= 1.0], np.full(int((y >= 1.0).sum()), top - 1))
    assert np.array_equal(codes[y <= -1.0], np.full(int((y <= -1.0).sum()), -top))


@pytest.mark.parametrize("fmt", ["s16", "s24"])
def test_a_nan_tap_gives_zero_codes_only_where_it_is_bound(eng, fmt):
    B, P = 512, 4
    R = _rows(B)
    C = 80 * R
    lo, hi = 10 * R, 30 * R                             # whole tiles bound to IR 1
    clean, dirty = _ir(9500, P * B - 3), _ir(9501, P * B - 3)
    dirty_nan = dirty.copy()
    dirty_nan[B + 17] = np.nan
    x = random_input((P + 4, C, B), fmt, 9502)
    with eng.Engine(B, P, C, 2) as e:
        e.set_ir(0, clean)
        e.set_ir(1, dirty)
        e.bind(lo, hi, 1)
        e.reset()
        ref = e.process(x, out_format=fmt)
        e.set_ir(1, dirty_nan)
        e.reset()
        got = e.process(x, out_format=fmt)
        e.reset()
        yf = e.process(decode(x, fmt))
    assert np.isnan(yf[:, lo:hi]).all()
    assert not np.count_nonzero(got[:, lo:hi])
    others = np.r_[0:lo, hi:C]
    assert _same(got[:, others], ref[:, others])


# ---- device pointers at odd element offsets ------------------------------------------------------------------------------------
@pytest.mark.parametrize("fin,fout", [("s16", "s16"), ("s24", "s24"), ("s16", "s24"), ("s24", "f32")])
def test_device_pointers_at_odd_element_offsets(eng, fin, fout):
    import torch

    B, P, C = 300, 3, 75 * _rows(300) + 1
    nb = P + 3
    x = random_input((nb, C, B), fin, 9600)
    esz = {"f32": 4, "s16": 2, "s24": 3}
    nin, nout = x.nbytes, nb * C * B * esz[fout]
    with eng.Engine(B, P, C, 1) as e:
        e.set_ir(0, _ir(9601, P * B - 1))

        def run(in_off, out_off):
            """element offsets into larger byte tensors; -> (output bytes, bytes around the output)"""
            din = torch.full((nin + 64,), 0x5A, dtype=torch.uint8, device="cuda")
            dout = torch.full((nout + 64,), 0xA5, dtype=torch.uint8, device="cuda")
            a, b = in_off * esz[fin], out_off * esz[fout]
            din[a:a + nin] = torch.from_numpy(np.ascontiguousarray(x).view(np.uint8).reshape(-1)).cuda()
            torch.cuda.synchronize()                        # the engine runs on its own non-blocking stream
            e.reset()
            e.process_device(din.data_ptr() + a, dout.data_ptr() + b, nb, in_format=fin, out_format=fout)
            e.synchronize()
            h = dout.cpu().numpy()
            return h[b:b + nout].copy(), np.concatenate([h[:b], h[b + nout:]])

        base, _ = run(0, 0)
        for in_off, out_off in [(1, 0), (0, 1), (3, 5), (7, 1)]:
            got, around = run(in_off, out_off)
            assert np.array_equal(got, base), (in_off, out_off)
            assert (around == 0xA5).all(), (in_off, out_off)
        e.reset()
        y = e.process(decode(x, fin))
    assert np.array_equal(base, encode(y, fout).view(np.uint8).reshape(-1))


# ---- pipelines and captured graphs -------------------------------------------------------------------------------------------
def test_submitted_blocks_of_different_formats_follow_each_other(eng):
    """Back-to-back submit_pcm calls interleaved with float submits on one engine (the three-stage pipeline keeps running across
    them) equal the same blocks run one at a time."""
    B, P, C = 512, 4, 301
    plan = [("s16", "s16", 3), ("f32", "f32", 2), ("s24", "s24", 4), ("s16", "f32", 2), ("f32", "s24", 3), ("s24", "s16", 2)]
    xs = [random_input((n, C, B), fin, 9700 + k) for k, (fin, fout, n) in enumerate(plan)]
    with eng.Engine(B, P, C, 1) as e:
        e.set_ir(0, _ir(9701, P * B - 9))
        e.reset()
        want = []
        for (fin, fout, n), x in zip(plan, xs):
            want.append(np.stack([e.process(x[k], out_format=fout) for k in range(n)]))
        e.reset()
        ins, outs = [], []
        for (fin, fout, n), x in zip(plan, xs):
            xi = eng.pinned_empty(x.shape, x.dtype)
            xi[...] = x
            oshape = x.shape[:2] + (B * (3 if fout == "s24" else 1),)
            oi = eng.pinned_empty(oshape, {"f32": np.float32, "s16": np.int16, "s24": np.uint8}[fout])
            e.submit(xi, oi, out_format=fout)
            ins.append(xi)
            outs.append(oi)
        e.wait()
        for k, (w, o) in enumerate(zip(want, outs)):
            assert _same(np.array(o), w), plan[k]


def test_one_block_calls_that_alternate_formats_recapture_the_graph(eng):
    """Small blocks replay a captured graph; each run of one format recaptures it (the signature holds both formats), and every
    block equals the float engine's block, encoded."""
    B, P, C = 128, 5, 16
    seq = [("s16", "s16")] * 4 + [("s24", "s24")] * 4 + [("f32", "f32")] * 3 + [("s16", "s24")] * 3 + [("s24", "f32")] * 3 + [("s16", "s16")] * 3
    xs = [random_input((C, B), fin, 9800 + k) for k, (fin, _) in enumerate(seq)]
    with eng.Engine(B, P, C, 1) as e:
        e.set_ir(0, _ir(9801, P * B - 1))
        e.reset()
        yf = [e.process(decode(x, fin)) for x, (fin, _) in zip(xs, seq)]
        e.reset()
        for k, (x, (fin, fout)) in enumerate(zip(xs, seq)):
            assert _same(e.process(x, out_format=fout), encode(yf[k], fout)), (k, fin, fout)


# ---- the C++ facade ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def pc(built, tmp_path_factory):
    fp_dir, lib_dir = os.path.join(ROOT, "irbaboon_b200", "fp"), os.path.join(ROOT, "irbaboon_b200")
    so = str(tmp_path_factory.mktemp("pcm_capi") / "libpcm_capi.so")
    subprocess.check_call(["g++", "-std=c++14", "-O2", "-fPIC", "-shared", "-Wl,-Bsymbolic", "-o", so, os.path.join(ROOT, "tests", "cpp", "pcm_capi.cpp"),
                           "-L" + fp_dir, "-lfp_b200", "-L" + lib_dir, "-lirb_b200", "-Wl,-rpath," + fp_dir, "-Wl,-rpath," + lib_dir])
    L = ctypes.CDLL(so)
    L.pc_create.restype = ctypes.c_void_p
    L.pc_create.argtypes = [ctypes.c_int] * 6
    L.pc_destroy.argtypes = [ctypes.c_int, ctypes.c_void_p]
    L.pc_set_ir.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int]
    L.pc_process.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_int]
    return L


@pytest.mark.parametrize("kind", [0, 1, 2])
def test_cpp_facade_process_pcm(eng, pc, kind):
    """StreamingConvolver / MatrixConvolver (1, 2) / MultiGpuConvolver::process(const void*, irb_sample_format, ...) against the
    python binding on the same IR and blocks."""
    B, P, C = 512, 3, 40
    nb = P + 3
    irs = [_ir(9900 + j, P * B - 5 - j) for j in range(2 if kind == 1 else 1)]
    ndev = max(1, eng.device_count()) if kind == 2 else 1
    h = pc.pc_create(kind, B, P, C, 1, ndev)
    assert h
    try:
        for j, ir in enumerate(irs):
            assert pc.pc_set_ir(kind, h, j, ir.ctypes.data, len(ir)) == 0
        for fin, fout in PCM_PAIRS + [("s16", "s24"), ("s24", "f32")]:
            x = random_input((nb, C, B), fin, 9950)
            if kind == 1:
                py = eng.MatrixEngine(B, P, C, 1, 2, 2)
            elif kind == 2:
                py = eng.Group(list(range(ndev)), B, P, C, 1)
            else:
                py = eng.Engine(B, P, C, 1)
            with py:
                for j, ir in enumerate(irs):
                    py.set_ir(j, ir)
                want = py.process(x, out_format=fout)
            out = np.zeros_like(want)
            assert pc.pc_process(kind, h, x.ctypes.data, eng.sample_format(fin), out.ctypes.data, eng.sample_format(fout), nb) == 0
            assert _same(out, want), (kind, fin, fout)
            # the C++ object keeps its stream state: run the next pair from a fresh one
            pc.pc_destroy(kind, h)
            h = pc.pc_create(kind, B, P, C, 1, ndev)
            for j, ir in enumerate(irs):
                assert pc.pc_set_ir(kind, h, j, ir.ctypes.data, len(ir)) == 0
    finally:
        pc.pc_destroy(kind, h)
