"""The batched IR chop on the device (irb_ir_chop_batch_device) and the capture batch that ends with it (irb_deconvolve_chop_batch):
rows and positions bit-identical to the facade's fp::ir::IRchop + fp::tools::normalize on every corner of the rule (after checking
in float64 that no row sits on a glibc-vs-correctly-rounded decision flip), the documented rule on a row that does, isolation of
NaN / Inf rows, both peak-pass routes, the capture batch equal to the full division chopped afterwards on every pipeline route and
plan class, a known-answer capture, and the facade's capturesToIRs equal to captureToIR + chopAndNormalize per capture."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import chop_rule
from irbaboon_b200 import synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_f32p = ctypes.POINTER(ctypes.c_float)
SIZES = [16, 256, 4096, 8192, 1 << 15, 1 << 18, 1 << 20, 1 << 22]        # one N per plan class of the FFT


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available()
    return torch


@pytest.fixture(scope="module")
def fac(built):
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "tests", "cpp")])
    h = ctypes.CDLL(os.path.join(ROOT, "tests", "cpp", "libfacade_capi.so"))
    h.fac_ir_chop.argtypes = [_f32p, ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_int, _f32p]
    h.fac_normalize.argtypes = [_f32p, ctypes.c_int, ctypes.c_int, ctypes.c_float]
    h.fac_capture_to_ir.argtypes = [_f32p, ctypes.c_int, ctypes.c_int, _f32p, ctypes.c_int, ctypes.c_double, _f32p, _f32p]
    h.fac_chop_and_normalize.argtypes = [_f32p, ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_int, _f32p]
    return h


@pytest.fixture(scope="module")
def helper(built, tmp_path_factory):
    return chop_rule.build_helper(tmp_path_factory.mktemp("chop_rule_gpu"))


@pytest.fixture
def sub_batch(eng):
    old = eng.get_tuning("deconv_sub")
    yield lambda n: eng.set_tuning("deconv_sub", n)
    eng.set_tuning("deconv_sub", old)


def _fp(a):
    return a.ctypes.data_as(_f32p)


def _same(a, b):
    """bit for bit, except that any NaN equals any NaN (the device's arithmetic returns the canonical NaN, x86 keeps the payload)"""
    a, b = np.ascontiguousarray(a, np.float32), np.ascontiguousarray(b, np.float32)
    if a.shape != b.shape or not np.array_equal(np.isnan(a), np.isnan(b)):
        return False
    keep = ~np.isnan(a)
    return np.array_equal(a[keep].view(np.uint32), b[keep].view(np.uint32))


def _facade(fac, x, L, thr, c, normalize=True, goal_db=0.0):
    x = np.ascontiguousarray(x, np.float32)
    out = np.empty(L, np.float32)
    assert fac.fac_ir_chop(_fp(x), len(x), L, thr, c, _fp(out)) == L
    if normalize:
        fac.fac_normalize(_fp(out), 1, L, goal_db)
    return out


def _device(eng, torch, rows, L, thr, c, normalize=True, goal_db=0.0, offset=0):
    """rows [batch][n] -> (out [batch][L], positions [batch][2]); offset: floats of padding in front (a 4-byte aligned x)"""
    rows = np.ascontiguousarray(rows, np.float32)
    b, n = rows.shape
    flat = torch.zeros(offset + b * n, dtype=torch.float32, device="cuda")
    flat[offset:] = torch.from_numpy(rows.reshape(-1)).cuda()
    out = torch.full((b, L), 7.0, dtype=torch.float32, device="cuda")
    pos = torch.full((b, 2), -1, dtype=torch.int32, device="cuda")
    eng.ir_chop_batch_device(flat.data_ptr() + 4 * offset, b, n, L, out.data_ptr(), thr, c, normalize, goal_db, pos.data_ptr())
    torch.cuda.synchronize()
    return out.cpu().numpy(), pos.cpu().numpy()


@pytest.mark.parametrize("seed", [0, 1, 2])
@pytest.mark.parametrize("normalize,goal_db", [(True, 0.0), (False, 0.0), (True, -6.0)])
def test_rows_equal_the_facade(eng, torch_cuda, fac, helper, seed, normalize, goal_db):
    for name, x, L, thr, c in chop_rule.cases(seed):
        assert chop_rule.decisions_agree(helper, x, L, thr), name          # the facade and the rule decide alike on this row
        got, pos = _device(eng, torch_cuda, x[None, :], L, thr, c, normalize, goal_db)
        want = _facade(fac, x, L, thr, c, normalize, goal_db)
        _, q, start = chop_rule.chop(helper, x, L, thr, c, rule=True)
        assert _same(got[0], want), (name, pos, q, start)
        assert tuple(pos[0]) == (q, start), name


def test_rows_equal_the_reference(eng, torch_cuda, helper, ref):
    for name, x, L, thr, c in chop_rule.cases(3):
        if not chop_rule.decisions_agree(helper, x, L, thr):
            continue
        got, _ = _device(eng, torch_cuda, x[None, :], L, thr, c, normalize=False)
        assert _same(got[0], ref.ir_chop(x, L, thr, c)[0]), name


def test_a_row_on_a_decision_flip_follows_the_documented_rule(eng, torch_cuda, fac, helper):
    """samples whose facade level is one ulp below the rule's, with the threshold at the rule's level: loud for the device, quiet for
    the facade, so the cuts differ, and the device's is the rule's"""
    v = (ctypes.c_float * 1)()
    assert helper.chop_find_level_flips(np.float32(1e-3).view(np.uint32).item(), v, 1) == 1
    v = np.float32(v[0])
    thr = float(chop_rule.levels(helper, np.array([v]), True)[0])       # level(peak 1.0) = 0 dB on both sides
    x = np.full(256, 1e-9, np.float32)
    x[200] = 1.0
    x[190:200] = v
    got, pos = _device(eng, torch_cuda, x[None, :], 64, thr, 5)
    want_rule, q, start = chop_rule.chop(helper, x, 64, thr, 5, rule=True, normalize=True)
    assert (q, start) == (200, 200 - 16) and tuple(pos[0]) == (q, start)   # walk positions 1..10 loud, 11..15 quiet
    assert _same(got[0], want_rule)
    assert chop_rule.chop(helper, x, 64, thr, 5, rule=False)[2] == 200 - 6   # the facade: quiet from position 1
    assert not _same(got[0], _facade(fac, x, 64, thr, 5))


@pytest.mark.parametrize("n,L", [(4096, 1024), (1 << 22, 48000), (1 << 20, 2048)])
def test_batches_rows_and_routes(eng, torch_cuda, fac, helper, n, L):
    """a batch is its rows chopped one by one; both peak-pass routes (16-byte aligned rows, and rows at an odd float offset) agree;
    a NaN or Inf row changes no other row by a bit"""
    rng = np.random.default_rng(n)
    b = 6 if n >= 1 << 20 else 40
    rows = np.stack([synth.white_noise(10 + r, 0, n) * np.float32(1e-6) for r in range(b)]).astype(np.float32)
    for r in range(b):
        q = int(rng.integers(0, n))
        t = np.arange(min(n - q, 20000))
        rows[r, q:q + len(t)] += (np.exp(-t / 3000.0) * synth.white_noise(100 + r, 1, len(t)) * 0.5).astype(np.float32)
        rows[r, q] = 1.0
    got, pos = _device(eng, torch_cuda, rows, L, -60.0, 50)
    for r in range(b) if n <= 4096 else (0, b - 1):
        assert chop_rule.decisions_agree(helper, rows[r], L, -60.0)
        assert _same(got[r], _facade(fac, rows[r], L, -60.0, 50)), r
    for r in range(b):
        one, p1 = _device(eng, torch_cuda, rows[r:r + 1], L, -60.0, 50)
        assert _same(got[r], one[0]) and np.array_equal(pos[r], p1[0]), r
    odd, podd = _device(eng, torch_cuda, rows, L, -60.0, 50, offset=1)
    assert _same(odd, got) and np.array_equal(podd, pos)
    for bad in (np.nan, np.inf, -np.inf):
        hurt = rows.copy()
        hurt[1, ::7] = bad
        h, hp = _device(eng, torch_cuda, hurt, L, -60.0, 50)
        keep = [r for r in range(b) if r != 1]
        assert _same(h[keep], got[keep]) and np.array_equal(hp[keep], pos[keep]), bad


def _captures(batch, n, seed):
    sweep = synth.exp_sine_sweep(max(n // 2, 8) / 48000.0, 48000.0, 20.0, 20000.0).astype(np.float32)[: max(n // 2, 8)]
    nums = np.stack([synth.white_noise(seed, b, n) * np.exp(-np.arange(n) / max(4.0, n / 8)).astype(np.float32) for b in range(batch)])
    return nums.astype(np.float32), sweep


@pytest.mark.parametrize("N", SIZES)
@pytest.mark.parametrize("smoothing", [0, 1])
@pytest.mark.parametrize("phase", [1, 0])
def test_capture_batch_equals_the_division_chopped(eng, torch_cuda, sub_batch, N, smoothing, phase):
    """irb_deconvolve_chop_batch row b == irb_deconvolve_batch row b chopped on the device: batch 1, and a batch of sub-batches of 2
    (several smoothing groups side by side), with positions"""
    if smoothing and N == 1 << 22 and phase == 0:
        pytest.skip("one smoothed 2^22 case (phase kept) covers the largest smoothed plan")
    L = min(N, 2048) if N > 16 else 16
    for batch, sub in ((1, 0), (5, 2)):
        sub_batch(sub)
        nums, den = _captures(batch, N, 7 + N)
        full = eng.deconvolve_batch(nums, den, smoothing=bool(smoothing), include_phase=bool(phase))
        got, pos = eng.deconvolve_chop_batch(nums, den, L, smoothing=bool(smoothing), include_phase=bool(phase), return_positions=True)
        want, wpos = _device(eng, torch_cuda, full, L, -60.0, 50)
        assert _same(got, want) and np.array_equal(pos, wpos), (batch, N)


def test_known_answer_capture(eng, torch_cuda, helper):
    """sweep * (a decaying IR delayed by d samples), divided by the sweep: the peak sits at d, the cut starts where the rule puts it,
    and the IR peaks at goal_db"""
    sr, d, L = 48000.0, 3000, 4096
    sweep = eng.ess(1.0, sr, 20.0, 24000.0).astype(np.float32)
    h = np.zeros(d + 2000, np.float32)
    h[d] = 1.0
    h[d + 1:] = 0.3 * synth.decaying_ir(5, 1999)
    caps = np.stack([eng.convolve_nonperiodic(sweep, g * h)[0] for g in (1.0, 0.25)]).astype(np.float32)
    out, pos = eng.deconvolve_chop_batch(caps, sweep, L, sample_rate=sr, goal_db=-3.0, return_positions=True)
    full = eng.deconvolve_batch(caps, sweep, sample_rate=sr)
    goal = np.float32(10.0 ** (-3.0 / 20.0))
    for b in range(2):
        _, q, start = chop_rule.chop(helper, full[b], L, -60.0, 50, rule=True)
        assert pos[b, 0] == d == q and pos[b, 1] == start
        assert d - 150 <= start <= d - 50                 # the division's floor is far below -60 dB: the walk stops soon after 50 samples
        assert abs(float(np.abs(out[b]).max()) - float(goal)) <= 2e-7
        assert np.argmax(np.abs(out[b])) == d - start


def test_captures_to_irs_equals_the_chain_per_capture(fac, helper):
    """fp::b200::capturesToIRs == captureToIR + chopAndNormalize on each capture (smoothing on, the plug-in's default)"""
    H, nb, L, sr = 1024, 64, 2048, 48000.0
    n = H * nb
    sweep = np.zeros(n, np.float32)
    sweep[:40000] = synth.exp_sine_sweep(40001 / sr, sr, 20.0, 24000.0).astype(np.float32)[:40000]
    caps, wants = [], []
    for j in range(3):
        hj = synth.decaying_ir(300 + j, 3000 + 500 * j, j)
        cap = np.ascontiguousarray(np.convolve(sweep.astype(np.float64), hj.astype(np.float64))[:n].astype(np.float32) + synth.white_noise(9 + j, 0, n) * np.float32(1e-4))
        rec, ir = np.zeros(n, np.float32), np.zeros(n, np.float32)
        assert fac.fac_capture_to_ir(_fp(cap), nb, H, _fp(sweep), n, sr, _fp(rec), _fp(ir)) == n
        assert chop_rule.decisions_agree(helper, ir, L, -60.0)
        want = np.empty(L, np.float32)
        assert fac.fac_chop_and_normalize(_fp(ir), n, L, -60.0, 50, _fp(want)) == L
        caps.append(rec)
        wants.append(want)
    caps = np.ascontiguousarray(np.stack(caps))
    got = np.empty((3, L), np.float32)
    assert helper.chop_captures_to_irs(_fp(caps), 3, n, _fp(sweep), n, sr, L, -60.0, 50, 1, _fp(got)) == 0
    assert _same(got, np.stack(wants))
