"""The batched linear convolution (irb_convolve_batch, irb_convolve_batch_device) on the device: bit-identical rows to
irb_convolve_nonperiodic at one N per FFT plan class, windows that are exact slices of the full result, float64 accuracy per row,
every pipeline route (sub-batches, slot reuse, host and device entries, staged and staging-free device paths), isolation of rows
under NaN / Inf, and the Farina capture (SURVEY section 4, KA1): the windowed IR of a sweep capture peaks where the delay puts it."""
import numpy as np
import pytest

from irbaboon_b200 import synth
from spectral64 import channel_error, conv_linear64

pytestmark = pytest.mark.gpu

TOL = 1e-5
# one N per plan class of the FFT (as tests/test_gpu_spectral64.py): one pass up to 4096, then 64x64 .. 2048x1024 four-step
SIZES = [16, 256, 4096, 8192, 1 << 15, 1 << 18, 1 << 20, 1 << 21, 1 << 22]


def _lengths(N, odd):
    """len_x, len_h whose linear result needs exactly N points (7N/8 .. N samples); odd: both lengths odd, else both even"""
    lh, lx = max(1, N // 4), N // 2 + N // 8
    if odd:
        lh, lx = lh + 1, lx + 1
    assert N // 2 < lx + lh - 1 <= N
    return lx, lh


def _levels(n, seed):
    return (10.0 ** np.random.default_rng(seed).uniform(-4.0, 2.0, n)).astype(np.float32)


def _signals(batch, n, seed, levels=None):
    lv = np.ones(batch, np.float32) if levels is None else levels
    return np.stack([synth.white_noise(seed, b, n) * lv[b] for b in range(batch)]).astype(np.float32)


def _irs(nh, n, seed, levels=None):
    lv = np.ones(nh, np.float32) if levels is None else levels
    return np.stack([synth.decaying_ir(seed + j, n, j) * lv[j] for j in range(nh)]).astype(np.float32)


def _judge(name, got, want, tol=TOL):
    e, l2 = channel_error(got, want)
    print("%s: %d rows, worst max-abs/own peak %.3g, worst L2/own norm %.3g" % (name, len(e), np.nanmax(e), np.nanmax(l2)))
    ok = (e <= tol) & (l2 <= tol)
    assert ok.all(), (name, np.flatnonzero(~ok)[:8], e, l2)


@pytest.fixture
def torch_cuda():
    import torch
    assert torch.cuda.is_available()
    return torch


@pytest.fixture
def sub_batch(eng):
    """sets the sub-batch size of the batched pipelines for one test, then restores it"""
    old = eng.get_tuning("deconv_sub")
    yield lambda n: eng.set_tuning("deconv_sub", n)
    eng.set_tuning("deconv_sub", old)


def _dev_call(torch, eng, x, h, per_item_on_device=False, off=0, n=None, x_shift=0, out_shift=0):
    """irb_convolve_batch_device on copies of x (and h) in device memory, x and out placed x_shift / out_shift floats past an
    allocation's start (1: only 4-byte aligned) -> host array"""
    batch, lx = x.shape
    lh = h.shape[-1]
    hb = 1 if h.ndim == 1 else h.shape[0]
    n = lx + lh - 1 - off if n is None else n
    dx = torch.zeros(batch * lx + 2, dtype=torch.float32, device="cuda")
    dx[x_shift:x_shift + batch * lx] = torch.from_numpy(np.ascontiguousarray(x).reshape(-1)).cuda()
    do = torch.full((batch * n + 2,), 7.0, dtype=torch.float32, device="cuda")
    xp, op = dx.data_ptr() + 4 * x_shift, do.data_ptr() + 4 * out_shift
    if per_item_on_device:
        dh = torch.from_numpy(np.ascontiguousarray(h, np.float32)).cuda()
        eng.convolve_batch_device(xp, batch, lx, dh.data_ptr(), op, len_h=lh, h_batch=hb, out_offset=off, out_len=n)
    else:
        eng.convolve_batch_device(xp, batch, lx, h, op, out_offset=off, out_len=n)
    torch.cuda.synchronize()
    got = do.cpu().numpy()
    assert (got[:out_shift] == 7.0).all() and (got[out_shift + batch * n:] == 7.0).all()     # nothing written outside the rows
    return got[out_shift:out_shift + batch * n].reshape(batch, n)


# ---- bit identity with irb_convolve_nonperiodic --------------------------------------------------------------------------------------
@pytest.mark.parametrize("N", SIZES)
@pytest.mark.parametrize("per_item", [False, True])
@pytest.mark.parametrize("odd", [False, True])
def test_full_window_rows_equal_convolve_nonperiodic(eng, N, per_item, odd):
    """irb_convolve_nonperiodic runs on the same core (batch 1 here), so this shows that batching, sub-batches and per-item
    strides leave every row's bits alone; what the rows are worth is judged against float64 below and by the existing tests of
    irb_convolve_nonperiodic"""
    lx, lh = _lengths(N, odd)
    batch = 3
    x = _signals(batch, lx, N + odd)
    h = _irs(batch if per_item else 1, lh, 17 + N)
    got = eng.convolve_batch(x, h if per_item else h[0])
    assert got.shape == (batch, lx + lh - 1)
    for b in range(batch):
        want = eng.convolve_nonperiodic(x[b], h[b if per_item else 0])[0]
        assert np.array_equal(got[b], want), (N, per_item, odd, b)
    assert eng.last_compute_ms() > 0.0


# ---- windows ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N", [256, 4096, 1 << 15, 1 << 20])
@pytest.mark.parametrize("per_item", [False, True])
def test_windows_are_exact_slices_of_the_full_result(eng, torch_cuda, N, per_item):
    lx, lh = _lengths(N, False)                                             # even lengths: an odd result length
    full_len = lx + lh - 1
    batch = 3
    x = _signals(batch, lx, 5 + N)
    h = _irs(batch if per_item else 1, lh, 23)
    hh = h if per_item else h[0]
    full = eng.convolve_batch(x, hh)
    windows = [(0, full_len), (0, 1), (full_len - 1, 1), (1, 1), (3, 7), (lh - 1, 2 * lx // 3 + 1), (full_len // 3, full_len - full_len // 3),
               (0, lx), (full_len - 5, 5)]
    for off, n in windows:
        want = full[:, off:off + n]
        assert np.array_equal(eng.convolve_batch(x, hh, off, n), want), (off, n)
        # device entry, staging-free for N > 4096 (x 8-byte aligned, even len_x); the windowed store takes a 4-byte aligned out
        assert np.array_equal(_dev_call(torch_cuda, eng, x, h if per_item else hh, per_item, off, n, out_shift=1), want), (off, n)
        assert np.array_equal(_dev_call(torch_cuda, eng, x, hh, False, off, n), want), (off, n)


# ---- float64 ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N", [256, 4096, 1 << 15, 1 << 20, 1 << 22])
@pytest.mark.parametrize("per_item", [False, True])
def test_rows_match_float64(eng, N, per_item):
    lx, lh = _lengths(N, False)
    batch = 6
    x = _signals(batch, lx, 31 + N, _levels(batch, N))
    h = _irs(batch if per_item else 1, lh, 41, _levels(batch if per_item else 1, N + 1))
    got = eng.convolve_batch(x, h if per_item else h[0])
    want = np.concatenate([conv_linear64(x[b], h[b if per_item else 0]) for b in range(batch)])
    _judge("convolve_batch N=%d per_item=%s" % (N, per_item), got, want)


# ---- pipeline routes ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,batch,sub", [(1 << 15, 1, 0), (1 << 15, 11, 3), (4096, 11, 3), (1 << 18, 40, 0), (1 << 20, 7, 2)])
@pytest.mark.parametrize("per_item", [False, True])
def test_every_route_gives_the_same_bits(eng, torch_cuda, sub_batch, N, batch, sub, per_item):
    """sub-batches that do not divide the batch and reuse both staging slots (and every compute stream of the device path); host
    and device entries; h in host and in device memory; x at 4-byte alignment and with an odd length (staged device route)"""
    lx, lh = _lengths(N, False)
    x = _signals(batch, lx, 61 + batch, _levels(batch, batch))
    h = _irs(batch if per_item else 1, lh, 71)
    hh = h if per_item else h[0]
    want = np.stack([eng.convolve_nonperiodic(x[b], h[b if per_item else 0])[0] for b in range(batch)])
    sub_batch(sub)
    assert np.array_equal(eng.convolve_batch(x, hh), want)
    assert np.array_equal(_dev_call(torch_cuda, eng, x, hh), want)
    assert np.array_equal(_dev_call(torch_cuda, eng, x, h, per_item_on_device=True), want)
    assert np.array_equal(_dev_call(torch_cuda, eng, x, h, per_item_on_device=True, x_shift=1, out_shift=1), want)
    xo = np.ascontiguousarray(x[:, :lx - 1])
    want_o = np.stack([eng.convolve_nonperiodic(xo[b], h[b if per_item else 0])[0] for b in range(batch)])
    assert np.array_equal(_dev_call(torch_cuda, eng, xo, h, per_item_on_device=True), want_o)
    assert np.array_equal(eng.convolve_batch(xo, hh), want_o)
    if per_item:                                                            # odd len_h: the per-item IRs are staged
        ho = np.ascontiguousarray(h[:, :lh - 1])
        want_h = np.stack([eng.convolve_nonperiodic(x[b], ho[b])[0] for b in range(batch)])
        assert np.array_equal(_dev_call(torch_cuda, eng, x, ho, per_item_on_device=True), want_h)


@pytest.mark.parametrize("per_item", [False, True])
def test_more_short_signals_than_one_launch_takes(eng, torch_cuda, per_item):
    """70 000 signals at N = 16: the per-item launches take at most 65 535 items each, so the batch runs in several sub-batches"""
    batch, lx, lh = 70000, 9, 4
    rng = np.random.default_rng(7)
    x = rng.standard_normal((batch, lx)).astype(np.float32)
    h = rng.standard_normal((batch if per_item else 1, lh)).astype(np.float32)
    hh = h if per_item else h[0]
    got = eng.convolve_batch(x, hh)
    want = np.stack([np.convolve(x[b].astype(np.float64), h[b if per_item else 0].astype(np.float64)) for b in range(batch)])
    _judge("70000 x N=16 per_item=%s" % per_item, got, want)
    for b in (0, 65534, 65535, 65536, batch - 1):
        assert np.array_equal(got[b], eng.convolve_nonperiodic(x[b], h[b if per_item else 0])[0]), b
    assert np.array_equal(_dev_call(torch_cuda, eng, x, h, per_item_on_device=per_item), got)


def test_shared_ir_given_as_one_row_equals_the_flat_ir(eng):
    x = _signals(4, 3000, 3)
    h = _irs(1, 700, 4)
    assert np.array_equal(eng.convolve_batch(x, h), eng.convolve_batch(x, h[0]))


# ---- isolation ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N", [4096, 1 << 18])
@pytest.mark.parametrize("bad", ["nan_signal", "inf_signal", "nan_ir", "inf_ir"])
def test_a_non_finite_row_changes_no_other_row(eng, torch_cuda, N, bad):
    lx, lh = _lengths(N, False)
    batch = 5
    x = _signals(batch, lx, 81)
    h = _irs(batch, lh, 91)
    clean = eng.convolve_batch(x, h)
    x2, h2 = x.copy(), h.copy()
    if bad.endswith("signal"):
        x2[2, lx // 3] = np.nan if bad.startswith("nan") else np.inf
    else:
        h2[2, lh // 2] = np.nan if bad.startswith("nan") else -np.inf
    for got in (eng.convolve_batch(x2, h2), _dev_call(torch_cuda, eng, x2, h2, per_item_on_device=True)):
        assert not np.isfinite(got[2]).all()
        for b in (0, 1, 3, 4):
            assert np.array_equal(got[b], clean[b]), (bad, b)
    if bad.endswith("signal"):                                              # and with one shared IR
        clean_s = eng.convolve_batch(x, h[0])
        got = eng.convolve_batch(x2, h[0])
        for b in (0, 1, 3, 4):
            assert np.array_equal(got[b], clean_s[b]), (bad, b)


# ---- Farina capture (SURVEY section 4, KA1) ---------------------------------------------------------------------------------------
SR = 48000.0
PRE, POST = 4800, 48000


@pytest.fixture(scope="module")
def sweeps(eng):
    n = 1 << 20
    sweep = eng.ess(n / SR, SR, 20.0, 24000.0).astype(np.float32)
    inv = eng.ess(n / SR, SR, 20.0, 24000.0, 0.0, True).astype(np.float32)
    return sweep, inv


@pytest.mark.parametrize("kind", ["pulse", "decaying"])
def test_farina_window_peaks_at_the_delay(eng, sweeps, kind):
    sweep, inv = sweeps
    n, d = 1 << 20, 1234
    h_true = np.zeros(d + 24000, np.float32)
    h_true[d] = 1.0
    if kind == "decaying":
        h_true[d + 1:] = 0.3 * synth.decaying_ir(5, len(h_true) - d - 1)
    caps = np.stack([eng.convolve_nonperiodic(sweep, h_true)[0, :n], eng.convolve_nonperiodic(sweep, 0.5 * h_true)[0, :n]])
    off = len(sweep) - 1 - PRE
    got = eng.convolve_batch(caps, inv, off, PRE + POST)
    assert got.shape == (2, PRE + POST)
    for b in range(2):
        assert int(np.argmax(np.abs(got[b]))) == PRE + d, (b, int(np.argmax(np.abs(got[b]))))
    want = np.concatenate([conv_linear64(caps[b], inv)[:, off:off + PRE + POST] for b in range(2)])
    _judge("farina %s" % kind, got, want)
    # the full result's slice, bit for bit
    full = eng.convolve_batch(caps[:1], inv)
    assert np.array_equal(full[0, off:off + PRE + POST], got[0])
