"""The offline spectral functions against the float64 references of tests/spectral64.py, every channel or capture judged
at its own level (channel_error: max-abs over its own peak, L2 over its own norm), at every FFT plan size class.

Plan classes of an N = 2M point transform (irb_spectral.cu, Plan::init): one pass (line length M) for N <= 4096; M1 x M2
column / row passes above: 64x64 .. 256x256 (N = 8192 .. 2^17), 256x512 .. 512x1024 (2^18 .. 2^20), 1024x1024 (2^21) and
2048x1024 (2^22, the only use of the 2048-point column pass with the split or reciprocal spectrum).

Limits: 1e-5 on both measures.  Where a float32 running sum is part of the reference (the log average of averagingFilter,
smoothed deconvolution), the device must be no farther from float64 than the C oracle's own float32 arithmetic:
err(device, ref64) <= max(1e-5, 2 err(oracle, ref64)) per capture, with err(oracle, ref64) itself bounded so that a broken
reference cannot make that limit vacuous.  Run with -s to see the measured numbers."""
import ctypes

import numpy as np
import pytest

from irbaboon_b200 import synth
from spectral64 import (avg64, channel_error, conv_linear64, conv_periodic64, deconv64, invert_filter64, ir_partition_spectra64,
                        periodic_written_length, shifteroo64)

pytestmark = pytest.mark.gpu

TOL = 1e-5
LAYOUTS = [(1, 1), (2, 1), (1, 2), (2, 2)]
# one N per plan class and both ends of the one-pass range; 2^22 is the largest transform
SIZES = [16, 256, 4096, 8192, 1 << 15, 1 << 18, 1 << 20, 1 << 21, 1 << 22]


def _levels(n, seed):
    """one level per channel or capture, log-uniform over 1e-4 .. 1e2"""
    return (10.0 ** np.random.default_rng(seed).uniform(-4.0, 2.0, n)).astype(np.float32)


def _judge(name, got, want, tol=TOL):
    """both measures <= tol on every row; prints the worst"""
    e, l2 = channel_error(got, want)
    print("%s: %d rows, worst max-abs/own peak %.3g, worst L2/own norm %.3g" % (name, len(e), np.nanmax(e), np.nanmax(l2)))
    ok = (e <= tol) & (l2 <= tol)                                          # NaN fails
    assert ok.all(), (name, np.flatnonzero(~ok)[:8], e, l2)
    return e, l2


def _judge_vs_oracle(name, got, oracle_out, want, drift_limit):
    """per row: err(got, want) <= max(1e-5, 2 err(oracle, want)) on both measures, and err(oracle, want) <= drift_limit"""
    eg, lg = channel_error(got, want)
    eo, lo = channel_error(oracle_out, want)
    print("%s: device max-abs %s L2 %s | oracle max-abs %s L2 %s" % (name, np.array2string(eg, precision=3), np.array2string(lg, precision=3),
                                                                       np.array2string(eo, precision=3), np.array2string(lo, precision=3)))
    assert (eo <= drift_limit).all() and (lo <= drift_limit).all(), (name, eo, lo)
    assert (eg <= np.maximum(TOL, 2 * eo)).all() and (lg <= np.maximum(TOL, 2 * lo)).all(), (name, eg, lg, eo, lo)


def _drift_limit(N):
    """How far the oracle's float32 running sum may sit from float64.  Measured for a white-noise capture over a
    well-conditioned denominator (max-abs over the capture's peak, three smoothing passes): 1e-5 at 2^16, 2e-4 at 2^18, and
    at 2^20 7.6e-4 for a capture at level 1e-4, 1.4e-3 at level 1 and 3.6e-3 at level 1e2 (the larger the log amplitudes,
    the larger the running sum and its rounding); 1.0e-3 at 2^18 for the round trip of a capture with a large DC bin (an
    all-zero denominator).  A float32 sequential sum over the same windows reproduces that gap."""
    return 1e-3 if N <= 1 << 16 else 1e-2


def _sig(ch, n, seed, levels):
    return np.stack([synth.white_noise(seed, c, n) * levels[c] for c in range(ch)]).astype(np.float32)


def _irs(ch, n, seed, levels):
    return np.stack([synth.decaying_ir(seed + c, n, c) * levels[c] for c in range(ch)]).astype(np.float32)


def _den(n, seed, level=1.0):
    """well conditioned: an impulse plus a decaying noise tail of L1 norm 0.9 (every bin within [0.1, 1.9] x level)"""
    t = synth.white_noise(seed, 7, n).astype(np.float64) * np.exp(-np.arange(n) / max(1.0, n / 8.0))
    t[0] = 0.0
    if n > 1:
        t *= 0.9 / np.abs(t).sum()
    t[0] = 1.0
    d = (t * level).astype(np.float32)
    D = np.abs(np.fft.rfft(d.astype(np.float64), max(16, 1 << (n - 1).bit_length())))
    assert D.min() / D.max() >= 1e-2
    return d


def _captures(batch, n, seed):
    return _sig(batch, n, seed, _levels(batch, seed))


# ---- convolveNonPeriodic ----------------------------------------------------------------------------------------------
def _run_layouts(eng, name, Lx, Lh, fn, ref):
    """one stereo input and one stereo IR, each channel at its own level, sliced into the four layouts"""
    x2, h2 = _sig(2, Lx, 100, _levels(2, Lx)), _irs(2, Lh, 200, _levels(2, Lh + 1))
    for chx, chh in LAYOUTS:
        x, h = x2[:chx], h2[:chh]
        _judge("%s %dx%d Lx=%d Lh=%d" % (name, chx, chh, Lx, Lh), fn(x, h), ref(x, h))


@pytest.mark.parametrize("k,extra", [(k, e) for k in range(4, 23) for e in (0, 1) if (k, e) != (22, 1)])
def test_convolve_nonperiodic_every_plan_class(eng, k, extra):
    """Lout = 2^k (N = 2^k) and 2^k + 1 (N = 2^(k+1)): both sides of every plan boundary, in all four layouts, the two audio
    channels and the two IR channels each at its own level."""
    Lout = (1 << k) + extra
    Lh = max(1, (Lout // 3) | 1)
    Lx = Lout - Lh + 1
    _run_layouts(eng, "nonperiodic", Lx, Lh, eng.convolve_nonperiodic, conv_linear64)


@pytest.mark.parametrize("Lx,Lh", [(1, 1), (2, 1), (1, 5), (3, 3), (10, 7)])
def test_convolve_nonperiodic_short_results_are_padded_to_16(eng, Lx, Lh):
    _run_layouts(eng, "nonperiodic", Lx, Lh, eng.convolve_nonperiodic, conv_linear64)


def test_convolve_nonperiodic_largest_result(eng):
    """Lout = 2^22 is accepted (above); 2^22 + 1 needs an FFT above 2^22 points and is refused without touching the output"""
    n = (1 << 21) + 1
    x = np.ones(n, np.float32)
    out = np.full(2 * n - 1, 7.0, np.float32)
    rc = eng.lib().irb_convolve_nonperiodic(eng._ptr(x), 1, n, eng._ptr(x), 1, n, eng._ptr(out))
    assert rc == eng.IRB_ERR_ARG and (out == 7.0).all()


def test_convolve_nonperiodic_rejected_layout(eng):
    x = _sig(3, 100, 1, [1.0, 2.0, 3.0])
    assert not eng.convolve_nonperiodic(x, x[:1]).any() and not conv_linear64(x, x[:1]).any()


# ---- convolvePeriodic ----------------------------------------------------------------------------------------------------
PERIODIC = [(1, 301, 17), (16, 153, 29), (100, 1093, 197), (256, 5000, 700), (2048, 20000, 4000), (2048, 1500, 600), (3000, 2500, 1000),
            (16384, 40000, 16000)]


@pytest.mark.parametrize("B,Lx,Lh", PERIODIC)
def test_convolve_periodic_every_layout(eng, B, Lx, Lh):
    """B = 3000 and 16384 exceed the block kernels and are computed with B = 2048, then cut at the reference's length.
    Every case but B = 1 is cut short of Lx + Lh - 1; past the cut the output is exactly 0."""
    Lw = periodic_written_length(Lx, Lh, B)
    assert B == 1 or Lw < Lx + Lh - 1

    def run(x, h):
        got = eng.convolve_periodic(x, h, B)
        assert not got[:, Lw:].any(), "written past the reference's length"
        return got

    _run_layouts(eng, "periodic B=%d" % B, Lx, Lh, run, lambda x, h: conv_periodic64(x, h, B))


# ---- plain deconvolve / deconvolve_batch ---------------------------------------------------------------------------------
@pytest.mark.parametrize("N", SIZES)
def test_deconvolve_plain_every_plan_class(eng, N):
    """len_num and len_den unequal both ways and odd; three captures at their own levels over one denominator; the single
    entry on the first capture; include_phase = false (the shifted plain division) on the same inputs."""
    for ln, ld in ((N - 3, N // 2 + 3), (N // 2 + 5, N - 1)):
        caps = _captures(3, ln, N + ln)
        den = _den(ld, ld, float(_levels(1, ld)[0]))
        want = np.stack([deconv64(c, den, False) for c in caps])
        tag = "deconvolve N=%d len_num=%d len_den=%d" % (N, ln, ld)
        _judge(tag, eng.deconvolve_batch(caps, den, 48000.0, False), want)
        _judge(tag + " single", eng.deconvolve(caps[0], den, 48000.0, False), want[:1])
        _judge(tag + " no phase", eng.deconvolve_batch(caps, den, 48000.0, False, False), shifteroo64(want))


@pytest.mark.parametrize("N", [4096, 1 << 16])
def test_deconvolve_batch_across_sub_batches(eng, N):
    caps = _captures(5, N - 1, N)
    den = _den(N // 3, 9, 3.0)
    want = np.stack([deconv64(c, den, False) for c in caps])
    try:
        eng.set_tuning("deconv_sub", 2)                      # sub-batches of 2, 2, 1
        got = eng.deconvolve_batch(caps, den, 48000.0, False)
        got_np = eng.deconvolve_batch(caps, den, 48000.0, False, False)
    finally:
        eng.set_tuning("deconv_sub", 0)
    _judge("deconvolve sub-batches N=%d" % N, got, want)
    _judge("deconvolve sub-batches no phase N=%d" % N, got_np, shifteroo64(want))


def _device_batch(eng, caps, den, N, phase, den_on_device):
    import torch

    d_caps = torch.from_numpy(np.ascontiguousarray(caps)).cuda()
    d_out = torch.zeros((caps.shape[0], N), dtype=torch.float32, device="cuda")
    if den_on_device:
        d_den = torch.from_numpy(den).cuda()
        torch.cuda.synchronize()
        rc = eng.lib().irb_deconvolve_batch_device(ctypes.c_void_p(d_caps.data_ptr()), caps.shape[0], caps.shape[1], ctypes.c_void_p(d_den.data_ptr()),
                                                   len(den), 48000.0, 0, int(phase), 1, ctypes.c_void_p(d_out.data_ptr()))
        assert rc == 0, eng.lib().irb_last_error()
    else:
        eng.deconvolve_batch_device(d_caps.data_ptr(), caps.shape[0], caps.shape[1], den, d_out.data_ptr(), 48000.0, False, phase, True)
    torch.cuda.synchronize()
    return d_out.cpu().numpy()


@pytest.mark.parametrize("N,ln", [(1 << 16, 1 << 16), (1 << 16, (1 << 16) - 1), (8192, 8190), (1 << 22, (1 << 22) - 2), (1 << 21, (1 << 21) - 3)])
@pytest.mark.parametrize("den_on_device", [False, True])
def test_deconvolve_batch_device_paths(eng, N, ln, den_on_device):
    """Even lengths (aligned torch buffers) take the unstaged path, odd ones the staged device-to-device copies; the phase-free
    division always goes through the staged path.  The denominator as a host and as a device pointer."""
    caps = _captures(3, ln, ln + 5)
    den = _den(N // 4 + 1, N, 0.3)
    want = np.stack([deconv64(c, den, False) for c in caps])
    tag = "deconvolve_batch_device N=%d len=%d den %s" % (N, ln, "device" if den_on_device else "host")
    _judge(tag, _device_batch(eng, caps, den, N, True, den_on_device), want)
    _judge(tag + " no phase", _device_batch(eng, caps, den, N, False, den_on_device), shifteroo64(want))


# ---- the zero-denominator rule ------------------------------------------------------------------------------------------
# DC and Nyquist share bin 0 of the packed spectrum and are the only bins that can be made exactly zero short of an all-zero
# denominator (tests/test_spectral64_ref.py checks that these constructions are exact).  Such a denominator is ill-conditioned
# next to its zero (|D[1]| ~ 2 pi / N), so only the untouched bin itself is compared: the output's own spectrum there must be
# the numerator's bin -- not 0, inf or NaN.
ZERO_DENS = {"dc": ([1.0, -1.0], [0]), "nyquist": ([1.0, 1.0], [-1]), "both": ([1.0, 0.0, -1.0], [0, -1])}


def _zero_num(N, seed):
    """noise plus a DC offset and a Nyquist tone, so both untouched bins stand well above the rest"""
    n = np.arange(N)
    return (synth.white_noise(seed, 0, N) * np.float32(0.5) + np.float32(0.75) + np.float32(0.5) * np.where(n % 2, -1.0, 1.0)).astype(np.float32)


@pytest.mark.parametrize("N", [16, 4096, 8192, 1 << 18, 1 << 21, 1 << 22])
@pytest.mark.parametrize("smoothing", [False, True])
def test_zero_denominator_bins(eng, orc, N, smoothing):
    num = _zero_num(N, N)
    X = np.fft.rfft(num.astype(np.float64))
    for kind, (taps, bins) in ZERO_DENS.items():
        den = np.asarray(taps, np.float32)
        got = eng.deconvolve(num, den, 48000.0, smoothing)[0]
        assert np.isfinite(got).all(), kind
        G = np.fft.rfft(got.astype(np.float64))
        W = np.fft.rfft(deconv64(num, den, smoothing))
        for b in bins:
            err = abs(G[b] - W[b]) / abs(X[b])
            print("zero-bin %s N=%d smoothing=%d bin %d: |got - want| / |X| = %.3g" % (kind, N, smoothing, b % (N // 2 + 1), err))
            assert err <= 1e-3, (kind, b, G[b], W[b], X[b])
    # an all-zero denominator leaves every bin: the numerator's own round trip
    zero = np.zeros(7, np.float32)
    caps = _captures(2, N - 1, N + 3)
    got = eng.deconvolve_batch(caps, zero, 48000.0, smoothing)
    assert np.isfinite(got).all()
    want = np.stack([deconv64(c, zero, smoothing) for c in caps])
    if not smoothing:
        _judge("zero-den all N=%d" % N, got, want)
    elif N <= 1 << 18:
        orc_out = np.concatenate([orc.deconvolve(c, zero, 48000.0, True) for c in caps])
        _judge_vs_oracle("zero-den all smoothed N=%d" % N, got, orc_out, want, _drift_limit(N))


# ---- smoothed deconvolution and averagingFilter ---------------------------------------------------------------------------
FLAGS = [(True, True), (False, True), (True, False), (False, False)]


@pytest.mark.parametrize("N,flags", [(n, f) for n in (1 << 12, 1 << 14, 1 << 16) for f in FLAGS] + [(n, f) for n in (1 << 18, 1 << 20) for f in FLAGS[:2]])
def test_deconvolve_smoothed(eng, orc, N, flags):
    caps = _captures(2, N - 5, N + 11)
    den = _den(N // 4 + 3, N + 1, 2.0)
    got = eng.deconvolve_batch(caps, den, 48000.0, True, *flags)
    orc_out = np.concatenate([orc.deconvolve(c, den, 48000.0, True, *flags) for c in caps])
    want = np.stack([deconv64(c, den, True, *flags) for c in caps])
    _judge_vs_oracle("deconvolve smoothed N=%d phase=%d ampl=%d" % ((N,) + flags), got, orc_out, want, _drift_limit(N))


def _spectra(N, ch, seed):
    x = _sig(ch, N, seed, _levels(ch, seed)) * np.exp(-np.arange(N) / (N / 6.0)).astype(np.float32)
    S = np.fft.rfft(x.astype(np.float64), axis=1)
    spec = np.zeros((ch, 2 * N), np.float32)
    spec[:, 0:N + 2:2], spec[:, 1:N + 2:2] = S.real, S.imag
    spec[:, N + 2:] = np.float32(0.5)                        # bins past N/2: never read, never written
    return spec


def _avg_case(eng, orc, N, fraction, sr, log_avg, flags, seed):
    spec = _spectra(N, 2, seed)
    got = eng.averaging_filter(spec, fraction, sr, log_avg, *flags)
    assert np.array_equal(got[:, N + 2:], spec[:, N + 2:])
    S = spec[:, 0:N + 2:2].astype(np.float64) + 1j * spec[:, 1:N + 2:2].astype(np.float64)
    A = np.stack([avg64(s, fraction, sr, log_avg, *flags) for s in S])
    want = np.zeros((2, N + 2))
    want[:, 0::2], want[:, 1::2] = A.real, A.imag
    tag = "averaging_filter N=%d fraction=1/%g sr=%g log=%d phase=%d ampl=%d" % ((N, 1 / fraction, sr, log_avg) + tuple(flags))
    if log_avg:
        _judge_vs_oracle(tag, got[:, :N + 2], orc.averaging_filter(spec, fraction, sr, True, *flags)[:, :N + 2], want, _drift_limit(N))
    else:
        _judge(tag, got[:, :N + 2], want)


@pytest.mark.parametrize("N", [1 << 12, 1 << 16, 1 << 20])
@pytest.mark.parametrize("flags", FLAGS[:3])
def test_averaging_filter_log(eng, orc, N, flags):
    _avg_case(eng, orc, N, 1.0 / 13.0, 48000.0, True, flags, N)


@pytest.mark.parametrize("N", [1 << 12, 1 << 16, 1 << 20])
def test_averaging_filter_linear(eng, orc, N):
    _avg_case(eng, orc, N, 1.0 / 3.0, 48000.0, False, (True, True), N + 1)


@pytest.mark.parametrize("fraction", [1.0 / 6.0, 1.0 / 3.0])
@pytest.mark.parametrize("sr", [44100.0, 96000.0])
@pytest.mark.parametrize("log_avg", [True, False])
def test_averaging_filter_fractions_and_rates(eng, orc, fraction, sr, log_avg):
    _avg_case(eng, orc, 1 << 16, fraction, sr, log_avg, (True, True), int(sr) + int(1 / fraction))


@pytest.mark.parametrize("n", [1 << 16, 1 << 20, 1 << 21])
def test_ess_capture(eng, orc, n):
    """ESS capture deconvolution (a 20 Hz .. 20 kHz sweep, a decaying IR, -60 dB noise), plain and smoothed.  The sweep's
    spectrum falls outside its band, so the division is ill-conditioned there and the float32 reference itself moves."""
    sweep = synth.exp_sine_sweep(n / 48000.0, 48000.0, 20.0, 20000.0).astype(np.float32)[:n]
    h = synth.decaying_ir(3000 + n % 7, n // 8)
    cap = conv_linear64(sweep, h)[0, :n].astype(np.float32) + synth.white_noise(4000, 0, n) * np.float32(1e-3)
    for smoothing in (False, True):
        got = eng.deconvolve(cap, sweep, 48000.0, smoothing)
        _judge_vs_oracle("ESS n=%d smoothing=%d" % (n, smoothing), got, orc.deconvolve(cap, sweep, 48000.0, smoothing),
                         deconv64(cap, sweep, smoothing)[None], _drift_limit(n))


# ---- fftInvTransform, IRtoRealFFTRaw, invertFilter ----------------------------------------------------------------------------
@pytest.mark.parametrize("N", SIZES)
def test_fft_inv_transform(eng, N):
    """From a spectrum built in float64: the imaginary parts of DC and Nyquist and every bin past N/2 are ignored"""
    rng = np.random.default_rng(N)
    lev = _levels(2, N + 1)
    S = (rng.standard_normal((2, N // 2 + 1)) + 1j * rng.standard_normal((2, N // 2 + 1))) * lev[:, None]
    spec = rng.standard_normal((2, 2 * N)).astype(np.float32) * np.float32(1e3)
    spec[:, 0:N + 2:2], spec[:, 1:N + 2:2] = S.real, S.imag
    S32 = spec[:, 0:N + 2:2].astype(np.float64) + 1j * spec[:, 1:N + 2:2].astype(np.float64)
    _judge("fft_inv_transform N=%d" % N, eng.fft_inv_transform(spec), np.fft.irfft(S32, N, axis=1))


@pytest.mark.parametrize("part", [16, 32, 64, 128, 256, 512, 1024, 2048])
def test_ir_to_real_fft_raw(eng, part):
    """len a multiple of part (the extra partition is all zero) and not; every partition at its own level"""
    for n in (5 * part, 5 * part + 7):
        P = n // part + 1
        lev = np.repeat(_levels(P, part + n), part)[:n]
        x = (synth.white_noise(part, n, n) * lev).astype(np.float32)
        got = eng.ir_to_real_fft_raw(x, part).reshape(P, 2 * part)
        want = ir_partition_spectra64(x, part).reshape(P, 2 * part)
        if n % part == 0:
            assert not got[-1].any()
            got, want = got[:-1], want[:-1]
        _judge("ir_to_real_fft_raw part=%d len=%d" % (part, n), got, want)


@pytest.mark.parametrize("n", [1000, (1 << 15) + 3, 1 << 18])
def test_invert_filter(eng, orc, n):
    x = _den(n, n + 2, 0.4)
    N = 1 << (n - 1).bit_length()
    _judge_vs_oracle("invert_filter len=%d" % n, eng.invert_filter(x, 48000), orc.invert_filter(x, 48000), invert_filter64(x)[None], _drift_limit(N))
