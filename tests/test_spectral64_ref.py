"""The float64 references of tests/spectral64.py, checked on the CPU before they judge the device: against scipy / numpy,
and against the C oracle where its float32 arithmetic has not drifted yet (N <= 2^14)."""
import numpy as np
import pytest

from irbaboon_b200 import synth
from spectral64 import (SMOOTH_FRACTION, avg64, avg_windows, channel_error, conv_linear64, conv_periodic64, deconv64, invert_filter64,
                        ir_partition_spectra64, next_pow2, periodic_written_length, quotient64, shifteroo64)

LAYOUTS = [(1, 1), (2, 1), (1, 2), (2, 2)]


def _sig(ch, n, seed, levels):
    return np.stack([synth.white_noise(seed, c, n) * np.float32(levels[c]) for c in range(ch)])


def _ir(ch, n, seed, levels):
    return np.stack([synth.decaying_ir(seed + c, n, c) * np.float32(levels[c]) for c in range(ch)])


def well_conditioned_den(n, seed, level=1.0):
    """An impulse plus a decaying noise tail whose L1 norm is 0.9: every bin of its spectrum lies within [0.1, 1.9] x level"""
    t = synth.white_noise(seed, 7, n).astype(np.float64) * np.exp(-np.arange(n) / max(1.0, n / 8.0))
    t[0] = 0.0
    if n > 1:
        t *= 0.9 / np.abs(t).sum()
    t[0] = 1.0
    return (t * level).astype(np.float32)


def _err_ok(got, want, tol):
    e, l2 = channel_error(got, want)
    assert (e <= tol).all() and (l2 <= tol).all(), (e, l2)
    return e, l2


# ---- convolution layouts ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("chx,chh", LAYOUTS)
@pytest.mark.parametrize("Lx,Lh,B", [(1093, 197, 100), (153, 29, 16), (2500, 1000, 3000), (301, 17, 1), (1500, 600, 2048), (5000, 700, 256)])
def test_conv_references_match_scipy_and_the_oracle(orc, chx, chh, Lx, Lh, B):
    """Ragged lengths, B > Lx, Lh < B; channels six decades apart, so a quiet channel is judged at its own level."""
    from scipy.signal import fftconvolve

    x = _sig(chx, Lx, 10 + chx, [1e-3, 30.0][:chx])
    h = _ir(chh, Lh, 20 + chh, [2.0, 1e-2][:chh])
    got = conv_linear64(x, h)
    x64, h64 = x.astype(np.float64), h.astype(np.float64)
    if chh == 1:
        hh = [h64[0]] * chx
    else:
        hh = [(h64[0] + h64[1]) / 2] if chx == 1 else [h64[0], h64[1]]
    want = np.stack([fftconvolve(x64[c], hh[c]) for c in range(chx)])
    assert got.shape == want.shape == (chx, Lx + Lh - 1)
    assert (np.abs(got - want).max(axis=1) <= 1e-12 * np.abs(want).max(axis=1)).all()
    _err_ok(orc.convolve_nonperiodic(x, h), got, 1e-5)
    per = conv_periodic64(x, h, B)
    Lw = periodic_written_length(Lx, Lh, B)
    assert Lw == min(Lx + Lh - 1, orc.periodic_iterations(Lx, Lh, B) * B)
    assert np.array_equal(per[:, :Lw], got[:, :Lw]) and not per[:, Lw:].any()
    _err_ok(orc.convolve_periodic(x, h, B), per, 1e-5)
    assert not orc.convolve_periodic(x, h, B)[:, Lw:].any()


def test_conv_rejected_layout_is_cleared(orc):
    x, h = _sig(3, 50, 1, [1, 1, 1]), _ir(1, 7, 2, [1])
    assert not conv_linear64(x, h).any() and conv_linear64(x, h).shape == (3, 56)
    assert not conv_periodic64(x, _ir(3, 7, 2, [1, 1, 1]), 16).any()
    assert not orc.convolve_periodic(x, h, 16).any()


def test_periodic_partition_count_is_a_float_division():
    """P = ceil((float) Lh / (float) B): for Lh = 2^24 + 1 the float quotient rounds down to a whole number of blocks"""
    assert periodic_written_length(1, (1 << 24) + 1, 1 << 20) == (0 + 16) * (1 << 20)
    assert periodic_written_length(10, 100, 7) == min(109, (1 + 15) * 7)


# ---- deconvolution ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N", [16, 64, 1024, 4096, 1 << 14])
@pytest.mark.parametrize("smoothing,phase,ampl", [(s, p, a) for s in (False, True) for p in (False, True) for a in (False, True)])
def test_deconv64_matches_the_oracle(orc, N, smoothing, phase, ampl):
    for ln, ld in ((N - 3, N // 2 + 3), (N // 2 + 5, N - 1)):
        num = synth.white_noise(11, ln, ln) * np.float32(0.01)
        den = well_conditioned_den(ld, ld, 3.0)
        want = deconv64(num, den, smoothing, phase, ampl)
        assert want.shape == (N,)
        _err_ok(orc.deconvolve(num, den, 48000.0, smoothing, phase, ampl), want[None], 1e-5)


def test_deconv64_plain_is_the_circular_quotient_and_drops_the_phase_by_a_half_swap():
    N = 256
    num = synth.white_noise(1, 0, N).astype(np.float64)
    den = well_conditioned_den(N, 2).astype(np.float64)
    y = deconv64(num, den, False)
    back = np.real(np.fft.ifft(np.fft.fft(y) * np.fft.fft(den)))
    assert np.abs(back - num).max() <= 1e-12
    assert np.array_equal(deconv64(num, den, False, False), np.concatenate([y[N // 2:], y[:N // 2]]))
    assert np.array_equal(shifteroo64(np.arange(5)), [3, 4, 0, 1, 2])              # odd n: ceil(n/2) to the back


def test_invert_filter64_matches_the_oracle(orc):
    for n in (100, 1000, 3000):
        x = well_conditioned_den(n, n, 0.5)
        _err_ok(orc.invert_filter(x, 48000), invert_filter64(x)[None], 2e-6)


# ---- averagingFilter --------------------------------------------------------------------------------------------------
def _spec(N, seed, level):
    x = synth.white_noise(seed, 0, N) * np.exp(-np.arange(N) / (N / 6.0)).astype(np.float32) * np.float32(level)
    return x


@pytest.mark.parametrize("N", [64, 1024, 8192])
@pytest.mark.parametrize("fraction", [1.0 / 13.0, 1.0 / 6.0, 1.0 / 3.0])
@pytest.mark.parametrize("sr", [44100.0, 48000.0, 96000.0])
@pytest.mark.parametrize("log_avg", [True, False])
def test_avg64_matches_the_oracle(orc, N, fraction, sr, log_avg):
    M = N // 2
    for flags in ((True, True), (False, True), (True, False)):
        x = _spec(N, N + int(sr), 0.05)
        spec = orc.fft_transform(x)                            # [1][2N] interleaved
        got = orc.averaging_filter(spec, fraction, sr, log_avg, *flags)[0, :N + 2]
        S = spec[0, 0:N + 2:2].astype(np.float64) + 1j * spec[0, 1:N + 2:2].astype(np.float64)
        want = avg64(S, fraction, sr, log_avg, *flags)
        assert want.shape == (M + 1,)
        w = np.empty(N + 2)
        w[0::2], w[1::2] = want.real, want.imag
        _err_ok(got[None], w[None], 2e-6)


def test_avg_windows_reach_past_nyquist_and_count_skipped_bins():
    """The top windows reach past Nyquist (bins M < b < 2M count as amplitude 0, clamped to 1e-16 before the log): a flat
    spectrum of amplitude 1 averages to exp(n_past * log(1e-16) / len) at the top bins.  Bins b >= 2M are skipped but counted
    in the window length: a wide fraction at a tiny M shows it."""
    for M, fraction in ((64, 1.0 / 3.0), (8, 4.0)):        # 4 octaves: two per side, the top windows reach 4M > 2M
        lo, hi = avg_windows(M, fraction, 48000.0)
        assert hi[M] > M and lo[0] == 0 and hi[0] == 0
        past = np.clip(np.minimum(hi, 2 * M - 1) - np.maximum(lo, M + 1) + 1, 0, None)
        got = np.abs(avg64(np.ones(M + 1, np.complex128), fraction, 48000.0))
        assert np.allclose(got, np.exp(past * np.log(1e-16) / (hi - lo + 1)), rtol=1e-12)
    assert hi.max() >= 2 * M


def test_avg64_linear_has_no_floor_and_phase_is_taken_after_rounding_to_zero():
    S = np.array([4.0, 1e-12 - 1e-12j, -2.0 + 5e-12j, 3.0, 0.0], np.complex128)
    out = avg64(S, 1e-9, 48000.0, False)                   # a window of one bin: the amplitude is kept
    assert np.allclose(np.abs(out), np.maximum(np.abs(S), 1e-16), rtol=1e-12)
    assert out[1] == np.abs(S[1]) and np.angle(out[2]) == np.pi and out[0] == 4.0


# ---- IRtoRealFFTRaw ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("part", [16, 256, 2048])
def test_ir_partition_spectra64(orc, part):
    for n in (3 * part, 3 * part + 7):
        x = synth.white_noise(5, part, n)
        got = ir_partition_spectra64(x, part).reshape(-1, 2 * part)
        assert got.shape[0] == n // part + 1
        for p in range(got.shape[0]):
            seg = np.zeros(2 * part)
            s = x[p * part:(p + 1) * part].astype(np.float64)
            seg[:len(s)] = s
            X = np.fft.rfft(seg)
            assert got[p, 0] == X[0].real and got[p, 1] == X[part].real
            assert np.array_equal(got[p, 2::2], X[1:part].real) and np.array_equal(got[p, 3::2], X[1:part].imag)
        if n % part == 0:
            assert not got[-1].any()
    buf = np.zeros(4 * part, np.float32)
    buf[:part] = x[:part]
    full = orc.real_forward(buf, 2 * part)                    # 2*part interleaved complex bins
    want = np.concatenate([[full[0], full[2 * part]], full[2:2 * part]])
    assert np.abs(ir_partition_spectra64(x, part)[:2 * part] - want).max() <= 1e-5 * np.abs(want).max()


# ---- zero-denominator constructions ------------------------------------------------------------------------------
# Only bin 0 of the packed spectrum -- DC and Nyquist, both real -- can be made exactly zero short of an all-zero
# denominator: the DC bin is a plain sum and the Nyquist bin an alternating sum of the samples, both exact for small
# integers, while every other bin involves roots of unity that are irrational in float and never cancel exactly.
ZERO_DENS = {"dc": ([1.0, -1.0], [0], [-1]), "nyquist": ([1.0, 1.0], [-1], [0]), "both": ([1.0, 0.0, -1.0], [0, -1], []),
             "all": ([0.0] * 5, None, None)}


@pytest.mark.parametrize("N", [16, 4096, 1 << 16])
@pytest.mark.parametrize("kind", list(ZERO_DENS))
def test_zero_denominator_constructions_are_exact(N, kind):
    taps, zero_bins, nonzero_bins = ZERO_DENS[kind]
    D = np.fft.rfft(np.asarray(taps, np.float64), N)
    D32 = np.fft.rfft(np.asarray(taps, np.float32), N)
    if zero_bins is None:
        assert not D.any()
        return
    for b in zero_bins:
        assert D[b] == 0 and D32[b] == 0
    for b in nonzero_bins:
        assert D[b] != 0
    assert (D[1:-1] != 0).all()
    num = synth.white_noise(3, 0, N).astype(np.float64) + 0.25
    X = np.fft.rfft(num, N)
    Q = quotient64(X, D)
    for b in zero_bins:
        assert Q[b] == X[b]
    y = deconv64(num, taps, False)
    Y = np.fft.rfft(y)
    for b in zero_bins:
        assert abs(Y[b] - X[b]) <= 1e-9 * abs(X).max()


def test_channel_error_judges_each_row_at_its_own_level():
    want = np.stack([np.linspace(-1, 1, 100) * 100.0, np.linspace(-1, 1, 100) * 1e-3])
    got = want.copy()
    got[1] *= 1 + 1e-3
    e, l2 = channel_error(got, want)
    assert e[0] == 0 and abs(e[1] - 1e-3) < 1e-9 and abs(l2[1] - 1e-3) < 1e-9
    e, _ = channel_error(np.array([[0.0, 2e-9]]), np.zeros((1, 2)))
    assert e[0] == 2e-9
    e, _ = channel_error(np.array([[np.nan, 0.0]]), np.ones((1, 2)))
    assert not (e <= 1).any()


def test_next_pow2_and_smooth_fraction():
    assert [next_pow2(n) for n in (1, 2, 3, 16, 17)] == [1, 2, 4, 16, 32]
    assert SMOOTH_FRACTION == float(np.float32(1.0 / 13.0)) and SMOOTH_FRACTION != 1.0 / 13.0
