"""float64 statements of the offline spectral functions, written from the reference's semantics (paths relative to the
reference tree), not from oracle/irb_oracle.c: a misreading shared by the C restatement and the kernels does not pass
through these.  tests/test_spectral64_ref.py checks each one against scipy / numpy and the oracle on the CPU before
tests/test_gpu_spectral64.py uses them to judge the device.

Spectra are complex float64 arrays of the bins 0 .. N/2 of an N-point real transform (np.fft.rfft layout) unless a
docstring says otherwise."""
import numpy as np

AMPL_FLOOR = 1e-16          # tools::roundTo1TenQuadrillionth (fp/tools.cpp:212-218)
PHASE_ZERO = 1e-11          # tools::roundToZero threshold of averagingFilter (fp/convolution.cpp:530-543)
SMOOTH_FRACTION = float(np.float32(1.0 / 13.0))     # fp/convolution.cpp:390: a float, widened to double for the call
SMOOTH_PASSES = 3           # fp/convolution.cpp:389-394


def next_pow2(x):
    """tools::nextPowerOfTwo (fp/tools.cpp:184-196): x itself when already a power of two."""
    x = int(x)
    if x > 0 and x & (x - 1) == 0:
        return x
    return 1 << x.bit_length()


def _planar(a):
    a = np.asarray(a, np.float64)
    return a[None, :] if a.ndim == 1 else a


def _lin(a, b, L):
    """linear convolution of rows a [C][La] with b [C or 1][Lb], first L samples, float64"""
    n = next_pow2(a.shape[1] + b.shape[1] - 1)
    return np.fft.irfft(np.fft.rfft(a, n, axis=1) * np.fft.rfft(b, n, axis=1), n, axis=1)[:, :L]


def conv_linear64(x, h):
    """fp::convolution layouts (fp/convolution.cpp:28-42, 176-181, 301-302, 320-323): mono x mono; stereo audio with a mono
    IR (the IR broadcast); mono audio with a stereo IR folded to (L + R) / 2 first (tools::sumToMono, fp/tools.cpp:14-30);
    stereo x stereo channel-wise.  Any other layout: a cleared [ch_x][Lx + Lh - 1].  -> float64 [ch_x][Lx + Lh - 1]"""
    x, h = _planar(x), _planar(h)
    cx, ch = x.shape[0], h.shape[0]
    Lo = x.shape[1] + h.shape[1] - 1
    if cx not in (1, 2) or ch not in (1, 2):
        return np.zeros((cx, Lo))
    if ch == 2 and cx == 1:
        h = (h[0:1] + h[1:2]) / 2
    return _lin(x, h, Lo)


def periodic_written_length(Lx, Lh, B):
    """How much of the linear convolution convolvePeriodic writes (fp/convolution.cpp:52, 104-233): iterations
    Lx / B + P of B samples, P = ceil((float) Lh / (float) B) in float, the last overlap never flushed."""
    P = int(np.ceil(np.float32(Lh) / np.float32(B)))
    return min(Lx + Lh - 1, (Lx // B + P) * B)


def conv_periodic64(x, h, B):
    """fp::convolution::convolvePeriodic: conv_linear64 cut at periodic_written_length; exactly 0 past it."""
    x, h = _planar(x), _planar(h)
    out = conv_linear64(x, h)
    out[:, periodic_written_length(x.shape[1], h.shape[1], B):] = 0.0
    return out


def shifteroo64(y):
    """ir::shifteroo (fp/ir.cpp:85-103): the last floor(n/2) samples move to the front, i.e. out[i] = y[(i + ceil(n/2)) % n]"""
    y = np.asarray(y)
    n = y.shape[-1]
    return np.roll(y, -(n - n // 2), axis=-1)


def _c_round(v):
    """C round() of non-negative doubles: halves away from zero (numpy's round is half to even)"""
    f = np.floor(v)
    return np.where(v - f >= 0.5, f + 1.0, f)


def avg_windows(M, fraction, sr):
    """averagingFilter's window [lo[k], hi[k]] of every bin k = 0 .. M in complex-bin units, with the reference's own double
    operations (fp/convolution.cpp:425, 451-458): freqPerBin = (sr / 2) / M; binFreq = k * freqPerBin;
    lo = round(binFreq / 2^(f/2) / freqPerBin), hi = round(binFreq * 2^(f/2) / freqPerBin)."""
    fpb = (sr / 2.0) / float(M)
    c = 2.0 ** (fraction / 2.0)
    f = np.arange(M + 1, dtype=np.float64) * fpb
    return _c_round((f / c) / fpb).astype(np.int64), _c_round((f * c) / fpb).astype(np.int64)


def _window_sums(v, lo, hi):
    """sum(v[lo[k] .. hi[k]]) of non-negative v, each window summed afresh (no difference of prefix sums, which would lose a
    quiet window next to loud ones): the window is cut into power-of-two blocks whose sums are built pairwise."""
    n = len(v)
    blocks = [np.asarray(v, np.float64)]
    while (1 << len(blocks)) <= n:
        b, s = blocks[-1], 1 << (len(blocks) - 1)
        blocks.append(b[:len(b) - s] + b[s:])                # blocks[j][i] = sum(v[i : i + 2^j])
    out = np.zeros(len(lo))
    pos, width = lo.copy(), hi - lo + 1
    for j in range(len(blocks) - 1, -1, -1):
        take = (width >> j) & 1 == 1
        out[take] += blocks[j][pos[take]]
        pos[take] += 1 << j
    return out


def avg64(spec, fraction, sr, log_avg=True, include_phase=True, include_amplitude=True):
    """fp::convolution::averagingFilter (fp/convolution.cpp:406-546), one pass, in float64, on spec = bins 0 .. M
    (N = 2M-point transform; the reference's fftSize is 4M floats).
    * amplitudes |S[b]| for b <= M (:429-436); bins M < b < 2M (past Nyquist) hold amplitude 0; bins b >= 2M
      ("addBin < fftSize") are skipped, but the window length hi - lo + 1 still counts them;
    * log: each amplitude clamped to >= 1e-16 before the log (:482-505), the window mean, exp, the clamp again (:518-523);
      the window sums come from a float64 cumulative sum -- deliberately NOT the reference's float32 running sum;
    * linear: each window summed afresh (:508-514), no clamp before the mean;
    * each bin's parts rounded to zero below 1e-11 before its phase is taken, include_* acting as INCLUDE flags although
      convolution.hpp:44 names them nullify* (:530-543).
    -> complex float64 bins 0 .. M"""
    S = np.asarray(spec, np.complex128)
    M = S.shape[-1] - 1
    lo, hi = avg_windows(M, fraction, sr)
    top = int(hi.max())
    amp = np.zeros(max(top, M) + 1)
    amp[:M + 1] = np.abs(S)
    if log_avg:
        v = np.log(np.maximum(amp, AMPL_FLOOR))
        v[2 * M:] = 0.0                                      # skipped, never added
        cs = np.concatenate([[0.0], np.cumsum(v)])
        na = np.exp((cs[hi + 1] - cs[lo]) / (hi - lo + 1))
    else:
        na = _window_sums(amp, lo, hi) / (hi - lo + 1)
    na = np.maximum(na, AMPL_FLOOR)
    re = np.where(np.abs(S.real) < PHASE_ZERO, 0.0, S.real)
    im = np.where(np.abs(S.imag) < PHASE_ZERO, 0.0, S.imag)
    ph = np.arctan2(im, re) if include_phase else np.zeros(M + 1)
    a = na if include_amplitude else np.ones(M + 1)
    return a * np.exp(1j * ph)


def quotient64(X, D):
    """tools::complexDivCartesian per bin (fp/tools.cpp:72-86): a denominator bin that is exactly 0 + 0i leaves the numerator bin"""
    zero = D == 0
    return np.where(zero, X, X / np.where(zero, 1.0, D))


def deconv64(num, den, smoothing=True, include_phase=True, include_amplitude=True, sample_rate=48000.0):
    """fp::convolution::deconvolve (fp/convolution.cpp:351-403): N = nextPowerOfTwo(max(len)), both signals zero-padded to N
    (circular division); per-bin quotient (quotient64); with smoothing three 1/13-octave log passes of avg64; inverse
    transform; ir::shifteroo when the phase is dropped (:400), with smoothing or without.  -> float64 [N]"""
    num = np.asarray(num, np.float64).reshape(-1)
    den = np.asarray(den, np.float64).reshape(-1)
    N = next_pow2(max(len(num), len(den)))
    Q = quotient64(np.fft.rfft(num, N), np.fft.rfft(den, N))
    if smoothing:
        for _ in range(SMOOTH_PASSES):
            Q = avg64(Q, SMOOTH_FRACTION, sample_rate, True, include_phase, include_amplitude)
    y = np.fft.irfft(Q, N)
    return y if include_phase else shifteroo64(y)


def invert_filter64(x, sample_rate=48000.0):
    """ir::invertFilter (fp/ir.cpp:13-18): deconvolve(generatePulse(len), x) with the default flags (smoothing on)"""
    x = np.asarray(x, np.float64).reshape(-1)
    pulse = np.zeros(len(x))
    pulse[0] = 1.0                                           # tools::generatePulse (fp/tools.cpp:235-241)
    return deconv64(pulse, x, True, True, True, sample_rate)


def ir_partition_spectra64(x, part):
    """ir::IRtoRealFFTRaw (fp/ir.cpp:106-147): len // part + 1 partitions of `part` samples (the last zero-extended; all zero
    when part divides len), each zero-padded to 2 part and transformed, packed as {Re X[0], Re X[part], re 1, im 1, ...,
    re part-1, im part-1}.  -> float64 [(len // part + 1) * 2 part]"""
    x = np.asarray(x, np.float64).reshape(-1)
    P = len(x) // part + 1
    seg = np.zeros(P * part)
    seg[:len(x)] = x
    X = np.fft.rfft(seg.reshape(P, part), 2 * part, axis=1)
    out = np.empty((P, part, 2))
    out[:, :, 0] = X[:, :part].real
    out[:, :, 1] = X[:, :part].imag
    out[:, 0, 1] = X[:, part].real
    return out.reshape(-1)


def channel_error(got, want):
    """Per row (channel or capture) of got / want [C][n]: (max-abs error over the row's own peak, L2 error over its own
    norm).  A row whose expected value is all zero is judged absolutely.  NaN / Inf in `got` give NaN / Inf."""
    g = np.asarray(got, np.float64)
    w = np.asarray(want, np.float64)
    g = g.reshape(1, -1) if g.ndim == 1 else g.reshape(g.shape[0], -1)
    w = w.reshape(1, -1) if w.ndim == 1 else w.reshape(w.shape[0], -1)
    assert g.shape == w.shape, (g.shape, w.shape)
    d = np.abs(g - w)
    peak = np.abs(w).max(axis=1)
    norm = np.sqrt((w * w).sum(axis=1))
    with np.errstate(invalid="ignore", over="ignore"):
        e = d.max(axis=1) / np.where(peak > 0, peak, 1.0)
        l2 = np.sqrt((d * d).sum(axis=1)) / np.where(norm > 0, norm, 1.0)
    return e, l2
