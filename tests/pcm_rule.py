"""numpy statement of the engine's PCM conversions (include/irb_b200.h, irb_sample_format), shared by the PCM tests.

decode: integer -> float32 value / 2^(bits-1).  encode: float32 -> the integer-WAV writer's rule in float64 (y <= -1 -> INT32_MIN,
y >= 1 -> INT32_MAX, NaN -> 0, otherwise round-half-even(2147483647 * y)), then an arithmetic shift right by 32 - bits.
tests/test_pcm_abi.py pins encode to the facade's formats::writeWav bytes."""
import numpy as np

BITS = {"s16": 16, "s24": 24}


def quantise(y, bits):
    """float32 array -> int64 codes of `bits` bits"""
    d = np.asarray(y, np.float32).astype(np.float64)
    with np.errstate(invalid="ignore"):
        q = np.rint(d * 2147483647.0)
        q = np.where(np.isnan(d), 0.0, np.where(d <= -1.0, -2147483648.0, np.where(d >= 1.0, 2147483647.0, q)))
    return q.astype(np.int64) >> (32 - bits)


def pack24(q):
    """int codes [..][n] -> uint8 [..][3n], little-endian, packed"""
    u = np.asarray(q, np.int64) & 0xFFFFFF
    b = np.stack([u & 0xFF, (u >> 8) & 0xFF, (u >> 16) & 0xFF], axis=-1).astype(np.uint8)
    return np.ascontiguousarray(b.reshape(b.shape[:-2] + (-1,)))


def unpack24(b):
    """uint8 [..][3n] -> int64 codes [..][n]"""
    b = np.asarray(b, np.uint8)
    t = b.reshape(b.shape[:-1] + (-1, 3)).astype(np.int64)
    u = t[..., 0] | (t[..., 1] << 8) | (t[..., 2] << 16)
    return np.where(u >= 1 << 23, u - (1 << 24), u)


def encode(y, fmt):
    """float32 [..][n] -> the engine's output array of format fmt ("f32", "s16", "s24")"""
    if fmt == "f32":
        return np.ascontiguousarray(y, np.float32)
    if fmt == "s16":
        return quantise(y, 16).astype(np.int16)
    return pack24(quantise(y, 24))


def decode(a, fmt):
    """the engine's input array of format fmt -> float32 [..][n], exactly as the device reads it"""
    if fmt == "f32":
        return np.asarray(a, np.float32)
    if fmt == "s16":
        return (np.asarray(a, np.int16).astype(np.float64) / 32768.0).astype(np.float32)
    return (unpack24(a).astype(np.float64) / 8388608.0).astype(np.float32)


def random_input(shape, fmt, seed, level=0.5):
    """[..][B] input in format fmt: uniform at `level` of full scale"""
    rng = np.random.default_rng(seed)
    if fmt == "f32":
        return ((rng.random(shape) * 2 - 1) * level).astype(np.float32)
    bits = BITS[fmt]
    top = 1 << (bits - 1)
    q = rng.integers(-int(top * level), int(top * level), size=shape, dtype=np.int64)
    return q.astype(np.int16) if fmt == "s16" else pack24(q)
