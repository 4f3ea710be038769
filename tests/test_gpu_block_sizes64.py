"""The small-block streaming step against float64 on every channel, and both sides of each block-size boundary.

Block sizes 1 .. 128 run FFT half sizes M = 16, 32, 64, 128 (B <= 8 still uses M = 16), below the persistent kernel's
M >= 256, so their block step runs other kernels (irb_engine.cu, launch_mac_t):
* shared IR, many rows: k_mac<M, 1, true, FUSE, WIDE> in one launch per block (forward transform in its prologue), or
  k_fwd + k_mac (the two-launch form);
* per-row IRs: k_fwd + k_mac_slots, two launches per block even with the fused step on;
* few rows (automatic or forced split): k_mac_slots over tile slots and a thread-block cluster, the forward transform on
  cluster rank 0, one launch per block.
Every case asserts mac_plan() and the launch count, so it shows which kernel ran, and compares EVERY channel with ref64
(test_gpu_isolation.py), each channel at its own input level and judged against its own peak and norm.  Also: long IRs,
no IR at all, the persistent kernel at B = 129, 257, 513, 1025 (half of each transform is padding), the matrix engine's
smallest block size and the multi-device group at B = 64.
"""
import numpy as np
import pytest

from irbaboon_b200 import synth
from test_gpu_isolation import _every_channel, _gains, _irs, _noise, _planar, ref64, ref64_matrix

SMS = 148                  # B200: a launch of at most SMS / 2 tiles splits its rows' partitions (engine_check_binding)


def _half(B):
    """FFT half size of a block size (irb_engine.cu, half_size_for_block)"""
    N = 1
    while N < 2 * B - 1:
        N *= 2
    return max(16, N // 2)


def _rows(B):
    """rows (channels) per kernel tile"""
    return 2048 // _half(B)


def _noise_many(C, nb, B, seed, gains=None):
    """_noise, vectorised over the channels: the same samples (synth.white_noise stream c for channel c)"""
    n = nb * B
    x = np.empty((C, n), np.float32)
    t = np.arange(n, dtype=np.uint64)[None, :]
    for c0 in range(0, C, 4096):
        c = np.arange(c0, min(C, c0 + 4096), dtype=np.uint64)[:, None]
        with np.errstate(over="ignore"):
            u = synth.splitmix64(np.uint64(seed) + (c << np.uint64(40)) + t)
        x[c0:c0 + len(c)] = ((u >> np.uint64(40)).astype(np.float64) * (1.0 / 16777216.0) * 2.0 - 1.0).astype(np.float32)
    if gains is not None:
        x *= gains[:, None]
    return np.ascontiguousarray(x.reshape(C, nb, B).transpose(1, 0, 2))


def _judge(name, y, x, irs, bind, B, nb):
    """y, x: [nb][C][B] output and input; every channel against the float64 convolution with its IR"""
    _every_channel(name, _planar(y), ref64(_planar(x), irs, bind, B, nb))


def _judge_matrix(name, y, x, irs, mats, ins, B, nb):
    """the same for an IR-matrix engine with two outputs per group"""
    _every_channel(name, _planar(y), ref64_matrix(_planar(x), irs, mats, ins, 2, B, nb))


def _run(e, x, singles, chunk):
    """x [nb][C][B] through e.process: the first `singles` blocks one per call (small blocks replay a CUDA graph from the
    second call on), the rest in calls of up to `chunk` blocks (the multi-block pipeline).  -> (y, launches)"""
    l0 = e.launches
    ys = [e.process(x[k]) for k in range(min(singles, len(x)))]
    for k in range(singles, len(x), chunk):
        ys.extend(e.process(x[k:k + chunk]))
    return np.stack(ys), e.launches - l0


def _bind_runs(e, bind):
    """bind channel c to IR bind[c], one call per run of equal IRs"""
    c0 = 0
    for c in range(1, len(bind) + 1):
        if c == len(bind) or bind[c] != bind[c0]:
            e.bind(c0, c, int(bind[c0]))
            c0 = c


def _per_row_irs(B, ring, n, seed):
    """n IRs of 1 .. ring partitions, IR j scaled by its own gain (1e-2 .. 1e2)"""
    irs = [synth.decaying_ir(seed + j, (1 + j * (ring - 1) // (n - 1)) * B - j % B, j) for j in range(n)]
    return [(h * np.float32(10.0 ** (-2.0 + 4.0 * j / (n - 1)))).astype(np.float32) for j, h in enumerate(irs)]


def _mixed_bind(C, n):
    """IR per channel such that every tile of at least 3 rows holds several IRs"""
    return (np.arange(C) * 5 + np.arange(C) // 3) % n


# ---- 0. the model at these block sizes, on the CPU --------------------------------------------------------------------
@pytest.mark.parametrize("B", [1, 2, 8, 9, 17, 33, 65, 128, 1025])
def test_ref64_at_small_block_sizes(orc, B):
    """IRs of 1 tap, exactly k*B taps and k*B + 1 taps; an input that ends inside a block (a whole block early at B = 1);
    channels at levels six decades apart.  ref64 against scipy (1e-12) and the oracle's streaming form (1e-5 per channel)."""
    from scipy.signal import fftconvolve

    k = 3
    lens = [1, k * B, k * B + 1]
    nb = max(5, 64 // B + k + 2)
    n = nb * B - (B // 3 + 1)
    C = 2 * len(lens) + 1
    irs = [synth.decaying_ir(900 + j, L, j) for j, L in enumerate(lens)]
    bind = np.arange(C) % len(lens)
    x = np.stack([synth.white_noise(901, c, n) for c in range(C)]) * _gains(C, B)[:, None]
    got = ref64(x, irs, bind, B, nb)
    assert got.shape == (C, nb * B)
    off = np.zeros((C, nb * B))
    for c in range(C):
        want = np.zeros(nb * B)
        full = fftconvolve(x[c].astype(np.float64), irs[bind[c]].astype(np.float64))[:nb * B]
        want[:len(full)] = full
        assert np.abs(got[c] - want).max() <= 1e-12 * np.abs(want).max(), c
        o = orc.convolve_periodic(x[c], irs[bind[c]], B)[0, :nb * B]
        off[c, :len(o)] = o
    _every_channel("oracle B=%d" % B, off, got)


def test_vectorised_noise_is_the_per_channel_noise():
    g = _gains(5, 3)
    assert np.array_equal(_noise_many(5, 3, 7, 123, g), _noise(5, 3, 7, 123, g))
    assert np.array_equal(_noise_many(4100, 1, 2, 9)[:, 4097], _noise(4100, 1, 2, 9)[:, 4097])


# ---- 1. shared IR, many rows: k_mac fused and its two-launch form ---------------------------------------------------------
# (B, P, IR length): every small M, B on both sides of each M boundary; more than SMS / 2 tiles, a partial last tile,
# nb = P + 4 blocks so the FDL ring wraps
_SHARED = [(1, 6, "PB"), (8, 5, "1"), (9, 4, "PB-1"), (16, 5, "(P-1)B+1"), (17, 3, "PB"), (32, 6, "PB-1"),
           (33, 4, "(P-1)B+1"), (64, 5, "1"), (65, 4, "PB"), (128, 5, "PB-1")]


def _ir_len(kind, P, B):
    return {"1": 1, "PB": P * B, "PB-1": max(1, P * B - 1), "(P-1)B+1": (P - 1) * B + 1}[kind]


@pytest.mark.gpu
@pytest.mark.parametrize("fused", [True, False])
@pytest.mark.parametrize("B,P,kind", _SHARED)
def test_every_channel_shared_ir_small_blocks(eng, B, P, kind, fused):
    R = _rows(B)
    C = (76 + B % 5) * R + R // 2 + 1
    nb = P + 4
    h = synth.decaying_ir(9100 + B, _ir_len(kind, P, B))
    x = _noise_many(C, nb, B, 9101 + B, _gains(C, B))
    with eng.Engine(B, P, C, 1) as e:
        assert e.tile_channels == R and e.fft_size == 2 * _half(B)
        e.set_ir(0, h)
        e.set_fused_step(fused)
        assert e.mac_plan() == (False, 1, 1)
        y, launches = _run(e, x, 3, 4)
    assert launches == (1 if fused else 2) * nb
    _judge("M=%d shared IR B=%d C=%d P=%d Lh=%d fused=%d" % (_half(B), B, C, P, len(h), fused), y, x, [h], 0, B, nb)


# ---- 2. one full-GPU case per small M ---------------------------------------------------------------------------------------
# k_mac<M, 1, true, true, true> (the fused step): 72 registers x 288 threads (cuobjdump --dump-resource-usage), 17-21 KB of
# shared memory, __launch_bounds__(288, 3): 3 CTAs per SM, so 444 tiles run at once on 148 SMs at every M = 16 .. 128.
# 925 tiles are 2.1 waves (118 358 channels at B = 13); 14 blocks are 3.5 laps of a 4-slot FDL ring.
@pytest.mark.gpu
@pytest.mark.parametrize("B", [13, 32, 50, 128])
def test_full_gpu_every_channel_small_blocks(eng, B):
    R, P, nb = _rows(B), 4, 14
    C = 925 * R - R // 3
    h = synth.decaying_ir(9200 + B, P * B - 2)
    x = _noise_many(C, nb, B, 9201 + B, _gains(C, 7 + B))
    with eng.Engine(B, P, C, 1) as e:
        e.set_ir(0, h)
        assert e.mac_plan() == (False, 1, 1)
        y, launches = _run(e, x, 2, 4)
    assert launches == nb
    _judge("M=%d full GPU B=%d C=%d (%d tiles)" % (_half(B), B, C, -(-C // R)), y, x, [h], 0, B, nb)


# ---- 3. per-row IRs at each small M: k_fwd + k_mac_slots ---------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("B", [11, 32, 40, 128])
def test_every_channel_per_row_irs_small_blocks(eng, B):
    """8 IRs of 1 .. ring partitions, each at its own gain, bound so that every tile mixes them.  k_mac_slots holds one CTA
    per SM (126 registers x 288 threads), so 160 tiles are more than one wave."""
    R, ring = _rows(B), 7
    C = 160 * R + R // 2 + 3
    nb = ring + 4
    irs = _per_row_irs(B, ring, 8, 9300)
    assert len(set(-(-len(h) // B) for h in irs)) >= 6 and max(-(-len(h) // B) for h in irs) == ring
    bind = _mixed_bind(C, len(irs))
    assert all(len(set(bind[t:t + R])) > 1 for t in range(0, C, R))
    x = _noise_many(C, nb, B, 9301 + B, _gains(C, 11 + B))
    with eng.Engine(B, ring, C, len(irs)) as e:
        for j, h in enumerate(irs):
            e.set_ir(j, h)
        _bind_runs(e, bind)
        e.set_fused_step(True)
        assert e.mac_plan() == (True, 1, 1)
        y, launches = _run(e, x, 3, 4)
    assert launches == 2 * nb
    _judge("M=%d per-row IRs B=%d C=%d" % (_half(B), B, C), y, x, irs, bind, B, nb)


# ---- 4. few rows: k_mac_slots split over tile slots and a cluster --------------------------------------------------------------
# the automatic plan (engine_check_binding: two CTAs per SM, at least 4 partitions per range)
_AUTO = [  # (B, C, IR taps, plan)
    (16, 3, 2000, (True, 16, 1)),
    (32, 5, 24000, (True, 64, 2)),
    (64, 2, 48000, (True, 32, 4)),              # a plug-in's stereo pair at B = 64 with a 1 s IR at 48 kHz
    (100, 1, 48000, (True, 16, 4)),
]


@pytest.mark.gpu
@pytest.mark.parametrize("B,C,Lh,plan", _AUTO)
def test_every_channel_automatic_split(eng, B, C, Lh, plan):
    P = -(-Lh // B)
    nb = P + 3
    h = synth.decaying_ir(9400 + B, Lh)
    x = _noise_many(C, nb, B, 9401 + B, _gains(C, 13 + B))
    with eng.Engine(B, P, C, 1) as e:
        e.set_ir(0, h)
        assert e.mac_plan() == plan
        y, launches = _run(e, x, 6, 64)
    assert launches == nb
    _judge("M=%d auto plan %s B=%d C=%d P=%d" % (_half(B), plan, B, C, P), y, x, [h], 0, B, nb)


_FEW_B = [7, 24, 64, 97]          # one block size per small M


def _forced(B):
    """(split, cluster, C, P) forced plans: split = rows per tile with the largest cluster the engine allows (16, or 8 at
    M = 16 where a tile of one row has 8 float4 per rank), a 16-CTA cluster, and a slot split with 8 ranges over 5 partitions"""
    R = _rows(B)
    return [(R, 16, 3, 6), (1, 16, 5, 40), (4, 2, R // 4 + 1, 5)]


@pytest.mark.gpu
@pytest.mark.parametrize("per_row", [False, True])
@pytest.mark.parametrize("plan_i", [0, 1, 2])
@pytest.mark.parametrize("B", _FEW_B)
def test_every_channel_forced_split(eng, B, plan_i, per_row):
    """Forced plans, a shared IR or per-row IRs (3 IRs of P, P/2 + 1 and 1 partitions at gains 1, 1e-2, 30); one block
    per call (graph replays), then multi-block calls."""
    R = _rows(B)
    split, cluster, C, P = _forced(B)[plan_i]
    nb = P + 5
    if per_row:
        irs = [synth.decaying_ir(9500 + B, P * B - 2), synth.decaying_ir(9501 + B, (P // 2) * B + 1, 1) * np.float32(1e-2),
               synth.decaying_ir(9502 + B, max(1, B - 1), 2) * np.float32(30.0)]
        bind = np.arange(C) % 3
    else:
        irs = [synth.decaying_ir(9500 + B, P * B - 2)]
        bind = np.zeros(C, np.int64)
    x = _noise_many(C, nb, B, 9503 + B, _gains(C, 17 + B + plan_i))
    with eng.Engine(B, P, C, len(irs)) as e:
        for j, h in enumerate(irs):
            e.set_ir(j, h)
        _bind_runs(e, bind)
        e.set_mac_split(split, cluster)
        want_plan = (True, split, min(cluster, 16, 1024 // split))
        assert e.mac_plan() == want_plan
        assert (split * want_plan[2] > P) == (plan_i != 1)             # more ranges than partitions, or 40 over 16 ranges
        y, launches = _run(e, x, 5, 4)
    assert launches == nb                                               # the cluster kernel transforms the new blocks itself
    _judge("M=%d forced plan %s %s B=%d C=%d P=%d" % (_half(B), want_plan, "per-row IRs" if per_row else "shared IR", B, C, P),
           y, x, irs, bind, B, nb)


# ---- 5. long IRs -------------------------------------------------------------------------------------------------------------
# The float32 oracle sits 0.6 - 3.3e-6 from float64 at these shapes (per channel), so the limit stays 1e-5.
_LONG = [(1, 4000, (True, 128, 4)), (16, 3000, (True, 128, 4)), (64, 1500, (True, 32, 8)), (128, 750, (True, 16, 8))]


@pytest.mark.gpu
@pytest.mark.parametrize("B,P,plan", _LONG)
def test_every_channel_long_ir(eng, B, P, plan):
    """Three channels at levels 1e-4, 1 and 1e2, P partitions (the last one full but for 3 taps), P + 3 blocks."""
    C, nb = 3, P + 3
    h = synth.decaying_ir(9600 + B, P * B - min(3, B - 1))
    x = _noise_many(C, nb, B, 9601 + B, np.array([1e-4, 1.0, 1e2], np.float32))
    with eng.Engine(B, P, C, 1) as e:
        e.set_ir(0, h)
        assert e.partitions(0) == P
        assert e.mac_plan() == plan
        y, launches = _run(e, x, 4, 512)
    assert launches == nb
    _judge("M=%d long IR B=%d P=%d plan %s" % (_half(B), B, P, plan), y, x, [h], 0, B, nb)


# ---- 6. edges ----------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["shared", "per-row", "split"])
@pytest.mark.parametrize("B", [3, 32, 64, 128])
def test_no_ir_loaded_gives_exact_zeros(eng, B, kind):
    """No set_ir at all: every IR has 0 partitions; every kernel form finishes its steps and writes exact zeros."""
    R, ring, nb = _rows(B), 4, 7
    C = {"shared": 75 * R + 1, "per-row": 75 * R + 1, "split": 3}[kind]
    x = _noise_many(C, nb, B, 9700 + B)
    with eng.Engine(B, ring, C, 2) as e:
        if kind == "per-row":
            _bind_runs(e, np.arange(C) % 2)
        if kind == "split":
            e.set_mac_split(R, 16)
        plan = {"shared": (False, 1, 1), "per-row": (True, 1, 1), "split": (True, R, min(16, 1024 // R))}[kind]
        assert e.mac_plan() == plan
        y, launches = _run(e, x, 3, 2)
    assert launches == (2 if kind == "per-row" else 1) * nb
    assert y.shape == x.shape and np.all(y == 0.0), (kind, np.abs(y).max())


@pytest.mark.gpu
@pytest.mark.parametrize("B,per_row", [(129, False), (129, True), (257, False), (257, True), (513, False), (513, True), (1025, False)])
def test_every_channel_persistent_step_boundary_blocks(eng, B, per_row):
    """The smallest block size of each persistent FFT size (M = 256 .. 2048): half of each transform is padding.  More
    units than the 296 resident CTAs.  Per-row IRs need a tile of several rows: not at B = 1025 (one row per tile)."""
    R = _rows(B)
    ring = 5
    C = 300 * R + R // 2 + 1
    nb = ring + 4
    if per_row:
        irs = _per_row_irs(B, ring, 8, 9800)
        bind = _mixed_bind(C, len(irs))
    else:
        irs = [synth.decaying_ir(9800, ring * B - 7)]
        bind = np.zeros(C, np.int64)
    x = _noise_many(C, nb, B, 9801 + B, _gains(C, 19 + B))
    with eng.Engine(B, ring, C, len(irs)) as e:
        assert e.fft_size == 2 * _half(B) and _half(B) >= 256 and _half(B - 1) == _half(B) // 2
        for j, h in enumerate(irs):
            e.set_ir(j, h)
        _bind_runs(e, bind)
        assert e.mac_plan() == (per_row, 1, 1)
        y, launches = _run(e, x, 2, 4)
    assert launches == nb                                               # k_mac_p: one launch per step, shared or per-row
    _judge("M=%d persistent %s B=%d C=%d" % (_half(B), "per-row IRs" if per_row else "shared IR", B, C), y, x, irs, bind, B, nb)


def _mats(ins, G, mixed):
    if ins == 1:
        return [[(g * 3) % 4, (g * 5 + 1 + g // 7) % 4] for g in range(G)] if mixed else [[0, 1]] * G
    return [[(g + k) % 6 for k in range(4)] for g in range(G)] if mixed else [[0, 1, 2, 3]] * G


@pytest.mark.gpu
@pytest.mark.parametrize("ins,mixed", [(1, False), (1, True), (2, False), (2, True)])
def test_every_channel_matrix_engine_smallest_block(eng, ins, mixed):
    """MatrixEngine at B = 129 (M = 256, its smallest FFT size): mono -> stereo and true stereo, shared and mixed matrices."""
    B, P, nb = 129, 5, 9
    G = 4 * 296 + 4 * 37 + 3 if ins == 1 else 2 * 296 + 77
    irs = _irs(B, P, 6, 9900)
    mats = _mats(ins, G, mixed)
    x = _noise_many(ins * G, nb, B, 9901 + ins, _gains(ins * G, 23 + ins))
    with eng.MatrixEngine(B, P, G, ins, 2, len(irs)) as m:
        for j, h in enumerate(irs):
            m.set_ir(j, h)
        for g in range(G):
            if list(mats[g]) != list(range(ins * 2)):
                m.bind_matrix(g, g + 1, mats[g])
        assert m.mac_plan() == (mixed, 1, 1)
        l0 = m.launches
        y = m.process(x)
        assert m.launches - l0 == nb
    _judge_matrix("M=256 matrix (%d, 2) B=%d G=%d mixed=%d" % (ins, B, G, mixed), y, x, irs, mats, ins, B, nb)


@pytest.mark.gpu
@pytest.mark.parametrize("private", [False, True])
def test_every_channel_group_block_64(eng, private):
    """Group at B = 64 over every device: two shared IRs bound by tile-aligned ranges, or one private IR per channel.
    (A group has no mac_plan(): each device's engine plans its own channel range.)"""
    B, P, nb = 64, 6, 10
    R = _rows(B)
    C = 300 if private else 80 * R + 5
    x = _noise_many(C, nb, B, 9950 + private, _gains(C, 29 + private))
    if private:
        irs = [synth.decaying_ir(9960 + c, (1 + c % P) * B - 1 - c % 13, c) for c in range(C)]
        bind = np.arange(C)
    else:
        irs = [synth.decaying_ir(9960, P * B - 3), synth.decaying_ir(9961, 2 * B + 1, 1)]
        bind = np.zeros(C, np.int64)
        bind[3 * R:13 * R] = 1
    devices = list(range(max(1, eng.device_count())))
    with eng.Group(devices, B, P, C, 0 if private else 2) as g:
        for j, h in enumerate(irs):
            g.set_ir(j, h)
        if not private:
            g.bind(3 * R, 13 * R, 1)
        y = g.process(x)
    _judge("M=64 group of %d devices, %s IRs" % (len(devices), "private" if private else "shared"), y, x, irs, bind, B, nb)
