"""Every output channel against float64, stream isolation under NaN / Inf input, and offsets past 2^32 FDL elements.

* ref64: a float64 FFT convolution of every channel with its own IR (or, for the IR-matrix engine, the sum of its terms),
  checked on the CPU against scipy and the C oracle; the GPU tests trust it because of that test.
* Every block-step form (k_mac_p shared and per-row IRs, the two-launch form, the fused cluster step, k_mac_mx, the
  multi-device group) against ref64 on EVERY channel, each channel at its own input level (log-uniform 1e-4 .. 1e2) and
  judged at its own scale: max-abs over the channel's own peak, L2 over its own norm.
* One stream's NaN or Inf changes no other stream's output, bit for bit; the poisoned stream is back, bit for bit, once the
  bad block has left its delay line: P + 1 blocks after it, P the partition count of its own IR.
* The plain and the matrix engine with more than 2^32 float2 of delay line, every channel checked on the device.
* irb_deconvolve_batch_device with captures or results at an odd float offset (4-byte, not 8-byte aligned).
"""
import numpy as np
import pytest

from conftest import TOL, parity
from irbaboon_b200 import synth
from irbaboon_b200.engine import next_pow2


# ---- float64 reference -----------------------------------------------------------------------------------------
def ref64(x, irs, bind, B, nb):
    """x: planar [C][n] (n <= nb*B; missing samples are zero), irs: list of IRs, bind: IR index per channel (or one for all).
    -> float64 [C][nb*B], the first nb*B samples of each channel's linear convolution with its IR."""
    x = np.asarray(x)
    C, n = x.shape[0], nb * B
    bind = np.broadcast_to(np.asarray(bind, np.int64), (C,))
    out = np.zeros((C, n))
    for j in np.unique(bind):
        h = np.asarray(irs[j], np.float64)
        L = next_pow2(n + len(h))
        H = np.fft.rfft(h, L)
        rows = np.flatnonzero(bind == j)
        step = max(1, (1 << 22) // L)                                   # about 64 MB of spectra per chunk
        for r0 in range(0, len(rows), step):
            r = rows[r0:r0 + step]
            out[r] = np.fft.irfft(np.fft.rfft(x[r, :n].astype(np.float64), L, axis=1) * H, L, axis=1)[:, :n]
    return out


def ref64_matrix(x, irs, mats, ins, outs, B, nb):
    """IR-matrix engine: out[g*outs + o] = sum_i x[g*ins + i] * h[mats[g][i*outs + o]]  (x planar [G*ins][n])."""
    G = x.shape[0] // ins
    mats = np.broadcast_to(np.asarray(mats, np.int64).reshape(-1, ins * outs), (G, ins * outs))
    out = np.zeros((G * outs, nb * B))
    for i in range(ins):
        for o in range(outs):
            out[o::outs] += ref64(x[i::ins], irs, mats[:, i * outs + o], B, nb)
    return out


def _planar(blocks):
    """[nb][C][B] -> [C][nb*B]"""
    nb, C, B = blocks.shape
    return np.ascontiguousarray(blocks.transpose(1, 0, 2)).reshape(C, nb * B)


def _gains(C, seed):
    """one input level per channel, log-uniform over 1e-4 .. 1e2"""
    return (10.0 ** np.random.default_rng(seed).uniform(-4.0, 2.0, C)).astype(np.float32)


def _noise(C, nb, B, seed, gains=None):
    """[nb][C][B] float32: synth white noise, stream c for channel c, times the channel's gain"""
    x = np.stack([synth.white_noise(seed, c, nb * B) for c in range(C)])
    if gains is not None:
        x *= gains[:, None]
    return np.ascontiguousarray(x.reshape(C, nb, B).transpose(1, 0, 2))


def _per_channel(got, want):
    """per channel: (max-abs error / the channel's own peak, L2 error / the channel's own norm)"""
    d = np.asarray(got, np.float64) - want
    peak = np.abs(want).max(axis=1)
    norm = np.sqrt((want * want).sum(axis=1))
    assert (peak > 0).all()
    return np.abs(d).max(axis=1) / peak, np.sqrt((d * d).sum(axis=1)) / norm


def _every_channel(name, got, want):
    """got [C][n] float32 against want [C][n] float64: both errors <= TOL on every channel; prints the worst."""
    e, l2 = _per_channel(got, want)
    ok = (e <= TOL) & (l2 <= TOL)                                       # NaN fails
    print("%s: %d channels, worst max-abs/own peak %.3g (channel %d), worst L2/own norm %.3g (channel %d)"
          % (name, len(e), np.nanmax(e), int(np.nanargmax(e)), np.nanmax(l2), int(np.nanargmax(l2))))
    bad = np.flatnonzero(~ok)
    assert bad.size == 0, (name, bad[:10], e[bad[:10]], l2[bad[:10]])


def _irs(B, P, n, seed):
    """n IRs of different partition counts P, P-1, ... (never below 1), none a whole number of blocks"""
    return [synth.decaying_ir(seed + j, max(1, (P - j % max(P, 1)) * B - 5 * j - 3), j) for j in range(n)]


def _devices(eng):
    return list(range(max(1, eng.device_count())))


# ---- 0. the reference itself, on the CPU -------------------------------------------------------------------------
@pytest.mark.parametrize("B,nb,lens", [(256, 7, [1, 100, 255, 256, 257, 1501]), (300, 5, [7, 299, 301, 1203]), (129, 9, [1, 50, 128, 1001])])
def test_ref64_matches_scipy_and_the_oracle(orc, B, nb, lens):
    """Odd lengths, block sizes that are not powers of two, IRs shorter than one block, an input that ends inside a block,
    channels at levels six decades apart."""
    from scipy.signal import fftconvolve

    C = 2 * len(lens) + 1
    irs = [synth.decaying_ir(500 + j, n, j) for j, n in enumerate(lens)]
    bind = (np.arange(C) * 3) % len(irs)
    n = nb * B - 37
    x = np.stack([synth.white_noise(600, c, n) for c in range(C)]) * _gains(C, 1)[:, None]
    got = ref64(x, irs, bind, B, nb)
    assert got.shape == (C, nb * B)
    for c in range(C):
        h = irs[bind[c]]
        want = np.zeros(nb * B)
        full = fftconvolve(x[c].astype(np.float64), h.astype(np.float64))[:nb * B]
        want[:len(full)] = full
        assert np.abs(got[c] - want).max() <= 1e-12 * np.abs(want).max(), c
        off = np.zeros(nb * B)
        o = orc.convolve_periodic(x[c], h, B)[0, :nb * B]
        off[:len(o)] = o
        e, l2 = _per_channel(off[None, :], got[c:c + 1])
        assert e[0] <= TOL and l2[0] <= TOL, (c, e, l2)
        assert max(parity(off, got[c])) <= TOL
    # the matrix form is the sum of its terms
    G, ins, outs = 3, 2, 2
    mats = [[(g + k) % len(irs) for k in range(4)] for g in range(G)]
    xm = x[:G * ins]
    got = ref64_matrix(xm, irs, mats, ins, outs, B, nb)
    for g in range(G):
        for o in range(outs):
            want = sum(ref64(xm[g * ins + i:g * ins + i + 1], irs, mats[g][i * outs + o], B, nb)[0] for i in range(ins))
            assert np.abs(got[g * outs + o] - want).max() <= 1e-12 * np.abs(want).max()


# ---- 1. every channel against float64 --------------------------------------------------------------------------------
# the stream counts of test_gpu_persistent.py: ragged last units, the last wave on narrowed units, fewer rows than one wave
@pytest.mark.gpu
@pytest.mark.parametrize("B,C,P,nb,fused", [
    (512, 1879, 5, 9, True),
    (512, 1879, 5, 9, False),                    # the same step in its two-launch form (k_fwd, then k_mac)
    (512, 1186, 3, 7, True),
    (512, 4 * 296 * 2 + 4 * 100 + 3, 4, 6, True),
    (256, 8 * 296 + 4 * 296 + 2 * 100 + 1, 4, 6, True),
    (1024, 2 * 296 + 150, 6, 8, True),
    (2048, 300, 3, 5, True),
    (300, 1000, 4, 6, True),
    (512, 640, 9, 12, True),
])
def test_every_channel_shared_ir(eng, B, C, P, nb, fused):
    h = synth.decaying_ir(7001, P * B - 7)
    x = _noise(C, nb, B, 7101, _gains(C, B + C))
    with eng.Engine(B, P, C, 1) as e:
        e.set_ir(0, h)
        e.set_fused_step(fused)
        assert e.mac_plan() == (False, 1, 1)
        l0 = e.launches
        y = e.process(x)
        assert e.launches - l0 == (1 if fused else 2) * nb
    _every_channel("shared IR B=%d C=%d P=%d fused=%d" % (B, C, P, fused), _planar(y), ref64(_planar(x), [h], 0, B, nb))


@pytest.mark.gpu
@pytest.mark.parametrize("B,C,ring,fused", [(1024, 2 * 296 + 151, 9, True), (512, 4 * 296 + 2 * 200 + 3, 7, True), (512, 4 * 296 + 2 * 200 + 3, 7, False)])
def test_every_channel_per_row_irs(eng, B, C, ring, fused):
    """Rows of one tile bound to IRs of 8 different lengths (1 .. ring partitions): k_mac_p PERROW, or k_fwd + k_mac_slots."""
    irs = [synth.decaying_ir(7200 + j, max(1, (1 + j * (ring - 1) // 7) * B - 3 * j), j) for j in range(8)]
    assert len(set(-(-len(h) // B) for h in irs)) >= 6
    bind = (np.arange(C) * 5 + np.arange(C) // 3) % 8
    nb = ring + 4
    x = _noise(C, nb, B, 7201, _gains(C, C))
    with eng.Engine(B, ring, C, len(irs)) as e:
        for j, h in enumerate(irs):
            e.set_ir(j, h)
        for c in range(C):
            e.bind(c, c + 1, int(bind[c]))
        e.set_fused_step(fused)
        assert e.mac_plan() == (True, 1, 1)
        y = e.process(x)
    _every_channel("per-row IRs B=%d C=%d fused=%d" % (B, C, fused), _planar(y), ref64(_planar(x), irs, bind, B, nb))


# few rows: a row's partitions split over tile slots and over the CTAs of a cluster, forward transform fused (one launch per step)
_CLUSTER = [(512, 512 * 21, 5, 2, 2), (256, 256 * 37 + 11, 3, 2, 4), (1024, 1024 * 9 + 1, 3, 2, 8), (256, 256 * 37 + 11, 2, 8, 16)]


@pytest.mark.gpu
@pytest.mark.parametrize("B,Lh,C,split,cluster", _CLUSTER)
def test_every_channel_fused_cluster_step(eng, B, Lh, C, split, cluster):
    P = -(-Lh // B)
    nb = P + 6
    h = synth.decaying_ir(7300, Lh)
    x = _noise(C, nb, B, 7301, _gains(C, cluster))
    with eng.Engine(B, P, C, 1) as e:
        e.set_ir(0, h)
        e.set_mac_split(split, cluster)
        assert e.mac_plan() == (True, split, cluster)
        l0 = e.launches
        y = np.stack([e.process(x[k]) for k in range(nb)])           # one block per call: the latency path, graph replays
        assert e.launches - l0 == nb
    _every_channel("cluster %d split %d B=%d C=%d" % (cluster, split, B, C), _planar(y), ref64(_planar(x), [h], 0, B, nb))


_MATRIX = [  # (ins, B, G, P, nb, mixed): every FFT size of k_mac_mx, partial last units, more units than resident CTAs
    (1, 256, 4 * 296 + 4 * 37 + 3, 5, 9, False), (1, 512, 777, 6, 13, True), (1, 1024, 311, 3, 8, True), (1, 700, 333, 3, 7, False),
    (2, 512, 1201, 5, 9, False), (2, 256, 150, 4, 8, True), (2, 1024, 333, 6, 9, False), (2, 700, 64, 3, 7, True),
]


def _mats(ins, G, mixed):
    if ins == 1:
        return [[(g * 3) % 4, (g * 5 + 1 + g // 7) % 4] for g in range(G)] if mixed else [[0, 1]] * G
    return [[(g + k) % 6 for k in range(4)] for g in range(G)] if mixed else [[0, 1, 2, 3]] * G


def _matrix(eng, B, P, G, ins, irs, mats):
    m = eng.MatrixEngine(B, P, G, ins, 2, len(irs))
    for j, h in enumerate(irs):
        m.set_ir(j, h)
    for g in range(G):
        if list(mats[g]) != list(range(ins * 2)):
            m.bind_matrix(g, g + 1, mats[g])
    return m


@pytest.mark.gpu
@pytest.mark.parametrize("ins,B,G,P,nb,mixed", _MATRIX)
def test_every_channel_matrix_engine(eng, ins, B, G, P, nb, mixed):
    """Mono -> stereo and true stereo; the IRs of one matrix differ in length; shared matrices and matrices that differ
    inside a unit (PERGROUP)."""
    irs = _irs(B, P, 6, 7400)
    mats = _mats(ins, G, mixed)
    x = _noise(ins * G, nb, B, 7401, _gains(ins * G, G))
    with _matrix(eng, B, P, G, ins, irs, mats) as m:
        assert m.mac_plan()[0] == (mixed and B <= 512)
        y = m.process(x)
    _every_channel("matrix (%d, 2) B=%d G=%d mixed=%d" % (ins, B, G, mixed), _planar(y), ref64_matrix(_planar(x), irs, mats, ins, 2, B, nb))


@pytest.mark.gpu
@pytest.mark.parametrize("private", [False, True])
def test_every_channel_group(eng, private):
    B, P, nb = 512, 4, 9
    C = 300 if private else 700
    x = _noise(C, nb, B, 7501, _gains(C, 3 + private))
    if private:
        irs = [synth.decaying_ir(7600 + c, (1 + c % P) * B - 1 - c % 13, c) for c in range(C)]
        bind = np.arange(C)
    else:
        irs = [synth.decaying_ir(7500, P * B - 3), synth.decaying_ir(7501, 2 * B + 1, 1)]
        bind = np.zeros(C, np.int64)
        bind[100:400] = 1
    with eng.Group(_devices(eng), B, P, C, 0 if private else 2) as g:
        for j, h in enumerate(irs):
            g.set_ir(j, h)
        if not private:
            g.bind(100, 400, 1)
        y = g.process(x)
    _every_channel("group of %d devices, %s IRs" % (len(_devices(eng)), "private" if private else "shared"), _planar(y), ref64(_planar(x), irs, bind, B, nb))


# ---- 2. NaN / Inf containment and exact recovery ------------------------------------------------------------------------
def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _poison(x, marks):
    """marks: (channel, block, value); the value goes to sample B // 3 of that block"""
    xp = x.copy()
    for c, k, v in marks:
        xp[k, c, x.shape[2] // 3] = v
    return xp


def _contained(name, clean, dirty, hit):
    """clean, dirty: [nb][C][B].  hit: {output channel: (block k of the bad sample, P)}.  Every other channel equals the
    clean run bit for bit; a hit channel equals it before block k, is non-finite at block k and equals it again from block
    k + P + 1 on (and not before).  -> {channel: blocks from the bad one to the first recovered block}"""
    nb, C = clean.shape[:2]
    others = np.setdiff1d(np.arange(C), list(hit))
    assert np.array_equal(_bits(dirty[:, others]), _bits(clean[:, others])), name
    rec = {}
    for c, (k, P) in hit.items():
        assert k + P + 1 < nb, "too few blocks to see the recovery"
        assert np.array_equal(_bits(dirty[:k, c]), _bits(clean[:k, c])), (name, c)
        assert not np.isfinite(dirty[k, c]).all(), (name, c, k)
        diff = [b for b in range(nb) if not np.array_equal(_bits(dirty[b, c]), _bits(clean[b, c]))]
        first = diff[-1] + 1
        rec[c] = first - k
        assert first == k + P + 1, (name, c, k, P, first)
    print("%s: recovery %s (blocks after the bad one, per poisoned channel)" % (name, rec))
    return rec


def _three_runs(run, x, nan_marks, inf_marks):
    clean = run(x)
    assert np.isfinite(clean).all()
    return clean, run(_poison(x, nan_marks)), run(_poison(x, inf_marks))


@pytest.mark.gpu
@pytest.mark.parametrize("per_row,fused", [(False, True), (False, False), (True, True), (True, False)])
def test_nan_inf_stay_in_their_stream(eng, per_row, fused):
    """k_mac_p shared / per-row IRs, and their two-launch forms k_mac / k_mac_slots.  The shared IR is one partition
    shorter than the ring, so a kernel that multiplied ring slots past the IR by zero spectra would keep the NaN longer."""
    B, ring, C, nb = 512, 5, 300, 14
    if per_row:
        irs = [synth.decaying_ir(7700 + j, (j + 1) * B - 9, j) for j in range(ring)]
        bind = (np.arange(C) * 5 + np.arange(C) // 3) % ring
    else:
        irs = [synth.decaying_ir(7700, (ring - 1) * B - 9)]
        bind = np.zeros(C, np.int64)
    x = _noise(C, nb, B, 7701)
    with eng.Engine(B, ring, C, len(irs)) as e:
        for j, h in enumerate(irs):
            e.set_ir(j, h)
        if per_row:
            for c in range(C):
                e.bind(c, c + 1, int(bind[c]))
        e.set_fused_step(fused)
        assert e.mac_plan()[0] == per_row
        R = e.tile_channels
        a, b, c = 5 * R + R // 2, 9 * R + R // 2, 13 * R + (R - 1) // 2          # inside a tile: its mates are checked
        P = [e.partitions(int(bind[ch])) for ch in (a, b, c)]

        def run(xx):
            e.reset()
            return e.process(xx)

        clean, d1, d2 = _three_runs(run, x, [(a, 2, np.nan)], [(b, 3, np.inf), (c, 5, -np.inf)])
    name = "k_mac_p %s fused=%d" % ("per-row" if per_row else "shared", fused)
    _contained(name + " NaN", clean, d1, {a: (2, P[0])})
    _contained(name + " +-Inf", clean, d2, {b: (3, P[1]), c: (5, P[2])})


@pytest.mark.gpu
@pytest.mark.parametrize("B,Lh,C,split,cluster", [(512, 512 * 6 + 3, 5, 2, 2), (1024, 1024 * 5 + 1, 3, 2, 8)])
def test_nan_inf_stay_in_their_stream_cluster_step(eng, B, Lh, C, split, cluster):
    P = -(-Lh // B)
    nb = P + 8
    h = synth.decaying_ir(7800, Lh)
    x = _noise(C, nb, B, 7801)
    with eng.Engine(B, P, C, 1) as e:
        e.set_ir(0, h)
        e.set_mac_split(split, cluster)
        assert e.mac_plan() == (True, split, cluster)

        def run(xx):
            e.reset()
            return np.stack([e.process(xx[k]) for k in range(nb)])

        mid = C // 2
        clean, d1, d2 = _three_runs(run, x, [(mid, 2, np.nan)], [(0, 3, np.inf), (C - 1, 5, -np.inf)])
    name = "cluster %d split %d" % (cluster, split)
    _contained(name + " NaN", clean, d1, {mid: (2, P)})
    _contained(name + " +-Inf", clean, d2, {0: (3, P), C - 1: (5, P)})


@pytest.mark.gpu
@pytest.mark.parametrize("ins,B,mixed", [(1, 256, True), (1, 512, False), (2, 256, True), (2, 1024, False)])
def test_nan_inf_stay_in_their_group_matrix_engine(eng, ins, B, mixed):
    """A bad sample on input i of group g reaches only the outputs of g; output o is back P(mats[g][i*outs + o]) + 1 blocks
    later; every other group is bit-identical to the clean run."""
    G, P, nb = 240, 5, 14
    irs = _irs(B, P, 6, 7900)
    mats = _mats(ins, G, mixed)
    x = _noise(ins * G, nb, B, 7901)
    with _matrix(eng, B, P, G, ins, irs, mats) as m:
        parts = [m.partitions(j) for j in range(len(irs))]

        def run(xx):
            m.reset()
            return m.process(xx)

        # (group, input, block, value): groups inside a unit of 4 (B = 256) or 2 (B = 512) groups
        marks1 = [(21, ins - 1, 2, np.nan)]
        marks2 = [(37, 0, 3, np.inf), (54, ins - 1, 5, -np.inf)]
        clean, d1, d2 = _three_runs(run, x, [(g * ins + i, k, v) for g, i, k, v in marks1], [(g * ins + i, k, v) for g, i, k, v in marks2])

    def hit(marks):
        return {g * 2 + o: (k, parts[mats[g][i * 2 + o]]) for g, i, k, _ in marks for o in range(2)}

    name = "matrix (%d, 2) B=%d mixed=%d" % (ins, B, mixed)
    _contained(name + " NaN", clean, d1, hit(marks1))
    _contained(name + " +-Inf", clean, d2, hit(marks2))


@pytest.mark.gpu
@pytest.mark.parametrize("private", [False, True])
def test_nan_inf_stay_in_their_stream_group(eng, private):
    B, P, C, nb = 256, 4, 200, 12
    if private:
        irs = [synth.decaying_ir(8000 + c, max(1, (1 + c % P) * B - 7), c) for c in range(C)]
    else:
        irs = [synth.decaying_ir(8000, P * B - 7)]
    x = _noise(C, nb, B, 8001)
    with eng.Group(_devices(eng), B, P, C, 0 if private else 1) as g:
        for j, h in enumerate(irs):
            g.set_ir(j, h)

        def run(xx):
            g.reset()
            return g.process(xx)

        a, b, c = 41, 90, 133
        clean, d1, d2 = _three_runs(run, x, [(a, 2, np.nan)], [(b, 3, np.inf), (c, 4, -np.inf)])
    Pc = [-(-len(irs[ch if private else 0]) // B) for ch in (a, b, c)]
    name = "group %s IRs" % ("private" if private else "shared")
    _contained(name + " NaN", clean, d1, {a: (2, Pc[0])})
    _contained(name + " +-Inf", clean, d2, {b: (3, Pc[1]), c: (4, Pc[2])})


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["tiles", "rows", "matrix"])
def test_nan_tap_in_one_ir_and_clean_reload(eng, kind):
    """A NaN tap in IR 1 (set_ir) reaches only what is bound to IR 1: shared-IR tiles (IR replicas), rows of one tile bound to
    different IRs (per-row staging), or matrix groups (per-group staging).  After set_ir(1, clean) the affected outputs equal
    the clean run again from the second block on (the first still adds the poisoned overlap)."""
    B, P, nb, m = 256, 4, 10, 4
    irs = _irs(B, P, 4, 8100)                                           # (a true-stereo matrix engine holds at least 4)
    bad = irs[1].copy()
    bad[B + 17] = np.nan                                                # in partition 1
    if kind == "matrix":
        G = 150
        mats = [[(g + k) % 3 for k in range(4)] if g % 5 else [0, 2, 2, 0] for g in range(G)]
        x = _noise(2 * G, nb, B, 8101)
        e = _matrix(eng, B, P, G, 2, irs, mats)
        hit = [g * 2 + o for g in range(G) for o in range(2) if 1 in (mats[g][o], mats[g][2 + o])]
    else:
        C = 600
        x = _noise(C, nb, B, 8101)
        e = eng.Engine(B, P, C, len(irs))
        for j, h in enumerate(irs):
            e.set_ir(j, h)
        R = e.tile_channels
        bind = (np.arange(C) // R) % 3 if kind == "tiles" else (np.arange(C) * 5 + np.arange(C) // 3) % 3
        for c in range(C):
            e.bind(c, c + 1, int(bind[c]))
        assert e.mac_plan()[0] == (kind == "rows")
        hit = list(np.flatnonzero(bind == 1))
    with e:
        clean = e.process(x)
        e.reset()
        e.set_ir(1, bad)
        y0 = e.process(x[:m])
        e.set_ir(1, irs[1])
        dirty = np.concatenate([y0, e.process(x[m:])])
    others = np.setdiff1d(np.arange(clean.shape[1]), hit)
    assert len(hit) and len(others)
    assert np.array_equal(_bits(dirty[:, others]), _bits(clean[:, others]))
    for b in range(m + 1):
        assert not np.isfinite(dirty[b, hit]).all(axis=-1).any(), b            # every affected output, every block up to m
    assert np.array_equal(_bits(dirty[m + 1:, hit]), _bits(clean[m + 1:, hit]))
    print("NaN tap, %s: %d outputs affected, back to the clean run at block %d (IR reloaded before block %d)" % (kind, len(hit), m + 1, m))


@pytest.mark.gpu
@pytest.mark.parametrize("smoothing", [False, True])
def test_nan_capture_stays_in_its_deconvolution(eng, smoothing):
    """A batch of 6 captures, one with a NaN: the other 5 results equal the clean batch bit for bit, from host memory and
    from device memory (plain: the unstaged device path; smoothed: the staged one)."""
    import torch

    n, batch, bad = 1 << 14, 6, 2
    sweep = synth.exp_sine_sweep(n / 48000.0, 48000.0, 20.0, 20000.0).astype(np.float32)[:n]
    caps = np.stack([synth.white_noise(8200, j, n) for j in range(batch)])
    dirty = caps.copy()
    dirty[bad, n // 3] = np.nan
    others = [j for j in range(batch) if j != bad]
    host = [eng.deconvolve_batch(c, sweep, 48000.0, smoothing) for c in (caps, dirty)]
    dev = []
    for c in (caps, dirty):
        d_in = torch.from_numpy(c).cuda()
        d_out = torch.zeros((batch, n), dtype=torch.float32, device="cuda")
        torch.cuda.synchronize()
        eng.deconvolve_batch_device(d_in.data_ptr(), batch, n, sweep, d_out.data_ptr(), 48000.0, smoothing)
        torch.cuda.synchronize()
        dev.append(d_out.cpu().numpy())
    for clean, poisoned in (host, dev):
        assert np.isfinite(clean).all()
        assert np.array_equal(_bits(poisoned[others]), _bits(clean[others]))
        assert not np.isfinite(poisoned[bad]).all()
    assert np.array_equal(dev[0], host[0])


@pytest.mark.gpu
def test_nan_in_one_channel_of_stereo_convolve_periodic(eng):
    B, n, Lh = 256, 5000, 1501
    x = np.stack([synth.white_noise(8300, c, n) for c in range(2)])
    h = np.stack([synth.decaying_ir(8301 + c, Lh, c) for c in range(2)])
    clean = eng.convolve_periodic(x, h, B)
    x[0, 1234] = np.nan
    dirty = eng.convolve_periodic(x, h, B)
    assert np.isfinite(clean).all() and not np.isfinite(dirty[0]).all()
    assert np.array_equal(_bits(dirty[1]), _bits(clean[1]))


# ---- 3. offsets past 2^32 FDL elements, every channel ---------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("ins,outs,groups", [(1, 1, 56000), (1, 2, 56000), (2, 2, 28000)])
def test_fdl_past_two_to_the_32_every_channel(eng, ins, outs, groups):
    """56 000 delay lines of 160 slots at B = 512: 4.6e9 float2 (36.7 GB) of FDL, so row and slot offsets pass 2^32
    elements.  Every input gets one impulse in block 0 at its own offset with its own gain; for ring + 4 blocks, one block per
    process_device call, every output block of every channel is compared on the device with the shifted, scaled IR (the sum
    of two for true stereo).  A wrapped or truncated offset would return another row's delay and gain."""
    import torch

    B, ring = 512, 160
    rows, n_out = groups * ins, groups * outs
    est = rows * ring * B * 8                                           # FDL bytes: rows x ring slots x B packed complex bins
    assert est > (1 << 32) * 8
    free, total = torch.cuda.mem_get_info()
    print("free device memory %.1f GB of %.1f GB; FDL %.1f GB" % (free / 1e9, total / 1e9, est / 1e9))
    if free < 1.25 * est:
        pytest.skip("needs %.1f GB free on the device for a %.1f GB delay line; %.1f GB free" % (1.25 * est / 1e9, est / 1e9, free / 1e9))
    irs = [synth.decaying_ir(8400 + j, ring * B - 1000 * j - 7, j) for j in range(ins * outs)]
    rng = np.random.default_rng(8400 + rows + outs)
    gain = (0.5 + rng.random(rows)).astype(np.float32)
    delay = rng.integers(0, B, rows)
    nb = ring + 4
    Lp = (nb + 2) * B
    hp = np.zeros((len(irs), Lp), np.float32)                           # IR j at offset B of row j: index b*B + t - d + B >= 0
    for j, h in enumerate(irs):
        hp[j, B:B + len(h)] = h
    dev = torch.device("cuda")
    d_hp = torch.from_numpy(hp).to(dev).reshape(-1)
    d_gain = torch.from_numpy(gain).to(dev)
    d_delay = torch.from_numpy(delay).to(dev)
    t = torch.arange(B, device=dev)
    e = eng.Engine(B, ring, rows, 1) if outs == 1 else eng.MatrixEngine(B, ring, groups, ins, outs)
    with e:
        for j, h in enumerate(irs):
            e.set_ir(j, h)
        assert e.state_bytes >= est
        d_in = torch.zeros((rows, B), dtype=torch.float32, device=dev)
        d_in[torch.arange(rows, device=dev), d_delay] = d_gain
        d_out = torch.empty((n_out, B), dtype=torch.float32, device=dev)
        torch.cuda.synchronize()
        worst = 0.0
        for b in range(nb):
            e.process_device(d_in.data_ptr(), d_out.data_ptr(), 1)
            e.synchronize()
            if b == 0:
                d_in.zero_()
            want = torch.zeros((n_out, B), dtype=torch.float32, device=dev)
            for i in range(ins):
                r = torch.arange(i, rows, ins, device=dev)                  # input i of every group
                idx = b * B + t[None, :] - d_delay[r][:, None] + B
                for o in range(outs):
                    want[o::outs] += d_gain[r][:, None] * d_hp[(i * outs + o) * Lp + idx]
            err = (d_out - want).abs()
            tol = 2e-6 * want.abs().amax(dim=1, keepdim=True).clamp(min=1.0)
            bad = ~(err <= tol)
            if bool(bad.any()):
                ch = int(bad.any(dim=1).nonzero()[0])
                pytest.fail("block %d: %d outputs wrong, first %d (error %.3g)" % (b, int(bad.any(dim=1).sum()), ch, float(err[ch].max())))
            worst = max(worst, float(err.max()))
            torch.cuda.synchronize()
    print("(%d, %d) x %d groups, %d blocks: every output within 2e-6; worst absolute error %.3g" % (ins, outs, groups, nb, worst))


# ---- 4. device pointers at an odd float offset ----------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("odd_nums,odd_out", [(True, False), (False, True), (True, True)])
def test_deconvolve_batch_device_accepts_4_byte_aligned_pointers(eng, odd_nums, odd_out):
    """A torch view one float into a larger buffer is 4-byte but not 8-byte aligned.  The shape would take the unstaged
    device path (N = 2^16, plain division, phase kept, even length), whose column passes move float2; such pointers take the
    staged path instead, and give the host entry's bits.  The floats around the result stay untouched."""
    import torch

    n, batch = 1 << 16, 7
    rng = np.random.default_rng(8500)
    sweep = synth.exp_sine_sweep(n / 48000.0, 48000.0, 20.0, 20000.0).astype(np.float32)[:n]
    caps = (rng.random((batch, n), dtype=np.float32) * 2 - 1).astype(np.float32)
    want = eng.deconvolve_batch(caps, sweep, 48000.0, False, True, True)
    a, c = int(odd_nums), int(odd_out)
    d_caps = torch.zeros(batch * n + 2, dtype=torch.float32, device="cuda")
    d_caps[a:a + batch * n] = torch.from_numpy(caps.reshape(-1)).cuda()
    d_out = torch.full((batch * n + 2,), 7.0, dtype=torch.float32, device="cuda")
    nums_v, out_v = d_caps[a:a + batch * n], d_out[c:c + batch * n]
    assert (nums_v.data_ptr() % 8 != 0) == odd_nums and (out_v.data_ptr() % 8 != 0) == odd_out
    torch.cuda.synchronize()
    eng.deconvolve_batch_device(nums_v.data_ptr(), batch, n, sweep, out_v.data_ptr(), 48000.0, False, True, True)
    torch.cuda.synchronize()
    assert np.array_equal(out_v.cpu().numpy().reshape(batch, n), want)
    rest = torch.cat([d_out[:c], d_out[c + batch * n:]]).cpu().numpy()
    assert np.all(rest == 7.0)
