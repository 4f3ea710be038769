"""GPU: the IR-matrix engine (irb_engine_create_matrix, kernel k_mac_mx in irb_mac_mx.cuh).

Mono -> stereo (1, 2) is checked bit for bit against a plain Engine fed the duplicated inputs and bound to the same IRs (same
FDL spectra, same fmaf sequence per output); true stereo (2, 2) against a float64 reference, the sum of plain-engine outputs and
the offline convolution."""
import ctypes

import numpy as np
import pytest

from conftest import TOL, parity
from irbaboon_b200 import synth

pytestmark = pytest.mark.gpu


def _blocks(C, nb, B, seed):
    rng = np.random.default_rng(seed)
    return (rng.random((nb, C, B), dtype=np.float32) * 2 - 1).astype(np.float32)


def _irs(B, P, n, seed):
    """n IRs of different partition counts (P, P-1, ... never below 1)."""
    return [synth.decaying_ir(seed + j, max(1, (P - j % max(P, 1)) * B - 5 * j - 3), j) for j in range(n)]


def _plain_dup12(eng, B, P, x, irs, mats, stage=None):
    """plain engine on 2G channels: channel 2g+o gets input g and IR mats[g][o]"""
    nb, G, _ = x.shape
    with eng.Engine(B, P, 2 * G, len(irs)) as p:
        p.set_mac_split(1, 1)                     # one kernel tile per unit, no partition split: the summation order of k_mac_mx
        for j, h in enumerate(irs):
            p.set_ir(j, h)
        for g in range(G):
            for o in range(2):
                p.bind(2 * g + o, 2 * g + o + 1, mats[g][o])
        xd = np.ascontiguousarray(np.repeat(x, 2, axis=1))
        if stage is None:
            return p.process(xd)
        k, ir_id, taps = stage
        y0 = p.process(xd[:k])
        p.stage_ir(ir_id, taps)
        return np.concatenate([y0, p.process(xd[k:])])


def _pergroup(B, mixed):
    """mixed matrices need the per-group staging only where a unit holds several groups (FFT half size below 1024)"""
    return mixed and B <= 512


def _matrix(eng, B, P, G, ins, outs, irs, mats):
    m = eng.MatrixEngine(B, P, G, ins, outs, len(irs))
    for j, h in enumerate(irs):
        m.set_ir(j, h)
    for g in range(G):
        if mats[g] != list(range(ins * outs)):
            m.bind_matrix(g, g + 1, mats[g])
    return m


# (B, groups, P, blocks, mixed): every FFT size of the kernel, a partial last unit, more units than the 296 resident CTAs,
# more blocks than the ring holds, shared matrices and matrices that differ inside a unit (PERGROUP)
@pytest.mark.parametrize("B,G,P,nb,mixed", [
    (256, 4 * 296 + 4 * 37 + 3, 5, 9, False),      # 4 groups per unit, last unit partial, > 296 units
    (256, 303, 4, 7, True),
    (512, 2 * 296 * 2 + 1, 4, 9, False),           # 2 groups per unit, last unit partial, two and a bit waves
    (512, 777, 6, 13, True),
    (300, 333, 3, 7, False),                       # block size that is not a power of two (M = 512)
    (1024, 700, 6, 10, False),                     # 1 group per unit
    (1024, 311, 3, 8, True),
    (512, 5, 3, 6, False),                         # fewer units than CTAs
])
def test_mono_to_stereo_is_bit_identical_to_duplicated_plain_engine(eng, B, G, P, nb, mixed):
    irs = _irs(B, P, 4, 3100)                      # IR 0 has P partitions, IR 1 P-1, ...: the two IRs of a matrix differ in length
    mats = [[(g * 3) % 4, (g * 5 + 1 + g // 7) % 4] for g in range(G)] if mixed else [[0, 1]] * G
    x = _blocks(G, nb, B, 41 + G)
    with _matrix(eng, B, P, G, 1, 2, irs, mats) as m:
        assert m.mac_plan() == (_pergroup(B, mixed), 1, 1)
        l0 = m.launches
        y = m.process(x)
        assert m.launches - l0 == nb                                     # one launch per block step
    want = _plain_dup12(eng, B, P, x, irs, mats)
    assert y.shape == (nb, 2 * G, B)
    assert np.array_equal(y, want)


def test_mono_to_stereo_many_laps_full_gpu(eng):
    """Tens of thousands of output channels, the ring lapped several times: the race of an early stage release would show here."""
    B, G, P, nb = 512, 6000, 11, 40
    irs = _irs(B, P, 2, 3200)
    x = _blocks(G, nb, B, 5)
    with _matrix(eng, B, P, G, 1, 2, irs, [[0, 1]] * G) as m:
        y = m.process(x)
    assert np.array_equal(y, _plain_dup12(eng, B, P, x, irs, [[0, 1]] * G))


def _ref22(x, irs, mat, nb, B):
    """float64: out_o = sum_i fftconvolve(in_i, h[mat[i*2+o]]) cut to the streamed blocks"""
    from scipy.signal import fftconvolve

    out = np.zeros((2, nb * B))
    for o in range(2):
        for i in range(2):
            out[o] += fftconvolve(x[i].astype(np.float64), irs[mat[i * 2 + o]].astype(np.float64))[:nb * B]
    return out


@pytest.mark.parametrize("B,G,P,nb,mixed", [(512, 1201, 5, 9, False), (256, 150, 4, 8, True), (1024, 333, 6, 9, False), (700, 64, 3, 7, True)])
def test_true_stereo_matches_float64_plain_sum_and_offline(eng, orc, B, G, P, nb, mixed):
    irs = _irs(B, P, 6, 3300)
    mats = [[(g + k) % 6 for k in range(4)] if mixed else [0, 1, 2, 3] for g in range(G)]
    x = _blocks(2 * G, nb, B, 77)
    with _matrix(eng, B, P, G, 2, 2, irs, mats) as m:
        assert m.mac_plan()[0] == _pergroup(B, mixed)
        l0 = m.launches
        y = m.process(x)
        assert m.launches - l0 == nb and y.shape == (nb, 2 * G, B)
    # plain engine on 4G channels (channel 4g + 2i + o: input i of group g, IR mats[g][2i + o]), outputs summed on the host
    with eng.Engine(B, P, 4 * G, len(irs)) as p:
        for j, h in enumerate(irs):
            p.set_ir(j, h)
        for g in range(G):
            for t in range(4):
                p.bind(4 * g + t, 4 * g + t + 1, mats[g][t])
        xd = np.ascontiguousarray(np.repeat(x.reshape(nb, G, 2, B), 2, axis=2).reshape(nb, 4 * G, B))
        yp = p.process(xd).reshape(nb, G, 2, 2, B)
        ysum = yp[:, :, 0] + yp[:, :, 1]                                 # [nb][G][o][B]
    e_, l2 = parity(y.reshape(nb, G, 2, B), ysum)
    assert e_ <= TOL and l2 <= TOL, (e_, l2)
    for g in (0, 1, G // 2, G - 1):
        xs = np.ascontiguousarray(x[:, 2 * g:2 * g + 2].transpose(1, 0, 2)).reshape(2, nb * B)
        got = np.ascontiguousarray(y[:, 2 * g:2 * g + 2].transpose(1, 0, 2)).reshape(2, nb * B)
        e_, l2 = parity(got, _ref22(xs, irs, mats[g], nb, B))
        assert e_ <= TOL and l2 <= TOL, (g, e_, l2)
        # streaming == offline: the C restatement of the reference's convolvePeriodic, per term, summed
        off = np.zeros((2, nb * B))
        for o in range(2):
            for i in range(2):
                off[o] += orc.convolve_periodic(xs[i], irs[mats[g][i * 2 + o]], B)[0, :nb * B]
        e_, l2 = parity(got, off)
        assert e_ <= TOL and l2 <= TOL, (g, e_, l2)


@pytest.mark.parametrize("B,G", [(512, 900), (256, 41)])
def test_staged_ir_switch_matches_plain_engine(eng, B, G):
    """stage_ir on a matrix IR: the round-robin refresh (one partition per block step, in its own k_fwd launch) switches the
    right output channels exactly as on the plain engine."""
    P, nb, k = 6, 16, 5
    irs = _irs(B, P, 2, 3400)
    new = synth.decaying_ir(3499, P * B - 11, 3)
    x = _blocks(G, nb, B, 9)
    with _matrix(eng, B, P, G, 1, 2, irs, [[0, 1]] * G) as m:
        y0 = m.process(x[:k])
        m.stage_ir(1, new)
        l0 = m.launches
        y1 = m.process(x[k:])
        assert m.launches - l0 == 2 * (nb - k)                           # the block step + the refresh launch while an IR is staged
    y = np.concatenate([y0, y1])
    want = _plain_dup12(eng, B, P, x, irs, [[0, 1]] * G, stage=(k, 1, new))
    assert np.array_equal(y, want)


def test_host_paths_agree_and_reset_restores(eng):
    """process (one block per call: the captured-graph path; several blocks: the three-stage pipeline), process_device and
    submit/wait give the same bits; reset brings back the first outputs."""
    torch = pytest.importorskip("torch")
    for ins, G in ((1, 60), (2, 30)):                                   # one block in and out fits the captured graph's staging
        B, P, nb = 512, 5, 10
        irs = _irs(B, P, 4, 3500)
        x = _blocks(ins * G, nb, B, 11 + ins)
        with _matrix(eng, B, P, G, ins, 2, irs, [list(range(2 * ins))] * G) as m:
            d_in = torch.from_numpy(x).cuda()
            d_out = torch.empty((nb, 2 * G, B), device="cuda", dtype=torch.float32)
            torch.cuda.synchronize()
            for b in range(nb):
                m.process_device(d_in[b].data_ptr(), d_out[b].data_ptr(), 1)
            m.synchronize()
            want = d_out.cpu().numpy()
            m.reset()
            got = np.stack([m.process(x[b]) for b in range(nb)])
            assert np.array_equal(got, want), ins
            m.reset()
            assert np.array_equal(np.concatenate([m.process(x[:3]), m.process(x[3:])]), want), ins
            m.reset()
            hin, hout = eng.pinned_empty((nb, ins * G, B)), eng.pinned_empty((nb, 2 * G, B))
            hin[:] = x
            m.submit(hin[:4], hout[:4])
            m.submit(hin[4:], hout[4:])
            m.wait()
            assert np.array_equal(np.array(hout), want), ins
            eng.pinned_free(hin)
            eng.pinned_free(hout)


def test_fdl_spectrum_and_state_bytes(eng):
    B, G, P, nb = 512, 200, 7, 5
    irs = _irs(B, P, 2, 3600)
    x = _blocks(G, nb, B, 13)
    with _matrix(eng, B, P, G, 1, 2, irs, [[0, 1]] * G) as m, eng.Engine(B, P, 2 * G, 2) as p:
        for j, h in enumerate(irs):
            p.set_ir(j, h)
        p.bind(0, 2 * G, 0)
        m.process(x)
        p.process(np.ascontiguousarray(np.repeat(x, 2, axis=1)))
        for g in (0, 1, G - 1):
            for age in (0, 1, nb - 1):
                assert np.array_equal(m.fdl_spectrum(g, age), p.fdl_spectrum(2 * g, age)), (g, age)
        fdl_g = G * P * (B) * 8                                          # M = B: G input rows of P packed spectra of M complex
        assert p.state_bytes - m.state_bytes >= fdl_g, (p.state_bytes, m.state_bytes)
        with pytest.raises(eng.IrbError):
            m.fdl_spectrum(G, 0)                                         # `chan` is an input channel: there are G of them


def test_unsupported_calls_are_state_errors_and_the_engine_keeps_working(eng):
    B, G, P, nb = 512, 40, 4, 6
    irs = _irs(B, P, 2, 3700)
    x = _blocks(G, nb, B, 17)
    with _matrix(eng, B, P, G, 1, 2, irs, [[0, 1]] * G) as m:
        y0 = m.process(x[:3])
        calls = [lambda: m.bind(0, 1, 0), lambda: m.process_callback(x[3:4]), lambda: m.set_active_channels(G // 2),
                 lambda: m.set_mac_split(1, 1), lambda: m.set_fused_step(False)]
        for c in calls:
            with pytest.raises(eng.IrbError) as ex:
                c()
            assert ex.value.code == eng.IRB_ERR_STATE and "matrix" in str(ex.value)
        m.set_fused_step(True)                                           # the one form there is
        with pytest.raises(eng.IrbError) as ex:
            m.bind_matrix(0, G + 1, [0, 1])
        assert ex.value.code == eng.IRB_ERR_ARG
        with pytest.raises(eng.IrbError) as ex:
            m.bind_matrix(0, 1, [0, 2])
        assert ex.value.code == eng.IRB_ERR_ARG
        y1 = m.process(x[3:])
    assert np.array_equal(np.concatenate([y0, y1]), _plain_dup12(eng, B, P, x, irs, [[0, 1]] * G))
    with eng.Engine(B, P, 8, 2) as p:
        assert eng.lib().irb_engine_bind_matrix(p._h, 0, 1, (ctypes.c_int * 2)(0, 1)) == eng.IRB_ERR_STATE     # a plain engine binds channels


def test_timing_records_one_launch_per_step(eng):
    B, G, P, nb = 512, 1000, 8, 12
    irs = _irs(B, P, 2, 3800)
    with _matrix(eng, B, P, G, 1, 2, irs, [[0, 1]] * G) as m:
        m.set_timing(True)
        m.process(_blocks(G, nb, B, 3))
        step, mac = m.timings()
        assert len(step) == nb and np.all(step > 0) and np.array_equal(step, mac)
