#!/usr/bin/env python
"""bench_configs.py -- the BASELINE.json configurations that are NOT the headline bench line (bench.py measures
configs[2]): one JSON object per configuration, written to stdout and, with --out, to a file.

  c1  mono 48 kHz, B=512, 1 s IR, 10 s white noise through convolvePeriodic (offline; CPU reference beside it)
  c2  stereo 48 kHz, B=256, 4 s IR, single stream, block by block (latency path): p50/p99 device and round-trip time
  c4  S streams with per-stream 10 s IRs (480k taps), B=1024 (per-row-IR MAC kernel); S defaults to what one GPU holds
  c5  batched ESS IR capture: 2^20-sample sweep captures deconvolved by spectral division

The CPU reference legs (c1, c5) run the reference's own object code (oracle/_ref) as the reported baseline and as the
checker, exactly like bench.py's cpu_baseline leg -- never as the thing measured as "ours".
Synthetic inputs (irbaboon_b200/synth.py).  Times are CUDA-event device times where the library records them and
wall-clock around the C-ABI call otherwise (stated per entry).
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
SR = 48000.0


def peak():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        return 6650.0


def c1(eng, synth, args):
    x = synth.white_noise(1001, 0, 480000)
    h = synth.decaying_ir(2000, 48000)
    eng.convolve_periodic(x[:4096], h[:1024], 512)               # context + twiddles
    ts = []
    for _ in range(5):
        t0 = time.perf_counter()
        y = eng.convolve_periodic(x, h, 512)
        ts.append(time.perf_counter() - t0)
    out = {"config": "c1", "what": "irb_convolve_periodic(mono 10 s, 48000-tap IR, B=512), host buffers, wall clock (H2D + 4 kernels + D2H)",
           "seconds_best": min(ts), "seconds_median": float(np.median(ts)), "realtime_factor": 10.0 / min(ts), "output_samples": int(y.shape[1])}
    try:
        import oracle
        if oracle.have_reference():
            ref = oracle.Reference()
            t0 = time.perf_counter()
            yr = ref.convolve_periodic(x, h, 512)
            out["cpu_reference_seconds_1_thread"] = time.perf_counter() - t0
            out["max_abs_vs_reference"] = float(np.abs(y - yr).max())
    except Exception as ex:                                       # the checker is optional here
        out["cpu_reference"] = "unavailable: %s" % ex
    return out


def c2(eng, synth, args):
    B, Lh, C = 256, 192000, 2
    P = -(-Lh // B)
    nblk = args.c2_blocks
    with eng.Engine(B, P, C, 2) as e:
        for c in range(C):
            e.set_ir(c, synth.decaying_ir(2000 + c, Lh, c))
            e.bind(c, c + 1, c)                                   # channel-wise stereo IR (IRStereoAudioStereo)
        if args.c2_split:
            e.set_mac_split(*[int(v) for v in args.c2_split.split(",")])
        plan = e.mac_plan()
        x = eng.pinned_empty((nblk, C, B))
        y = eng.pinned_empty((nblk, C, B))
        rng = np.random.default_rng(1002)
        x[:] = rng.random((nblk, C, B), dtype=np.float32) * 2 - 1
        e.process(x[:P], y[:P])                                   # fill the FDL
        e.set_timing(True)
        rt = np.zeros(nblk)
        for i in range(nblk):
            t0 = time.perf_counter()
            e.process(x[i], y[i])                                 # one host round trip per block, as a live callback
            rt[i] = time.perf_counter() - t0
        step_ms, mac_ms = e.timings()
        e.set_timing(False)
        # the same round trip without the per-kernel timing events: copy-in, kernels and copy-out replay as one CUDA graph
        rtg = np.zeros(nblk)
        for i in range(nblk):
            t0 = time.perf_counter()
            e.process(x[i], y[i])
            rtg[i] = time.perf_counter() - t0
        eng.pinned_free(x); eng.pinned_free(y)
    period = 1e3 * B / SR
    return {"config": "c2", "what": "stereo, B=256, 4 s stereo IR (750 partitions/channel), one stream, one irb_engine_process call per block",
            "blocks": nblk, "block_period_ms": period, "mac_plan": {"slots_kernel": plan[0], "split_in_tile": plan[1], "cluster": plan[2]},
            "device_ms": {"p50": float(np.percentile(step_ms, 50)), "p99": float(np.percentile(step_ms, 99)), "max": float(step_ms.max())},
            "roundtrip_ms": {"p50": float(np.percentile(rt, 50) * 1e3), "p99": float(np.percentile(rt, 99) * 1e3), "max": float(rt.max() * 1e3)},
            "roundtrip_graph_ms": {"p50": float(np.percentile(rtg, 50) * 1e3), "p99": float(np.percentile(rtg, 99) * 1e3), "max": float(rtg.max() * 1e3)},
            "mac_kernel_ms_mean": float(mac_ms.mean()), "realtime": bool(np.percentile(rt, 99) * 1e3 < period)}


def c3cap(eng, synth, args):
    """Real-time capacity of configs[2]'s shape (SURVEY 8d): the largest stream count S whose p99 block step stays under
    the 10.667 ms block period with all S streams resident (FDL 0.77 MB per stream)."""
    import torch
    B, Lh = 512, 96000
    P = int(np.ceil(np.float32(Lh) / np.float32(B)))
    period = 1e3 * B / SR
    h = synth.decaying_ir(2000, Lh)
    rows = []
    for S in [int(v) for v in args.c3cap_streams.split(",")]:
        e = eng.Engine(B, P, S, 1)
        e.set_ir(0, h)
        stream = torch.cuda.Stream()
        torch.cuda.set_stream(stream)
        e.set_stream(stream.cuda_stream)
        d_in = (torch.rand((2, S, B), device="cuda") * 2 - 1).contiguous()
        d_out = torch.empty((S, B), device="cuda")
        for i in range(P + 5):
            e.process_device(d_in[i % 2].data_ptr(), d_out.data_ptr(), 1)
        torch.cuda.synchronize()
        e.set_timing(True)
        for i in range(args.c3cap_steps):
            e.process_device(d_in[i % 2].data_ptr(), d_out.data_ptr(), 1)
        step_ms, mac_ms = e.timings()
        e.set_timing(False)
        alg = (S + 1) * P * (B + 1) * 8
        rows.append({"streams": S, "state_gb": e.state_bytes / 1e9, "steps": int(len(step_ms)),
                     "step_ms": {"p50": float(np.percentile(step_ms, 50)), "p99": float(np.percentile(step_ms, 99)), "p99.9": float(np.percentile(step_ms, 99.9)),
                                 "max": float(step_ms.max()), "over_period": int((step_ms >= period).sum())}, "mac_gbs": alg / (mac_ms.mean() * 1e-3) / 1e9, "realtime": bool(np.percentile(step_ms, 99) < period),
                     "headroom": float(period / np.percentile(step_ms, 99))})
        e.close()
        del d_in, d_out
        torch.cuda.empty_cache()
    ok = [r["streams"] for r in rows if r["realtime"]]
    return {"config": "c3cap", "what": "streams sharing one 2 s IR, B=512, all resident on one GPU: block-step latency vs the %.3f ms block period, %d timed steps each" % (period, args.c3cap_steps),
            "block_period_ms": period, "runs": rows, "rt_channels_sustained": max(ok) if ok else 0}


def group(eng, synth, args):
    """configs[2] shape through ONE process driving every visible GPU (irb_group_*): host buffers in, host buffers out."""
    B, Lh = 512, 96000
    P = int(np.ceil(np.float32(Lh) / np.float32(B)))
    nd = eng.device_count()
    S = args.group_streams * nd
    K = args.group_blocks
    h = synth.decaying_ir(2000, Lh)
    with eng.Group(list(range(nd)), B, P, S, 1) as g:
        g.set_ir(0, h)
        x = eng.pinned_empty((K, S, B))
        y = eng.pinned_empty((K, S, B))
        rng = np.random.default_rng(1003)
        x[:] = rng.random((K, S, B), dtype=np.float32) * 2 - 1
        for _ in range(-(-P // K) + 1):                           # fill the FDLs
            g.process(x, y)
        ts = []
        for _ in range(3):
            t0 = time.perf_counter()
            g.process(x, y)
            ts.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        for i in range(min(K, 8)):
            g.process(x[i], y[i])
        one = (time.perf_counter() - t0) / min(K, 8)
        out = {"config": "group", "what": "one process, %d GPU(s), %d streams each sharing one 2 s IR, B=512: irb_group_process(host in, host out, %d blocks), "
                                         "pinned buffers, wall clock" % (nd, args.group_streams, K),
               "gpus": nd, "streams_total": S, "ranges": g.ranges, "seconds_best": min(ts), "rt_channels_e2e": S * B * K / min(ts) / SR,
               "ms_per_block": 1e3 * min(ts) / K, "single_block_roundtrip_ms": 1e3 * one, "block_period_ms": 1e3 * B / SR, "checksum": float(np.abs(y[-1]).sum())}
        eng.pinned_free(x); eng.pinned_free(y)
    return out


def c4(eng, synth, args):
    import torch
    B, Lh = 1024, 480000
    P = int(np.ceil(np.float32(Lh) / np.float32(B)))
    S = args.c4_streams
    t0 = time.perf_counter()
    e = eng.Engine(B, P, S, S)
    irs = [synth.decaying_ir(2000 + j, Lh, j) for j in range(8)]
    for s in range(S):
        e.set_ir(s, irs[s % 8])
        e.bind(s, s + 1, s)
    setup = time.perf_counter() - t0
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    e.set_stream(stream.cuda_stream)
    d_in = (torch.rand((2, S, B), device="cuda") * 2 - 1).contiguous()
    d_out = torch.empty((S, B), device="cuda")
    for i in range(5):
        e.process_device(d_in[i % 2].data_ptr(), d_out.data_ptr(), 1)
    torch.cuda.synchronize()
    e.set_timing(True)
    for i in range(args.c4_steps):
        e.process_device(d_in[i % 2].data_ptr(), d_out.data_ptr(), 1)
    step_ms, mac_ms = e.timings()
    e.set_timing(False)
    alg = S * 2 * P * (B + 1) * 8                                 # FDL + private IR per stream (SURVEY 8d)
    period = 1e3 * B / SR
    out = {"config": "c4", "what": "%d streams, per-stream 10 s IRs (480000 taps, %d partitions), B=1024, one GPU, device-resident I/O" % (S, P),
           "streams": S, "state_gb": e.state_bytes / 1e9, "setup_seconds": setup, "block_period_ms": period,
           "step_ms": {"p50": float(np.percentile(step_ms, 50)), "p99": float(np.percentile(step_ms, 99))},
           "mac_kernel_ms_mean": float(mac_ms.mean()), "algorithmic_bytes_per_launch": alg,
           "achieved_gbs": alg / (mac_ms.mean() * 1e-3) / 1e9, "frac_of_measured_peak": alg / (mac_ms.mean() * 1e-3) / 1e9 / peak(),
           "realtime": bool(np.percentile(step_ms, 99) < period), "rt_channels": S * period / float(np.mean(step_ms))}
    e.close()
    return out


def c5(eng, synth, args):
    n = 1 << 20
    nb = args.c5_captures
    sweep = eng.ess(n / SR, SR, 20.0, 24000.0).astype(np.float32)
    irs = [synth.decaying_ir(3000 + j, 48000, j) for j in range(4)]
    base = [eng.convolve_nonperiodic(sweep, h)[0, :n] for h in irs]
    caps = eng.pinned_empty((nb, n))
    res = eng.pinned_empty((nb, n))
    for j in range(nb):
        caps[j] = base[j % 4] + synth.white_noise(4000 + j, 0, n) * np.float32(1e-3)
    eng.deconvolve_batch(caps[:2], sweep, SR, False)              # warm-up
    out = {"config": "c5", "what": "%d captures of a 2^20-sample exponential sine sweep deconvolved by spectral division (fp::convolution::deconvolve), "
                                   "host buffers, wall clock around irb_deconvolve_batch" % nb, "captures": nb, "fft_points": n}
    for smoothing in (False, True):
        ts = []
        for _ in range(3 if not smoothing else 2):          # the first call of a shape pays its device allocations; later ones recycle them
            t0 = time.perf_counter()
            y = eng.deconvolve_batch(caps, sweep, SR, smoothing, out=res)
            ts.append((time.perf_counter() - t0, eng.last_compute_ms() * 1e-3))
        key = "smoothed" if smoothing else "plain"
        wall, dev = min(ts)
        # realistic traffic of the four-step path: 2 FFT passes (read+write) forward, fused divide, 2 passes inverse
        four_step = 5 * 2 * (n // 2) * 8
        out[key] = {"wall_seconds_pinned_host_buffers": wall, "captures_per_s_e2e": nb / wall, "device_seconds_kernels_only": dev,
                    "captures_per_s_device": nb / dev, "min_bytes_per_capture": 2 * n * 4, "four_step_bytes_per_capture": four_step,
                    "device_gbs_at_four_step_bytes": nb * four_step / dev / 1e9, "frac_of_measured_peak": nb * four_step / dev / 1e9 / peak(),
                    "peak_abs": float(np.abs(y).max())}
    # secondary (SURVEY 8d): the Farina form of the same capture, convolveNonPeriodic(capture, inverse sweep) at N = 2^21, as the
    # reference runs it (one irb_convolve_nonperiodic call per capture, the full result) and batched (irb_convolve_batch, every
    # capture at once, only the window from 4 800 samples before lag len_sweep - 1 to 48 000 after it)
    sweep_inv = eng.ess(n / SR, SR, 20.0, 24000.0, 0.0, True).astype(np.float32)
    eng.convolve_nonperiodic(caps[0], sweep_inv)
    kf, ts, dev = min(nb, 8), [], []
    for j in range(kf):
        t0 = time.perf_counter()
        yf = eng.convolve_nonperiodic(caps[j], sweep_inv)
        ts.append(time.perf_counter() - t0)
        dev.append(eng.last_compute_ms() * 1e-3)
    out["farina_variant"] = {"what": "convolveNonPeriodic(capture, ExpSineSweep inverse filter), N = 2^21, one call per capture, pageable result",
                             "captures": kf, "wall_seconds_per_capture_median": float(np.median(ts)), "device_seconds_per_capture_median": float(np.median(dev)),
                             "output_samples": int(yf.shape[1])}
    off, win = len(sweep_inv) - 1 - 4800, 4800 + 48000
    wres = eng.pinned_empty((nb, win))
    eng.convolve_batch(caps[:2], sweep_inv, off, win, out=wres[:2])
    ts = []
    for _ in range(3):
        t0 = time.perf_counter()
        eng.convolve_batch(caps, sweep_inv, off, win, out=wres)
        ts.append((time.perf_counter() - t0, eng.last_compute_ms() * 1e-3))
    wall, dev_b = min(ts)
    out["farina_variant_batched"] = {"what": "irb_convolve_batch of all captures with the inverse filter, N = 2^21, pinned host buffers, window [%d, %d)" % (off, off + win),
                                     "captures": nb, "wall_seconds": wall, "wall_seconds_per_capture": wall / nb, "device_seconds": dev_b,
                                     "device_seconds_per_capture": dev_b / nb, "output_samples": win}
    eng.pinned_free(wres)
    try:
        import oracle
        if oracle.have_reference():
            ref = oracle.Reference()
            T = max(1, ref.hardware_threads())
            k = min(nb, T)
            secs, _ = ref.bench_deconvolve(T, np.array(caps[:k]), sweep, SR, False)
            out["cpu_reference"] = {"captures_per_s": k / secs, "threads": T, "captures": k, "smoothing": False}
    except Exception as ex:
        out["cpu_reference"] = "unavailable: %s" % ex
    eng.pinned_free(caps); eng.pinned_free(res)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="c1,c2,c4,c5")
    ap.add_argument("--out", default="")
    ap.add_argument("--c2-blocks", type=int, default=10000)
    ap.add_argument("--c2-split", default="", help="force the few-row MAC split 'split_in,cluster' (default: automatic)")
    ap.add_argument("--c3cap-streams", default="65536,81920,86016")
    ap.add_argument("--c3cap-steps", type=int, default=300)
    ap.add_argument("--group-streams", type=int, default=16384, help="group: streams per GPU")
    ap.add_argument("--group-blocks", type=int, default=16)
    ap.add_argument("--c4-streams", type=int, default=8192)
    ap.add_argument("--c4-steps", type=int, default=30)
    ap.add_argument("--c5-captures", type=int, default=256)
    args = ap.parse_args()
    from irbaboon_b200 import engine as eng
    from irbaboon_b200 import synth
    eng.set_device(0)
    res = []
    for name in args.configs.split(","):
        r = {"c1": c1, "c2": c2, "c3cap": c3cap, "c4": c4, "c5": c5, "group": group}[name](eng, synth, args)
        print(json.dumps(r, default=float), flush=True)
        res.append(r)
    if args.out:
        json.dump(res, open(args.out, "w"), indent=1, default=float)


if __name__ == "__main__":
    main()
