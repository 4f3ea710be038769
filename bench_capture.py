#!/usr/bin/env python
"""bench_capture.py -- the batched IR capture ending in IRs (irb_deconvolve_chop_batch, irb_ir_chop_batch_device) on one GPU.

The c5 shape: 256 captures x 2^20 samples of an exponential sine sweep (1/13-octave smoothing off and on), each divided by the
sweep, then cut to ir_length = 2 048 and 48 000 samples around its peak and normalised to 0 dB (fp::ir::IRchop + tools::normalize).
Four runs per (smoothing, ir_length), in one process:
  full_download  irb_deconvolve_batch from pinned host buffers, the whole [256][2^20] result downloaded (what a batch user paid before)
  chop_host      irb_deconvolve_chop_batch from pinned host buffers: only [256][ir_length] and the peak positions come back
  chop_device    irb_deconvolve_batch_device + irb_ir_chop_batch_device on device-resident captures (torch tensors)
  facade_loop    the host facade's fp::ir::IRchop + tools::normalize over the downloaded rows, one row at a time (host only)
Wall ms (host clock around a call that ends synchronised) and device ms (irb_last_compute_ms: CUDA events around the kernels), the
best of --reps calls after one warm-up.  The chop's own device ms is reported apart on the device-resident path.  Every line carries
the card's name and power limit, read in the same run, and whether the IRs of the runs are the same bits.

--ab LIB: the no-regression A/B of the division instead: device-resident plain division 256 x 2^20 (irb_deconvolve_batch_device),
this library and LIB (IRB_LIB) alternating in --rounds rounds, each a fresh process.

  python bench_capture.py [--reps 3] [--out profiles/r07_bench_capture.jsonl]
  python bench_capture.py --ab parent/libirb_b200.so [--rounds 3] [--out profiles/r07_division_ab.jsonl]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
SR = 48000.0
N = 1 << 20


def card():
    import torch
    info = {"card": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        info["power_limit_w"] = q.stdout.strip()
    except Exception as ex:
        info["power_limit_w"] = "unavailable: %s" % ex
    return info


def captures(eng, synth, batch):
    """the c5 captures (bench_configs.py): four decaying rooms convolved with the sweep, plus noise at -60 dB"""
    sweep = eng.ess(N / SR, SR, 20.0, 24000.0).astype(np.float32)
    base = [eng.convolve_nonperiodic(sweep, synth.decaying_ir(3000 + j, 48000, j))[0, :N] for j in range(4)]
    caps = eng.pinned_empty((batch, N))
    for j in range(batch):
        caps[j] = base[j % 4] + synth.white_noise(4000 + j, 0, N) * np.float32(1e-3)
    return caps, sweep


def facade(tmp):
    """the facade's C view (tests/cpp/facade_capi.cpp), compiled into a temporary directory"""
    fp = os.path.join(ROOT, "irbaboon_b200", "fp")
    so = os.path.join(tmp, "libfacade_capi.so")
    subprocess.check_call(["g++", "-std=c++14", "-O2", "-fPIC", "-shared", "-o", so, os.path.join(ROOT, "tests", "cpp", "facade_capi.cpp"), "-I" + fp,
                           "-I" + os.path.join(ROOT, "include"), "-L" + fp, "-lfp_b200", "-L" + os.path.dirname(fp), "-lirb_b200", "-Wl,-rpath," + fp,
                           "-Wl,-rpath," + os.path.dirname(fp)])
    h = ctypes.CDLL(so)
    f32p = ctypes.POINTER(ctypes.c_float)
    h.fac_ir_chop.argtypes = [f32p, ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_int, f32p]
    h.fac_normalize.argtypes = [f32p, ctypes.c_int, ctypes.c_int, ctypes.c_float]
    return h, f32p


def best(fn, reps):
    fn()                                                     # the first call of a shape pays its device allocations
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        extra = fn()
        ts.append((time.perf_counter() - t0, extra))
    return min(ts, key=lambda t: t[0])


def same(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return bool(np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(a[~np.isnan(a)].view(np.uint32), b[~np.isnan(b)].view(np.uint32)))


def capture_runs(eng, torch, info, args):
    from irbaboon_b200 import synth
    caps, sweep = captures(eng, synth, args.captures)
    B = args.captures
    full = eng.pinned_empty((B, N))
    d_caps = torch.from_numpy(np.asarray(caps)).cuda()
    d_full = torch.empty((B, N), dtype=torch.float32, device="cuda")
    tmp = tempfile.mkdtemp(prefix="irb_bench_capture_")
    fac, f32p = facade(tmp)
    lines = []
    for smoothing in (False, True):
        def full_call():
            eng.deconvolve_batch(caps, sweep, SR, smoothing, out=full)
            return eng.last_compute_ms()
        w_full, dev_full = best(full_call, args.reps)
        base = dict(info, captures=B, fft_points=N, smoothing=smoothing)
        lines.append(dict(base, run="full_download", ir_length=None, wall_ms=1e3 * w_full, device_ms=dev_full, d2h_bytes=4 * B * N))
        for L in (2048, 48000):
            out = eng.pinned_empty((B, L))
            pos = np.empty((B, 2), np.int32)

            def chop_call():
                _, p = eng.deconvolve_chop_batch(caps, sweep, L, SR, smoothing, out=out, return_positions=True)
                pos[:] = p
                return eng.last_compute_ms()
            w_chop, dev_chop = best(chop_call, args.reps)
            d_out = torch.empty((B, L), dtype=torch.float32, device="cuda")
            d_pos = torch.empty((B, 2), dtype=torch.int32, device="cuda")

            def dev_call():
                eng.deconvolve_batch_device(d_caps.data_ptr(), B, N, sweep, d_full.data_ptr(), SR, smoothing)
                div = eng.last_compute_ms()
                eng.ir_chop_batch_device(d_full.data_ptr(), B, N, L, d_out.data_ptr(), positions_ptr=d_pos.data_ptr())
                torch.cuda.synchronize()
                return div, eng.last_compute_ms()
            w_dev, (dev_div, dev_ch) = best(dev_call, args.reps)
            chop_ms = []                                     # the chop alone, repeated: its spread
            for _ in range(args.reps * 3):
                eng.ir_chop_batch_device(d_full.data_ptr(), B, N, L, d_out.data_ptr(), positions_ptr=d_pos.data_ptr())
                chop_ms.append(eng.last_compute_ms())
            ref = np.empty((B, L), np.float32)
            t0 = time.perf_counter()
            for b in range(B):
                row = full[b]
                fac.fac_ir_chop(row.ctypes.data_as(f32p), N, L, -60.0, 50, ref[b].ctypes.data_as(f32p))
                fac.fac_normalize(ref[b].ctypes.data_as(f32p), 1, L, 0.0)
            w_fac = time.perf_counter() - t0
            dev_irs = d_out.cpu().numpy()
            eq_dev = same(out, dev_irs) and bool(np.array_equal(pos, d_pos.cpu().numpy()))
            eq_fac = same(out, ref)
            common = dict(base, ir_length=L)
            lines.append(dict(common, run="chop_host", wall_ms=1e3 * w_chop, device_ms=dev_chop, d2h_bytes=4 * B * L + 8 * B,
                              same_as_chop_device=eq_dev, same_as_facade_loop=eq_fac, peak_positions_first4=pos[:4, 0].tolist()))
            lines.append(dict(common, run="chop_device", wall_ms=1e3 * w_dev, device_ms=dev_div + dev_ch, division_device_ms=dev_div,
                              chop_device_ms_min=min(chop_ms), chop_device_ms_median=float(np.median(chop_ms)),
                              chop_gbs_at_one_read=4.0 * B * N / (min(chop_ms) * 1e-3) / 1e9))
            lines.append(dict(common, run="facade_loop", wall_ms=1e3 * w_fac, rows=B))
    return lines


def division_only(torch, info, args):
    """the division through IRB_LIB's own irb_deconvolve_batch_device (an older build lacks the newer entry points the binding loads)"""
    L = ctypes.CDLL(os.environ["IRB_LIB"])
    vp = ctypes.c_void_p
    L.irb_deconvolve_batch_device.argtypes = [vp, ctypes.c_int, ctypes.c_int, vp, ctypes.c_int, ctypes.c_double, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp]
    L.irb_last_compute_ms.restype = ctypes.c_double
    data = np.load(args.division_only)
    caps, sweep = data["caps"], np.ascontiguousarray(data["sweep"])
    B = caps.shape[0]
    d_caps = torch.from_numpy(caps).cuda()
    d_full = torch.empty((B, N), dtype=torch.float32, device="cuda")
    ms = []
    for i in range(8):
        rc = L.irb_deconvolve_batch_device(vp(d_caps.data_ptr()), B, N, sweep.ctypes.data_as(vp), len(sweep), SR, 0, 1, 1, vp(d_full.data_ptr()))
        assert rc == 0, rc
        if i:
            ms.append(L.irb_last_compute_ms())
    return [dict(info, device_plain_ms_min=min(ms), device_plain_ms_median=float(np.median(ms)), checksum=float(d_full.abs().sum().item()),
                 what="device-resident plain batched division, %d captures x 2^20 (irb_deconvolve_batch_device), device ms of 7 calls after one warm-up" % B)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--captures", type=int, default=256)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out")
    ap.add_argument("--ab", help="another build of libirb_b200.so: A/B of the division against it")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--division-only", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.ab:
        from irbaboon_b200 import engine as eng
        from irbaboon_b200 import synth
        eng.set_device(0)
        caps, sweep = captures(eng, synth, args.captures)                # the c5 captures, made once and shared by both libraries
        inputs = os.path.join(tempfile.mkdtemp(prefix="irb_bench_capture_"), "c5.npz")
        np.savez(inputs, caps=np.asarray(caps), sweep=sweep)
        lines = []
        here = os.environ.get("IRB_LIB") or os.path.join(ROOT, "irbaboon_b200", "libirb_b200.so")
        for r in range(args.rounds):
            for label, lib in (("this commit", here), ("parent commit", os.path.abspath(args.ab))):
                env = dict(os.environ, IRB_LIB=lib)
                res = subprocess.run([sys.executable, os.path.abspath(__file__), "--division-only", inputs], env=env,
                                     capture_output=True, text=True, check=True).stdout.strip().splitlines()[-1]
                lines.append(dict(json.loads(res), library=label, round=r + 1))
                print(json.dumps(lines[-1]), flush=True)
    else:
        import torch
        if not torch.cuda.is_available():
            raise SystemExit("bench_capture.py needs a GPU")
        if args.division_only:
            lines = division_only(torch, card(), args)
        else:
            from irbaboon_b200 import engine as eng
            eng.set_device(0)
            lines = capture_runs(eng, torch, card(), args)
        for ln in lines:
            print(json.dumps(ln), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            for ln in lines:
                f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
