#!/usr/bin/env python
"""bench_convolve_batch.py -- the batched linear convolution (irb_convolve_batch / irb_convolve_batch_device) on one GPU.

Two workloads, each from pinned host buffers and device-resident (torch tensors), in one process:
  * farina: 256 captures x 2^20 samples convolved with one shared inverse sweep (irb_ess_generate(..., inverse=1), 2^20
            samples), N = 2^21, only the window from 4 800 samples before lag len_sweep - 1 to 48 000 after it is written (the linear
            IR, 1 s at 48 kHz, and the end of the harmonic IRs in front of it).  Compared in the same process with one
            irb_convolve_nonperiodic call per capture (the full 2^21-sample result each) and, device-resident, with the same batched
            call asking for the full result (what the window saves in bytes and time).
  * render: 1 024 clips x 192 000 samples, one 48 000-tap IR per clip, the full 239 999-sample result, N = 2^18.
For each: device ms (CUDA events, irb_last_compute_ms), wall ms, items/s, achieved GB/s under the byte model below, and for the
host path the host<->device bytes (uploads and downloads) over the wall time as a fraction of the copy-only ceiling with both
directions at once, measured in the same run (CopyProbe).
The card's name and power limit are read in the same run.  One JSON line per workload and path; --out writes them all (jsonl).

Byte model (HBM traffic of the four-step path, per item; M = N/2 complex points, 8 bytes each):
  signal column pass   read 4 len_x, write 8M;   row-pair kernel read + write 16M;   inverse column pass read 8M, write 4 out_len
  per-item IR, added:  column pass read 4 len_h, write 8M; row pass in place 16M; split read 8M, write 8M; the row-pair kernel's
                       read of the IR spectrum 8M.   A shared IR's spectrum is read from L2 and not counted.

  python bench_convolve_batch.py [--reps 3] [--out profiles/r05_bench_convolve_batch.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
SR = 48000.0


def card():
    import torch
    info = {"card": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"], info["sm_clock_max_mhz"] = float(q[0]), float(q[1])
    except Exception as ex:                                     # the numbers stand without it, but say so
        info["power_limit_w"] = "unavailable: %s" % ex
    return info


def hbm_bytes(N, len_x, len_h, out_len, per_item):
    M = N // 2
    b = 4 * len_x + 8 * M + 16 * M + 8 * M + 4 * out_len
    if per_item:
        b += 4 * len_h + 8 * M + 16 * M + 16 * M + 8 * M
    return b


def copy_ceiling(eng, nbytes, iters=8):
    """copy-only GB/s host -> device, device -> host and both at once (pinned, whole buffer per copy, no kernels)"""
    p = eng.CopyProbe(nbytes, 0)
    p.run(2, 3)
    out = {d: nbytes * iters * (2 if k == 3 else 1) / p.run(iters, k) / 1e9 for d, k in (("h2d_gbs", 1), ("d2h_gbs", 2), ("both_gbs", 3))}
    p.close()
    return out


def timed(fn, reps):
    """(wall s, device s) of the fastest of `reps` calls after one warm-up call"""
    from irbaboon_b200 import engine as eng
    fn()
    best = None
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        r = (time.perf_counter() - t0, eng.last_compute_ms() * 1e-3)
        best = r if best is None or r[0] < best[0] else best
    return best


def line(name, path, batch, N, len_x, len_h, out_len, per_item, wall, dev, ceiling=None, host_bytes=0, **extra):
    hb = hbm_bytes(N, len_x, len_h, out_len, per_item) * batch
    r = {"bench": "bench_convolve_batch", "workload": name, "path": path, "items": batch, "fft_points": N, "len_x": len_x, "len_h": len_h,
         "ir": "one per item" if per_item else "shared", "out_len": out_len, "device_ms": dev * 1e3, "wall_ms": wall * 1e3,
         "items_per_s_wall": batch / wall, "items_per_s_device": batch / dev, "hbm_bytes_model": hb, "device_gbs_at_model": hb / dev / 1e9}
    if ceiling:
        r["host_bytes_moved"] = host_bytes
        r["host_gbs_wall"] = host_bytes / wall / 1e9
        r["copy_ceiling"] = ceiling
        r["frac_of_both_directions_ceiling"] = host_bytes / wall / 1e9 / ceiling["both_gbs"]
    r.update(extra)
    return r


def farina(eng, torch, info, args):
    n, batch = 1 << 20, args.farina_captures
    sweep = eng.ess(n / SR, SR, 20.0, 24000.0).astype(np.float32)
    inv = eng.ess(n / SR, SR, 20.0, 24000.0, 0.0, True).astype(np.float32)
    ls = len(sweep)
    off, out_len = ls - 1 - 4800, 4800 + 48000
    N, full_len = 1 << 21, n + ls - 1
    from irbaboon_b200 import synth
    caps = eng.pinned_empty((batch, n))
    irs = [synth.decaying_ir(3000 + j, 48000, j) for j in range(4)]
    base = [eng.convolve_nonperiodic(sweep, h)[0, :n] for h in irs]
    for j in range(batch):
        caps[j] = base[j % 4] + synth.white_noise(4000 + j, 0, n) * np.float32(1e-3)
    out = eng.pinned_empty((batch, out_len))
    ceiling = copy_ceiling(eng, caps.nbytes)
    host_bytes = caps.nbytes + inv.nbytes + out.nbytes
    res = []
    wall, dev = timed(lambda: eng.convolve_batch(caps, inv, off, out_len, out=out), args.reps)
    res.append(line("farina", "host_pinned", batch, N, n, ls, out_len, False, wall, dev, ceiling, host_bytes, window=[off, off + out_len], **info))
    # the per-call loop in the same process: irb_convolve_nonperiodic, one capture at a time, the full result to pageable memory
    eng.convolve_nonperiodic(caps[0], inv)
    ts, ds = [], []
    for j in range(batch):
        t0 = time.perf_counter()
        eng.convolve_nonperiodic(caps[j], inv)
        ts.append(time.perf_counter() - t0)
        ds.append(eng.last_compute_ms() * 1e-3)
    res.append(line("farina", "per_call_loop_host", batch, N, n, ls, full_len, False, float(np.sum(ts)), float(np.sum(ds)),
                    per_call_wall_ms_median=float(np.median(ts)) * 1e3, per_call_device_ms_median=float(np.median(ds)) * 1e3, **info))
    # device-resident: windowed and full output
    d_caps = torch.from_numpy(np.asarray(caps)).cuda()
    d_inv = torch.from_numpy(inv).cuda()
    d_out = torch.empty((batch, out_len), dtype=torch.float32, device="cuda")
    d_full = torch.empty((batch, full_len), dtype=torch.float32, device="cuda")

    def dev_call(o, o_off, o_len):
        eng.convolve_batch_device(d_caps.data_ptr(), batch, n, d_inv.data_ptr(), o.data_ptr(), len_h=ls, h_batch=1, out_offset=o_off, out_len=o_len)
        torch.cuda.synchronize()
    wall_w, dev_w = timed(lambda: dev_call(d_out, off, out_len), args.reps)
    wall_f, dev_f = timed(lambda: dev_call(d_full, 0, full_len), args.reps)
    same = bool(torch.equal(d_full[:, off:off + out_len], d_out)) and bool(np.array_equal(d_out.cpu().numpy(), out))
    saved = 4 * (full_len - out_len) * batch
    res.append(line("farina", "device_resident", batch, N, n, ls, out_len, False, wall_w, dev_w, window=[off, off + out_len],
                    full_output_device_ms=dev_f * 1e3, full_output_wall_ms=wall_f * 1e3, window_saves_hbm_bytes=saved,
                    window_saves_device_ms=(dev_f - dev_w) * 1e3, window_equals_full_slice=same, **info))
    eng.pinned_free(caps); eng.pinned_free(out)
    return res


def render(eng, torch, info, args):
    batch, lx, lh = args.render_clips, 192000, 48000
    full_len, N = lx + lh - 1, 1 << 18
    from irbaboon_b200 import synth
    x = eng.pinned_empty((batch, lx))
    h = eng.pinned_empty((batch, lh))
    for j in range(batch):
        x[j] = synth.white_noise(5000 + j, 0, lx) * np.float32(0.1)
        h[j] = synth.decaying_ir(6000 + j, lh, j % 8)
    out = eng.pinned_empty((batch, full_len))
    ceiling = copy_ceiling(eng, x.nbytes)
    host_bytes = x.nbytes + h.nbytes + out.nbytes
    res = []
    wall, dev = timed(lambda: eng.convolve_batch(x, h, out=out), args.reps)
    res.append(line("render", "host_pinned", batch, N, lx, lh, full_len, True, wall, dev, ceiling, host_bytes, **info))
    d_x, d_h = torch.from_numpy(np.asarray(x)).cuda(), torch.from_numpy(np.asarray(h)).cuda()
    d_out = torch.empty((batch, full_len), dtype=torch.float32, device="cuda")

    def dev_call():
        eng.convolve_batch_device(d_x.data_ptr(), batch, lx, d_h.data_ptr(), d_out.data_ptr(), len_h=lh, h_batch=batch)
        torch.cuda.synchronize()
    wall, dev = timed(dev_call, args.reps)
    same = bool(np.array_equal(d_out.cpu().numpy(), out))
    res.append(line("render", "device_resident", batch, N, lx, lh, full_len, True, wall, dev, equals_host_path=same, **info))
    eng.pinned_free(x); eng.pinned_free(h); eng.pinned_free(out)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="farina,render")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--farina-captures", type=int, default=256)
    ap.add_argument("--render-clips", type=int, default=1024)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if args.reps < 1:
        ap.error("--reps must be >= 1")
    import torch
    from irbaboon_b200 import engine as eng
    eng.set_device(0)
    info = card()
    lines = []
    for w in args.workloads.split(","):
        for r in {"farina": farina, "render": render}[w](eng, torch, info, args):
            print(json.dumps(r), flush=True)
            lines.append(r)
    if args.out:
        with open(args.out, "w") as f:
            for r in lines:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
