#!/usr/bin/env python
"""bench_pcm.py -- the streaming engine fed float32, 16-bit and 24-bit PCM, in one process per GPU.

Headline shape by default: B = 512, P = 188 partitions, one shared IR, S streams per GPU.  For each format pair (F32/F32,
S16/S16, S24/S24) it reports, in one run:
  * device: the block step through irb_engine_process_device_pcm, the three formats alternating step by step (CUDA events);
  * feed:   the continuous host feed (REP back-to-back irb_engine_submit_pcm calls of K blocks, one wait), in real-time channels;
  * rt:     the largest stream count per GPU whose one-block-per-call host round trip (irb_engine_process_pcm, copies included)
            stays inside the block period (the search of bench.e2e_leg);
  * copy:   the copy-only ceiling at that format's bytes per block (CopyProbe: H2D and D2H at once, no kernels).
With the card's name and power limit read in the same run.  Rank 0 prints one JSON line.

  python bench_pcm.py --gpus 1
  python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29512 bench_pcm.py
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

import bench  # noqa: E402  (Ranks, percentiles, SR)

FORMATS = ("f32", "s16", "s24")
ESZ = {"f32": 4, "s16": 2, "s24": 3}
DTYPE = {"f32": np.float32, "s16": np.int16, "s24": np.uint8}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1, help="1, or the torchrun world size (one rank per GPU)")
    ap.add_argument("--streams", type=int, default=81920, help="streams per GPU")
    ap.add_argument("--block", type=int, default=512)
    ap.add_argument("--partitions", type=int, default=188)
    ap.add_argument("--steps", type=int, default=300, help="timed device steps per format (formats alternate)")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--feed-blocks", type=int, default=12, help="blocks per submit of the host feed")
    a = ap.parse_args()
    if a.steps < 1 or a.streams < 1:
        ap.error("--steps and --streams must be >= 1")
    return a


def card(local):
    """(name, power limit in W) of this rank's GPU, by PCI address"""
    import torch
    pr = torch.cuda.get_device_properties(local)
    bus = "%08x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
    try:
        out = subprocess.run(["nvidia-smi", "-i", bus, "--query-gpu=name,power.limit", "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout
        name, watts = [v.strip() for v in out.strip().split(",")[:2]]
        return name, float(watts)
    except Exception:
        return pr.name, None


def pcm_block(rng, shape, fmt):
    """random block array at half full scale in format fmt (S24: uint8 with a last axis of 3*B)"""
    if fmt == "f32":
        return ((rng.random(shape, dtype=np.float32) * 2 - 1) * 0.5).astype(np.float32)
    top = 1 << (15 if fmt == "s16" else 23)
    q = rng.integers(-top // 2, top // 2, size=shape, dtype=np.int32)
    if fmt == "s16":
        return q.astype(np.int16)
    b = (q.astype(np.int64) & 0xFFFFFF)
    return np.stack([b & 0xFF, (b >> 8) & 0xFF, (b >> 16) & 0xFF], -1).astype(np.uint8).reshape(shape[:-1] + (3 * shape[-1],))


def device_steps(a, R, eng, e, S, B):
    """block step p50 / p99 per format through process_device_pcm, the formats alternating step by step"""
    import torch
    K = 4
    buf = {}
    for f in FORMATS:
        din = torch.empty(K * S * B * ESZ[f], dtype=torch.uint8, device="cuda")
        din.copy_(torch.from_numpy(pcm_block(np.random.default_rng(7 + ESZ[f]), (K, S, B), f).view(np.uint8).reshape(-1)))
        buf[f] = (din, torch.empty(K * S * B * ESZ[f], dtype=torch.uint8, device="cuda"))
    torch.cuda.synchronize()

    def step(i, f):
        din, dout = buf[f]
        off = (i % K) * S * B * ESZ[f]
        e.process_device(din.data_ptr() + off, dout.data_ptr() + off, 1, in_format=f, out_format=f)

    for i in range(a.warmup):
        for f in FORMATS:
            step(i, f)
    e.synchronize()
    R.barrier()
    e.set_timing(True)
    for i in range(a.steps):
        for f in FORMATS:
            step(i, f)
    e.synchronize()
    ms, _ = e.timings()
    e.set_timing(False)
    out = {}
    for k, f in enumerate(FORMATS):
        s = ms[k::len(FORMATS)]
        out[f] = {"p50_ms": float(np.percentile(s, 50)), "p99_ms": float(np.percentile(s, 99)), "steps": int(len(s))}
    del buf
    torch.cuda.empty_cache()
    return out


def host_legs(a, R, eng, e, S, B, period_ms, tile, f):
    """continuous feed, block-by-block real-time stream count and copy-only ceiling of format f (the method of bench.e2e_leg)"""
    K2 = max(4, min(a.feed_blocks, (2 << 30) // (S * B * 4)))
    ishape = (K2, S, B * (3 if f == "s24" else 1))
    hin = eng.pinned_empty(ishape, DTYPE[f])
    hout = eng.pinned_empty(ishape, DTYPE[f])
    hin[:] = pcm_block(np.random.default_rng(1003 + R.rank), (K2, S, B), f)
    e.set_stream(None)
    e.process(hin[:4], hout[:4], out_format=f)
    R.barrier()
    REP = 4
    t0 = time.perf_counter()
    for _ in range(REP):
        e.submit(hin, hout, out_format=f)
    e.wait()
    dt = R.max((time.perf_counter() - t0) / REP)
    blk_bytes = S * B * ESZ[f]
    res = {"feed_channels": R.world * S * B * K2 / dt / bench.SR, "ms_per_step": 1e3 * dt / K2, "bytes_per_block_each_way": blk_bytes,
           "feed_used_gbs": R.world * 2 * blk_bytes / (dt / K2) / 1e9}
    nb1 = min(K2, 16)

    def roundtrip_at(n):
        e.set_active_channels(n)
        w = hin.shape[-1]
        x = hin.reshape(-1)[:nb1 * n * w].reshape(nb1, n, w)
        y = hout.reshape(-1)[:nb1 * n * w].reshape(nb1, n, w)
        e.process(x[0], y[0], out_format=f)
        R.barrier()
        ts = []
        for i in range(nb1):
            t0 = time.perf_counter()
            e.process(x[i], y[i], out_format=f)
            ts.append(time.perf_counter() - t0)
        return R.max(float(np.max(ts[1:]))) * 1e3

    rt_S, trail = 0, []
    ms = roundtrip_at(S)
    trail.append({"streams": S, "roundtrip_max_ms": ms})
    if ms < period_ms * 0.97:
        rt_S = S
    else:
        cand = int(S * period_ms / ms * 0.97) // 2048 * 2048
        for _ in range(6):
            cand = max(tile, min(cand, S)) // tile * tile
            ms = roundtrip_at(cand)
            trail.append({"streams": cand, "roundtrip_max_ms": ms})
            if ms < period_ms:
                rt_S = cand
                break
            cand = int(cand * min(0.95, period_ms / ms * 0.98)) // 2048 * 2048
    e.set_active_channels(S)
    res.update({"rt_streams_per_gpu": rt_S, "rt_streams_search": trail})
    eng.pinned_free(hin)
    eng.pinned_free(hout)
    try:
        probe = eng.CopyProbe(blk_bytes, 0, device=R.local)
        probe.run(2, 3)
        R.barrier()
        secs = R.max(probe.run(8, 3))
        probe.close()
        ceil = R.world * blk_bytes * 8 * 2 / secs / 1e9
        res.update({"copy_ceiling_gbs": ceil, "copy_ceiling_channels": ceil * 1e9 / (2 * ESZ[f] * bench.SR),
                    "frac_of_copy_ceiling": res["feed_used_gbs"] / ceil})
    except Exception as ex:
        res["copy_ceiling_gbs"] = None
        res["copy_note"] = "probe failed: %s" % ex
    return res


def main():
    a = parse()
    R = bench.Ranks()
    if R.world != a.gpus and not (a.gpus == 1 and R.world == 1):
        raise SystemExit("bench_pcm.py: --gpus %d but %d rank(s) running" % (a.gpus, R.world))
    from irbaboon_b200 import engine as eng
    from irbaboon_b200 import synth
    S, B, P = a.streams, a.block, a.partitions
    period_ms = 1e3 * B / bench.SR
    name, watts = card(R.local)
    e = eng.Engine(B, P, S, 1, device=R.local)
    e.set_ir(0, synth.decaying_ir(4242, P * B))
    tile = e.tile_channels
    dev = device_steps(a, R, eng, e, S, B)
    res = {"bench": "bench_pcm", "card": name, "power_limit_w": watts, "gpus": R.world, "streams_per_gpu": S, "block": B, "partitions": P,
           "block_period_ms": period_ms, "formats": {}}
    for f in FORMATS:
        r = {"device_step": dev[f]}
        r.update(host_legs(a, R, eng, e, S, B, period_ms, tile, f))
        res["formats"]["%s/%s" % (f, f)] = r
    e.close()
    if R.rank == 0:
        print(json.dumps(res), flush=True)
    R.close()


if __name__ == "__main__":
    main()
