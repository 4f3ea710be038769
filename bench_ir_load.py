#!/usr/bin/env python
"""bench_ir_load.py -- loading many IRs into the streaming engine in one call (irb_engine_set_irs / _stage_irs) on one GPU.

load   the configs[3] (c4) load: 8 192 IRs of 480 000 taps at B = 1 024, 469 partitions, into an engine holding 8 192 IRs.
       loop_set_ir    one irb_engine_set_ir per IR (pageable host rows), as bench.py and bench_configs.py load them
       pinned / pageable   irb_engine_set_irs from host rows, 1 024 rows per call (8 calls: the host holds 2 GB of taps, not 16)
       device         irb_engine_set_irs from device-resident taps (a torch tensor [8192][480000]), one call
       Wall ms (host clock around calls that end synchronised).  Host paths: GB/s of taps uploaded, against the copy-only
       host-to-device ceiling of the same process (irbx_copy_probe: pinned memory, copies only; both host paths are set against it).  Device path: HBM GB/s at the byte
       model below.  The spectra of the set_irs paths are compared with the loop's on a sample of IRs (every partition).
stage  staging on a live c4 engine (8 192 streams, each with its own IR): stage_irs of all 8 192 IRs (8 calls of 1 024 rows)
       against the stage_ir loop, restaging the same partition count, then p50 / p99 of the following block steps (device
       events, device-resident I/O), which carry the round-robin refresh rows.
ab     the no-regression A/B against another tree (its own library and bench.py), alternating in --rounds rounds: one-IR set_ir
       latency at the configs[2] shape (96 000 taps, B = 512, one shared IR) and
       `bench.py --gpus 1 --steps 200 --warmup 20`.
Every line carries the card's name and power limit, read in the same run.

  python bench_ir_load.py [--what load,stage] [--out profiles/r08_bench_ir_load.jsonl]
  python bench_ir_load.py --what ab --ab-root PARENT_TREE [--rounds 2]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
B, LH, N_IR, ROWS = 1024, 480000, 8192, 1024


def card():
    import torch
    info = {"card": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        info["power_limit_w"] = q.stdout.strip()
    except Exception as ex:
        info["power_limit_w"] = "unavailable: %s" % ex
    return info


def byte_model(n, P, M, reps=1):
    """HBM bytes a device-source load moves: taps read once, every spectrum partition (ring included) written to every copy"""
    return n * LH * 4 + n * P * M * 8 * reps


def host_rows(eng, pinned):
    """ROWS distinct 480 000-tap rows; IR j of the load is row j % ROWS"""
    rng = np.random.default_rng(7)
    env = np.exp(-6.9 * np.arange(LH) / LH).astype(np.float32)
    a = eng.pinned_empty((ROWS, LH)) if pinned else np.empty((ROWS, LH), np.float32)
    for j in range(ROWS):
        a[j] = rng.standard_normal(LH).astype(np.float32) * env
    return a


def wall(fn):
    t0 = time.perf_counter()
    fn()
    return 1e3 * (time.perf_counter() - t0)


def load(eng, out):
    import torch
    P = int(np.ceil(np.float32(LH) / np.float32(B)))
    host = host_rows(eng, False)
    pin = eng.pinned_empty(host.shape)
    pin[:] = host
    gb = N_IR * LH * 4 / 1e9
    cp = eng.CopyProbe(1 << 30)                                      # pinned host memory, host-to-device only
    cp.run(2, 1)
    ceiling = (1 << 30) * 4 / cp.run(4, 1) / 1e9
    cp.close()
    pick = [0, 1, 1023, 1024, 4097, N_IR - 1]
    with eng.Engine(B, P, 8, N_IR) as e:
        M = e.fft_size // 2
        e.set_irs(range(ROWS), pin)                                  # warm-up: kernels, pool, staging
        t_loop = wall(lambda: [e.set_ir(j, host[j % ROWS]) for j in range(N_IR)])
        ref = np.stack([np.stack([e.ir_spectrum(i, p) for p in range(P)]) for i in pick])
        res = {}
        for name, src in (("pinned", pin), ("pageable", host)):
            res[name] = wall(lambda: [e.set_irs(range(c, c + ROWS), src) for c in range(0, N_IR, ROWS)])
            got = np.stack([np.stack([e.ir_spectrum(i, p) for p in range(P)]) for i in pick])
            res[name + "_same"] = bool(np.array_equal(got.view(np.uint32), ref.view(np.uint32)))
        d = torch.empty((N_IR, LH), dtype=torch.float32, device="cuda")
        hd = torch.from_numpy(host).cuda()
        for c in range(0, N_IR, ROWS):
            d[c:c + ROWS] = hd
        del hd
        torch.cuda.synchronize()
        e.set_irs(range(N_IR), d.data_ptr(), ld=LH)
        t_dev = min(wall(lambda: e.set_irs(range(N_IR), d.data_ptr(), ld=LH)) for _ in range(3))
        got = np.stack([np.stack([e.ir_spectrum(i, p) for p in range(P)]) for i in pick])
        same_dev = bool(np.array_equal(got.view(np.uint32), ref.view(np.uint32)))
        reps = e.ir_copies                                           # every copy of the spectra is written
        mb = byte_model(N_IR, P, M, reps)
        out.append({"bench": "ir_load", "shape": "c4 load: %d IRs x %d taps, B=%d, %d partitions" % (N_IR, LH, B, P), **card(),
                    "loop_set_ir_ms": t_loop,
                    "set_irs_pinned_ms": res["pinned"], "set_irs_pinned_gbps": gb / (res["pinned"] / 1e3),
                    "set_irs_pageable_ms": res["pageable"], "set_irs_pageable_gbps": gb / (res["pageable"] / 1e3),
                    "h2d_copy_ceiling_pinned_gbps": ceiling, "host_calls": N_IR // ROWS,
                    "set_irs_device_ms": t_dev, "device_byte_model_gb": mb / 1e9, "ir_copies": reps, "device_hbm_gbps": mb / 1e9 / (t_dev / 1e3),
                    "loop_gbps": gb / (t_loop / 1e3),
                    "spectra_equal_to_loop": {"pinned": res["pinned_same"], "pageable": res["pageable_same"], "device": same_dev}})
        print(json.dumps(out[-1]), flush=True)
        del d
    eng.pinned_free(pin)


def stage(eng, out, steps=40):
    import torch
    P = int(np.ceil(np.float32(LH) / np.float32(B)))
    host = host_rows(eng, True)
    e = eng.Engine(B, P, N_IR, N_IR)
    for s in range(N_IR):
        e.bind(s, s + 1, s)
    e.set_irs(range(ROWS), host)
    d_in = (torch.rand((2, N_IR, B), device="cuda") * 2 - 1).contiguous()
    d_out = torch.empty((N_IR, B), device="cuda")
    torch.cuda.synchronize()

    def steps_ms():
        e.set_timing(True)
        for i in range(steps):
            e.process_device(d_in[i % 2].data_ptr(), d_out.data_ptr(), 1)
        st, _ = e.timings()
        e.set_timing(False)
        return {"p50": float(np.percentile(st, 50)), "p99": float(np.percentile(st, 99))}

    t_first = wall(lambda: [e.stage_ir(j, host[j % ROWS]) for j in range(N_IR)])      # first staging: buffers allocated
    s0 = steps_ms()
    t_loop = wall(lambda: [e.stage_ir(j, host[j % ROWS]) for j in range(N_IR)])
    s_loop = steps_ms()
    t_batch = wall(lambda: [e.stage_irs(range(c, c + ROWS), host) for c in range(0, N_IR, ROWS)])
    s_batch = steps_ms()
    out.append({"bench": "ir_stage", "shape": "live c4 engine: %d streams with their own %d-tap IRs, B=%d, %d partitions, restaged" % (N_IR, LH, B, P),
                **card(), "first_stage_ir_loop_ms": t_first, "stage_ir_loop_ms": t_loop, "stage_irs_ms": t_batch, "host_calls": N_IR // ROWS,
                "steps_after_first_staging_ms": s0, "steps_after_stage_ir_loop_ms": s_loop, "steps_after_stage_irs_ms": s_batch})
    print(json.dumps(out[-1]), flush=True)
    e.close()
    eng.pinned_free(host)


def latency(reps=200):
    """one-IR set_ir latency at the configs[2] shape, in this process's library"""
    from irbaboon_b200 import engine as eng
    from irbaboon_b200 import synth
    Bc, Lc = 512, 96000
    h = synth.decaying_ir(2000, Lc)
    with eng.Engine(Bc, -(-Lc // Bc), 1024, 1) as e:
        for _ in range(20):
            e.set_ir(0, h)
        t = []
        for _ in range(reps):
            t0 = time.perf_counter()
            e.set_ir(0, h)
            t.append(1e3 * (time.perf_counter() - t0))
    print(json.dumps({"p50_ms": float(np.percentile(t, 50)), "p99_ms": float(np.percentile(t, 99)), "min_ms": float(min(t))}))


def ab(args, out):
    trees = {"this": ROOT, "parent": os.path.abspath(args.ab_root)}
    for r in range(args.rounds):
        for name, tree in trees.items():
            p = subprocess.run([sys.executable, os.path.abspath(__file__), "--what", "latency", "--tree", tree], capture_output=True, text=True)
            lat = json.loads(p.stdout.strip().splitlines()[-1]) if p.returncode == 0 else {"error": p.stderr[-2000:]}
            b = subprocess.run([sys.executable, os.path.join(tree, "bench.py"), "--gpus", "1", "--steps", "200", "--warmup", "20"], cwd=tree,
                               capture_output=True, text=True)
            lines = [ln for ln in b.stdout.splitlines() if ln.startswith("{")]
            bench = json.loads(lines[-1]) if b.returncode == 0 and lines else {"error": b.stderr[-2000:]}
            out.append({"bench": "ir_load_ab", "round": r, "tree": name, **card(), "set_ir_latency_c2_shape": lat, "bench_py": bench})
            print(json.dumps(out[-1]), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--what", default="load,stage")
    ap.add_argument("--out", default=None)
    ap.add_argument("--ab-root", default=None)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--tree", default=ROOT, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.what == "latency":
        sys.path.insert(0, args.tree)
        return latency()
    sys.path.insert(0, ROOT)
    from irbaboon_b200 import engine as eng
    out = []
    for w in args.what.split(","):
        {"load": lambda: load(eng, out), "stage": lambda: stage(eng, out), "ab": lambda: ab(args, out)}[w]()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            for ln in out:
                f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
