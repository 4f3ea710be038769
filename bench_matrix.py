"""IR-matrix engine benchmark: mono -> stereo (1, 2) and true stereo (2, 2) against the plain engine on the duplicated inputs.

One JSON line per case on stdout (and appended to --out when given):
  shape, groups, B, P              the case; outputs = groups * outs
  matrix / plain                   block step p50 / p99 (CUDA events around every step, >= --steps steady-state steps) of the
                                   matrix engine and of the plain engine on the duplicated-input equivalent (outs * ins channels
                                   per group; for (2, 2) also with the sum of the two inputs' outputs on the device, "plain_sum")
  algorithmic bytes per step       P*(B+1)*8 of FDL per input row, the matrix IRs once per GPU (shared) or once per group
                                   (pergroup), (B+1)*8 per input row for the new spectrum, B*4 per input and per output row of
                                   audio; achieved GB/s = bytes / p50 step, and its fraction of the HBM copy peak measured in the
                                   same process (device-to-device copy, read + write bytes)
  ratio                            matrix p50 / plain p50 (plain_sum p50 for (2, 2))
With --capacity, the largest group count whose p99 over --ladder-steps consecutive steps stays under the block period (the
ladder rule of bench.py) for the matrix engine, and the largest channel count for the plain engine, in output channels.
The two engines run in the same process, alternating (--rounds), on device-resident buffers; the card name and its power limit
are recorded with the numbers.  Nothing is written to the source tree.
"""
import argparse
import json
import subprocess
import sys

import numpy as np

from bench import SR, capacity_search


def card():
    import torch

    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"], info["sm_clock_max_mhz"] = float(q[0]), float(q[1])
    except Exception as ex:                                     # the numbers stand without it, but say so
        info["power_limit_w"] = "unavailable: %s" % ex
    return info


def copy_peak_gbs(torch, nbytes=4 << 30, iters=10):
    a = torch.empty(nbytes // 4, device="cuda", dtype=torch.float32)
    b = torch.empty_like(a)
    b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    best = 0.0
    for _ in range(iters):
        e0.record(); b.copy_(a); e1.record(); e1.synchronize()
        best = max(best, 2 * nbytes / (e0.elapsed_time(e1) * 1e-3) / 1e9)
    del a, b
    torch.cuda.empty_cache()
    return best


def algo_bytes(B, P, n_in, n_out, ir_rows):
    """bytes a block step must move: FDL of every input row, the IR partitions it streams, the new spectrum, the audio"""
    spec = (B + 1) * 8
    return n_in * P * spec + ir_rows * P * spec + n_in * spec + (n_in + n_out) * B * 4


class Arm:
    """one engine with device-resident input / output blocks, timed step by step with CUDA events on its stream"""

    def __init__(self, torch, eng, B, P, G, ins, outs, pergroup, plain, irs):
        self.torch, self.plain, self.ins, self.outs, self.G = torch, plain, ins, outs, G
        terms = ins * outs
        n_mats = 8 if pergroup else 1
        if plain:
            # channel t*G + g is term t (input t // outs -> output t % outs) of group g: with one matrix every kernel tile shares
            # one IR (the headline kernel); with per-group matrices every channel stages its own IR
            self.n_in = self.n_out = G * terms
            self.e = eng.Engine(B, P, self.n_in, n_mats * terms)
            for j in range(n_mats * terms):
                self.e.set_ir(j, irs[j % len(irs)])
            for t in range(terms):
                if pergroup:
                    for g in range(G):
                        self.e.bind(t * G + g, t * G + g + 1, (g % n_mats) * terms + t)
                else:
                    self.e.bind(t * G, (t + 1) * G, t)
        else:
            self.n_in, self.n_out = G * ins, G * outs
            self.e = eng.MatrixEngine(B, P, G, ins, outs, n_mats * terms)
            for j in range(n_mats * terms):
                self.e.set_ir(j, irs[j % len(irs)])
            for g in range(G) if pergroup else []:
                self.e.bind_matrix(g, g + 1, [(g % n_mats) * terms + t for t in range(terms)])
        self.bytes = algo_bytes(B, P, self.n_in, self.n_out, (G if pergroup else 1) * terms)
        self.stream = torch.cuda.Stream()
        self.e.set_stream(self.stream.cuda_stream)
        gen = torch.Generator(device="cuda").manual_seed(7)
        self.x = torch.rand((self.n_in, B), device="cuda", generator=gen) * 2 - 1
        self.y = torch.empty((self.n_out, B), device="cuda")
        self.s = torch.empty((outs, G, B), device="cuda") if plain and ins > 1 else None

    def steps(self, n, with_sum=False):
        t = self.torch
        ev = [(t.cuda.Event(enable_timing=True), t.cuda.Event(enable_timing=True)) for _ in range(n)]
        with t.cuda.stream(self.stream):
            for a, b in ev:
                a.record()
                self.e.process_device(self.x.data_ptr(), self.y.data_ptr(), 1)
                if with_sum:                                  # out_o = in_0 * h_0o + in_1 * h_1o from the 4 duplicated channels
                    v = self.y.view(self.ins, self.outs, self.G, -1)
                    t.add(v[0], v[1], out=self.s)
                b.record()
        self.stream.synchronize()
        return np.array([a.elapsed_time(b) for a, b in ev])

    def close(self):
        self.e.close()
        self.x = self.y = self.s = None
        self.torch.cuda.empty_cache()


def stats(ms):
    return {"p50_ms": float(np.percentile(ms, 50)), "p99_ms": float(np.percentile(ms, 99)), "max_ms": float(ms.max()), "steps": int(len(ms))}


def run_case(torch, eng, args, ins, outs, pergroup, G, irs, peak):
    B, P = args.block, args.partitions
    m = Arm(torch, eng, B, P, G, ins, outs, pergroup, False, irs)
    p = Arm(torch, eng, B, P, G, ins, outs, pergroup, True, irs)
    two = ins > 1
    for arm in (m, p):
        arm.steps(args.warmup, with_sum=arm.plain and two)
    mm, pp, ps = [], [], []
    per = max(1, args.steps // args.rounds)
    for _ in range(args.rounds):                              # alternating, so drift of the card hits both alike
        mm.append(m.steps(per))
        pp.append(p.steps(per))
        if two:
            ps.append(p.steps(per, with_sum=True))
    mm, pp = np.concatenate(mm), np.concatenate(pp)
    rec = {"case": "%dx%d%s" % (ins, outs, "_pergroup" if pergroup else ""), "shape": [ins, outs], "pergroup": pergroup, "groups": G,
           "outputs": G * outs, "B": B, "P": P, "block_period_ms": 1e3 * B / SR,
           "matrix": dict(stats(mm), bytes_per_step=m.bytes, gbs=m.bytes / (np.percentile(mm, 50) * 1e-3) / 1e9),
           "plain": dict(stats(pp), channels=p.n_in, bytes_per_step=p.bytes, gbs=p.bytes / (np.percentile(pp, 50) * 1e-3) / 1e9)}
    rec["matrix"]["fraction_of_peak"] = rec["matrix"]["gbs"] / peak
    rec["plain"]["fraction_of_peak"] = rec["plain"]["gbs"] / peak
    base = rec["plain"]["p50_ms"]
    if two:
        ps = np.concatenate(ps)
        rec["plain_sum"] = stats(ps)
        base = rec["plain_sum"]["p50_ms"]
    rec["ratio_p50"] = rec["matrix"]["p50_ms"] / base
    rec["gbs_ratio_matrix_over_plain"] = rec["matrix"]["gbs"] / rec["plain"]["gbs"]
    m.close()
    p.close()
    return rec


def capacity(torch, eng, args, ins, outs, plain, irs):
    """largest output-channel count whose p99 step over --ladder-steps stays under the block period (bench.py's ladder rule);
    every rung builds its engine afresh (a matrix engine has no active-channel subset)"""
    B, P = args.block, args.partitions
    period = 1e3 * B / SR
    quantum = 2048 // outs                                    # in groups: 2048 output channels per rung

    def p99_at(groups, steps):
        a = Arm(torch, eng, B, P, groups, ins, outs, False, plain, irs)
        a.steps(20, with_sum=plain and ins > 1)
        ms = a.steps(steps, with_sum=plain and ins > 1)
        a.close()
        return float(np.percentile(ms, 99)), float(np.percentile(ms, 50))

    g_max = args.capacity_max_outputs // outs if not plain else args.capacity_max_outputs // 2      # the plain engine: bench.py's 98 304
    g, trail, failed = capacity_search(p99_at, g_max, period, args.ladder_steps, quantum=quantum)
    return {"output_channels": g * outs, "groups": g, "failed": failed, "trail": trail}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--block", type=int, default=512)
    ap.add_argument("--partitions", type=int, default=188)
    ap.add_argument("--outputs", type=str, default="16384", help="comma list of output-channel counts per case")
    ap.add_argument("--cases", type=str, default="1x2,2x2,1x2_pergroup,2x2_pergroup")
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=30)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--capacity", action="store_true", help="also run the real-time capacity ladder for 1x2 and the plain engine")
    ap.add_argument("--capacity-max-outputs", type=int, default=196608)
    ap.add_argument("--ladder-steps", type=int, default=300)
    ap.add_argument("--out", type=str, default="")
    args = ap.parse_args()
    if args.steps < 300 or args.rounds < 1:
        sys.exit("--steps must be >= 300 (the p99 needs them) and --rounds >= 1")
    import torch

    from irbaboon_b200 import engine as eng
    from irbaboon_b200 import synth

    if not torch.cuda.is_available():
        sys.exit("no GPU: bench_matrix.py measures on the device only")
    torch.cuda.set_device(0)
    gpu = card()
    peak = copy_peak_gbs(torch)
    try:
        commit = subprocess.run(["git", "rev-parse", "HEAD"], capture_output=True, text=True, timeout=10).stdout.strip() or None
    except Exception:
        commit = None
    irs = [synth.decaying_ir(5000 + j, args.block * args.partitions - 3 * j, j) for j in range(4)]
    lines = []

    def emit(rec):
        rec.update({"gpu": gpu, "copy_peak_gbs": peak, "commit": commit})
        s = json.dumps(rec)
        print(s, flush=True)
        lines.append(s)

    for outputs in [int(v) for v in args.outputs.split(",")]:
        for case in args.cases.split(","):
            ins, outs = (1, 2) if case.startswith("1x2") else (2, 2)
            emit(run_case(torch, eng, args, ins, outs, case.endswith("_pergroup"), outputs // outs, irs, peak))
    if args.capacity:
        emit({"case": "capacity", "B": args.block, "P": args.partitions, "ladder_steps": args.ladder_steps,
              "matrix_1x2": capacity(torch, eng, args, 1, 2, False, irs), "plain": capacity(torch, eng, args, 1, 1, True, irs)})
    if args.out:
        with open(args.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
