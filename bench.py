#!/usr/bin/env python
"""bench.py -- headline benchmark of the partitioned-convolution hot path.

Workload (BASELINE.json configs[2], the configuration the metric is quoted on): S independent mono 48 kHz
streams sharing one 2 s synthetic IR (96 000 taps -> P = 188 partitions), block B = 512.  One STEP = one UPOLA
block step for all S streams of a rank: forward FFT of the new block into the frequency-domain delay line (FDL),
multiply-accumulate over all P partitions, inverse FFT, overlap-add -- ONE launch of the persistent kernel k_mac_p.

  value   real-time 48 kHz channels per GPU that THIS RUN VERIFIED (SURVEY 8d: channels_RT = max S with p99(block step) <
          B/48000): a short ladder finds the largest stream count whose p99 over >= 300 consecutive steps stays under the
          10.667 ms block period; the K timed steps then run at that count.  The throughput equivalent S*B/step/48000 is
          config.channel_samples_per_s / 48000.  With --streams S the ladder is skipped (value_kind says which).
  e2e     the same metric through irb_engine_submit/_wait: HOST (pinned) buffers, H2D and D2H inside the timed region;
          e2e.host_copy_ceiling_gbs is a copy-only probe of the same sizes on the same ranks (no kernels),
          e2e.rt_streams_per_gpu the largest stream count whose block-by-block host round trip stays inside the period
  roofline  the block-step kernel: algorithmic bytes (SURVEY 8d) / its CUDA-event duration vs the measured HBM peak
  cpu_baseline / --impl reference: the reference's own fp::convolution::convolvePeriodic (oracle/_ref, compiled
          unmodified) on the box's host cores, one whole stream per thread

Other workloads (their own metric names; not the headline): --workload c4 = BASELINE configs[3] (per-stream 10 s IRs,
block 1024, strong scaling over the ranks), --workload c5 = configs[4] (256 x 2^20-sample ESS captures deconvolved).

Launch: `python bench.py --gpus 1` or, for N > 1, under torchrun (one rank per GPU, streams sharded by rank,
no data-path collective; torch.distributed is used only for the barrier and the max-over-ranks time).

--dump-outputs DIR writes what the last timed step computed as float32 .npy files, so that two builds run with the same
arguments (same seeded inputs) can be compared output for output: c3 / c4 block_output.npy [streams, B], the output block
of every stream or, past 48 MB, of a fixed seeded sample of streams in ascending order; c5 impulse_responses.npy
[captures, 2^20] (impulse_responses_rank<r>.npy per rank, the 48 MB split between the ranks, so at most 12 ranks), likewise
sampled by capture.  Under the c3 capacity ladder the sample is drawn from every stream held resident and keeps those
that ran, so on one GPU two runs whose ladders stopped at different counts share the leading rows.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SR = 48000.0
METRIC = "48kHz RT channels per B200 (block 512, 2s IR)"
UNIT = "channels"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--streams", type=int, default=0, help="c3: fixed streams per GPU (skips the capacity ladder; configs[2] names 1024)")
    ap.add_argument("--streams-max", type=int, default=98304, help="c3: streams resident per GPU for the capacity ladder (0.77 MB of FDL each)")
    ap.add_argument("--ladder-steps", type=int, default=300, help="consecutive steps a stream count must hold p99 < block period for")
    ap.add_argument("--block", type=int, default=512)
    ap.add_argument("--ir-seconds", type=float, default=2.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-selfcheck", action="store_true", help="skip the post-run comparison with the two-launch form and the CPU reference")
    ap.add_argument("--e2e-steps", type=int, default=0, help="steps of the host-buffer leg (default: min(steps, 32))")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target wall time of the bounded CPU sample")
    ap.add_argument("--two-launch", action="store_true", help="block step as k_fwd + MAC kernel instead of the fused single launch (A/B measurement)")
    ap.add_argument("--tune", action="append", default=[], metavar="KNOB=VALUE",
                    help="launch-policy knob of the library (include/irb_b200_bench.h), e.g. mac_persistent=0 for the one-CTA-per-tile kernel")
    ap.add_argument("--workload", default="c3", choices=["c3", "c4", "c5"],
                    help="c3 (default, the headline line): streams sharing one IR.  c4: BASELINE configs[3], --streams-total streams with PER-STREAM "
                         "10 s IRs, block 1024, sharded by stream over the ranks (strong scaling).  c5: configs[4], batched ESS deconvolution")
    ap.add_argument("--streams-total", type=int, default=8192, help="c4: streams of the whole job")
    ap.add_argument("--captures", type=int, default=256, help="c5: captures per batch (per GPU)")
    ap.add_argument("--smoothing", action="store_true", help="c5: with the plug-in's default 3 x 1/13-octave smoothing (not the headline c5 line)")
    ap.add_argument("--sample-ms", type=float, default=20.0, help="period of the NVML clock / power sampler during the timed region")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy (float32, at most 48 MB)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs: the reference arm times the CPU code and keeps no outputs")
    if a.workload == "c4":
        a.block, a.ir_seconds = 1024, 10.0
    return a


# ---------------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock, board power and throttle reasons DURING the timed region, sampled through NVML every few milliseconds
    with host timestamps (so a slow step can be put next to the clock the GPU ran at); nvidia-smi as the fallback."""
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake_slowdown"}

    def __init__(self, index, period_s=0.005):
        self.index, self.period, self.rows, self.stop_flag, self.thread, self.proc = index, period_s, [], False, None, None
        self.h = None
        self.smi_id = str(index)
        bus = None
        try:                                                 # CUDA device `index` of this process by PCI address: NVML and nvidia-smi count
            import torch                                     # the physical GPUs, which differs under CUDA_VISIBLE_DEVICES
            pr = torch.cuda.get_device_properties(index)
            bus = "%08x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
            self.smi_id = bus
        except Exception:
            bus = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            try:
                self.h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode() if bus else b"")
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.h = None

    def start(self):
        if self.h is not None:
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
            "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", self.smi_id, "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read_smi, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _poll(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.rows.append((time.perf_counter(), float(mhz), float(pw), int(rs)))
            except Exception:
                pass
            time.sleep(self.period)

    def _read_smi(self):
        for line in self.proc.stdout:
            c = [v.strip() for v in line.split(",")]
            if len(c) < 9:
                continue
            try:
                bits = 0
                for bit, v in zip([0x8, 0x40, 0x20, 0x4], c[5:9]):
                    if v.lower().startswith("active"):
                        bits |= bit
                self.max_mhz = float(c[2])
                self.rows.append((time.perf_counter(), float(c[1]), float(c[3]), bits))
            except ValueError:
                continue

    def mark(self):
        return len(self.rows)

    def stop(self):
        self.stop_flag = True
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        if self.thread:
            self.thread.join(timeout=2)

    def summary(self, lo=0, hi=None):
        rows = self.rows[lo:hi]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        bits = 0
        for r in rows:
            bits |= r[3]
        return {"sm_mhz": float(np.median([r[1] for r in rows])), "sm_max_mhz": float(getattr(self, "max_mhz", 0.0)), "sm_mhz_min": float(min(r[1] for r in rows)),
                "power_w_max": float(max(r[2] for r in rows)), "power_w_median": float(np.median([r[2] for r in rows])), "samples": len(rows),
                "source": "nvml" if self.h is not None else "nvidia-smi", "reasons": sorted(n for b, n in self.REASONS.items() if bits & b)}

    def near(self, t):
        """(sm_mhz, power_w, reasons) of the sample closest to host time t"""
        if not self.rows:
            return None
        ts = np.array([r[0] for r in self.rows])
        r = self.rows[int(np.argmin(np.abs(ts - t)))]
        return {"sm_mhz": r[1], "power_w": r[2], "reasons": sorted(n for b, n in self.REASONS.items() if r[3] & b), "dt_ms": 1e3 * (r[0] - t)}


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


DUMP_BYTES = 48 << 20


def dump_rows(n_rows, row_bytes, budget=DUMP_BYTES):
    """Indices of the rows (streams or captures) --dump-outputs writes: all of them when they fit the budget, else a fixed
    seeded sample, ascending."""
    if n_rows * row_bytes <= budget:
        return np.arange(n_rows)
    return np.sort(np.random.default_rng(0).choice(n_rows, budget // row_bytes, replace=False))


def write_outputs(path, arrays):
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), np.ascontiguousarray(a, np.float32))


def workload(args):
    B = args.block
    Lh = int(round(args.ir_seconds * SR))
    P = int(np.ceil(np.float32(Lh) / np.float32(B)))
    return B, Lh, P


def metric_of(args):
    if args.workload == "c4":
        return "48kHz RT channels (block 1024, per-stream 10s IRs)", UNIT
    if args.workload == "c5":
        return "ESS IR captures deconvolved per second (2^20-sample sweep, batched)", "captures/s"
    return METRIC, UNIT


# ---------------------------------------------------------------------------------------------------------
def cpu_reference_sample(args, target_seconds, threads=None, probe=None):
    """The reference's own code (oracle/_ref; the C port if _ref did not travel) on the host cores, a bounded sample of the
    workload: convolvePeriodic with `threads` workers, one whole mono stream each, same IR / block size as the GPU workload
    (c3, c4), or deconvolve of 2^20-sample captures, one capture per thread (c5)."""
    import oracle
    from irbaboon_b200 import synth
    if args.workload == "c5":
        return cpu_reference_sample_c5(args, target_seconds, threads)
    B, Lh, P = workload(args)
    h = synth.decaying_ir(2000, Lh)
    if oracle.have_reference():
        ref = oracle.Reference()
        T = threads or max(1, ref.hardware_threads())
        if probe is None:
            secs, _ = ref.bench_convolve_periodic(T, T, int(SR // 4), h, B, 1003)          # probe: 0.25 s of audio per stream
            probe = max(secs, 1e-3) / 0.25
        per_audio_second = probe                                                            # wall seconds per audio second with T streams on T threads
        # T..8T streams of up to 10 s each: about target_seconds of wall time on all host threads
        audio_s = float(np.clip(target_seconds / per_audio_second, 0.5, 10.0))
        rounds = int(np.clip(target_seconds / (audio_s * per_audio_second), 1, 8))
        Lx = int(audio_s * SR) // B * B
        streams = T * rounds
        secs, chk = ref.bench_convolve_periodic(T, streams, Lx, h, B, 1003)
        kind = "reference"
    else:                                                                                   # scalar C port, 1 thread
        orc = oracle.Oracle()
        T, streams = 1, 1
        Lx = int(2 * SR) // B * B
        x = synth.white_noise(1003, 0, Lx)
        t0 = time.perf_counter()
        orc.convolve_periodic(x, h, B)
        secs, chk, kind = time.perf_counter() - t0, 0.0, "port"
    rt = streams * (Lx / SR) / secs
    return {"value": rt, "unit": UNIT, "cores": T, "kind": kind, "seconds": secs, "probe": probe,
            "sample": "%d streams x %.2f s white noise each through fp::convolution::convolvePeriodic(B=%d, %d-tap IR), %d threads, one stream per thread"
                      % (streams, Lx / SR, B, Lh, T)}


def c5_inputs(n_captures, n=1 << 20, seed=4000):
    """Synthetic ESS captures: the sweep convolved with short decaying IRs plus a little noise (numpy only: no GPU, no oracle)."""
    from irbaboon_b200 import synth
    t = np.arange(n, dtype=np.float64) / SR
    T = n / SR
    w1, w2 = 2 * np.pi * 20.0, 2 * np.pi * 24000.0 * 0.999
    sweep = np.sin(w1 * T / np.log(w2 / w1) * (np.exp(t / T * np.log(w2 / w1)) - 1.0)).astype(np.float32)
    S = np.fft.rfft(sweep.astype(np.float64), 2 * n)
    base = []
    for j in range(4):
        h = synth.decaying_ir(3000 + j, 48000, j).astype(np.float64)
        base.append(np.fft.irfft(S * np.fft.rfft(h, 2 * n), 2 * n)[:n].astype(np.float32))
    return sweep, base


def cpu_reference_sample_c5(args, target_seconds, threads=None):
    import oracle
    from irbaboon_b200 import synth
    n = 1 << 20
    sweep, base = c5_inputs(4)
    if oracle.have_reference():
        ref = oracle.Reference()
        T = threads or max(1, ref.hardware_threads())
        k = T
        caps = np.stack([base[j % 4] + synth.white_noise(4000 + j, 0, n) * np.float32(1e-3) for j in range(k)])
        secs, _ = ref.bench_deconvolve(T, caps, sweep, SR, False)
        kind = "reference"
    else:
        orc = oracle.Oracle()
        T, k = 1, 1
        t0 = time.perf_counter()
        orc.deconvolve(base[0], sweep, SR, False)
        secs, kind = time.perf_counter() - t0, "port"
    return {"value": k / secs, "unit": "captures/s", "cores": T, "kind": kind, "seconds": secs, "probe": None,
            "sample": "%d captures of 2^20 samples through fp::convolution::deconvolve(smoothing=false), %d threads, one capture per thread" % (k, T)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    metric, unit = metric_of(args)
    # every step is a bounded sample of the workload; the whole run (warm-up included) is sized for about two minutes
    budget = 120.0 / max(1, args.steps + args.warmup)
    per_step = float(np.clip(budget, 0.25, args.cpu_seconds))
    vals, last = [], None
    for i in range(args.warmup + args.steps):
        last = cpu_reference_sample(args, per_step, probe=last["probe"] if last else None)
        if i >= args.warmup:
            vals.append(last)
    secs = sum(v["seconds"] for v in vals)
    rt = float(np.mean([v["value"] for v in vals]))
    B, Lh, P = workload(args)
    wl = {"c3": "configs[2]: streams sharing one %.1f s IR, block %d" % (args.ir_seconds, B), "c4": "configs[3]: streams with per-stream %.0f s IRs, block %d" % (args.ir_seconds, B),
          "c5": "configs[4]: 2^20-sample ESS captures deconvolved by spectral division"}[args.workload]
    line = {"metric": metric, "value": rt, "unit": unit, "impl": "reference", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * secs / max(1, len(vals)), "higher_is_better": True, "scaling": "strong" if args.workload == "c4" else "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": {"workload": "%s (CPU: %s)" % (wl, last["sample"]), "block": B, "ir_taps": Lh, "partitions": P},
            "cpu_baseline": {"value": rt, "unit": unit, "cores": last["cores"], "kind": last["kind"], "sample": last["sample"]},
            "e2e": {"value": rt, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------
class Ranks:
    """torch.distributed plumbing: the launch barrier and max-over-ranks reductions; nothing on the data path."""

    def __init__(self):
        import torch
        self.torch = torch
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
        torch.cuda.set_device(self.local)
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            # NCCL announces its version on stdout when the communicator is created; stdout must carry one JSON line, so the
            # file descriptor points at stderr while the process group comes up (first barrier included)
            sys.stdout.flush()
            saved = os.dup(1)
            os.dup2(2, 1)
            try:
                dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
                dist.barrier()
                torch.cuda.synchronize()
            finally:
                sys.stdout.flush()
                os.dup2(saved, 1)
                os.close(saved)
            self.dist = dist

    def barrier(self):
        if self.dist:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max(self, v):
        from irbaboon_b200 import sharding
        return sharding.max_over_ranks(float(v), device="cuda")

    def close(self):
        if self.dist:
            self.dist.destroy_process_group()


def percentiles(ms, period):
    ms = np.asarray(ms, np.float64)
    return {"block_period_ms": period, "steps": int(len(ms)), "p50_ms": float(np.percentile(ms, 50)), "p99_ms": float(np.percentile(ms, 99)),
            "p999_ms": float(np.percentile(ms, 99.9)), "max_ms": float(ms.max()), "over_period": int((ms >= period).sum()),
            "realtime": bool(np.percentile(ms, 99) < period)}


def capacity_search(p99_at, s_alloc, period_ms, ladder_steps, quantum=2048, max_rungs=12):
    """SURVEY 8d channels_RT: the largest stream count (a multiple of `quantum`, at most s_alloc) whose p99 block step over
    `ladder_steps` consecutive steps stays under the block period.  p99_at(streams, steps) -> (p99_ms, p50_ms), already reduced
    over the ranks (every rank walks the same rungs).  A 40-step probe at everything resident gives the first rung; a failed rung
    is verified once more when only its p99 missed (a stray slow step), then steps one quantum down, or straight to the estimate
    when even the MEDIAN step is over the period.  -> (streams, trail, failed): failed = no rung held (then `streams` is the last rung tried)."""
    log = []
    p99, p50 = p99_at(s_alloc, 40)
    log.append({"streams": s_alloc, "steps": 40, "p50_ms": p50, "p99_ms": p99})
    cand = s_alloc if p99 < period_ms else int(s_alloc * period_ms / (p50 * 1.02)) // quantum * quantum
    for _ in range(max_rungs):
        cand = max(quantum, min(cand, s_alloc))
        for attempt in (1, 2):
            p99, p50 = p99_at(cand, ladder_steps)
            ok = p99 < period_ms
            log.append({"streams": cand, "steps": ladder_steps, "attempt": attempt, "p50_ms": p50, "p99_ms": p99, "realtime": bool(ok)})
            # Isolated slow steps (memory-side stalls, 0.4 - 0.6 % of steps) make the p99 of 300 samples noisy, the more so as every
            # rank must pass: a rung whose MEDIAN is inside the period gets one more full verification before the search moves down.
            if ok or p50 >= period_ms:
                break
        if ok:
            return cand, log, False
        if cand <= quantum:
            break
        cand = min(cand - quantum, int(cand * period_ms / (p50 * 1.02)) // quantum * quantum) if p50 >= period_ms else cand - quantum
    return max(quantum, min(cand, s_alloc)), log, True


def run_b200(args):
    from irbaboon_b200 import engine as eng
    for kv in args.tune:
        k, v = kv.split("=")
        eng.set_tuning(k, int(v))
    R = Ranks()
    if args.workload == "c5":
        return run_c5(args, R, eng)
    torch = R.torch
    from irbaboon_b200 import sharding, synth
    rank, world, local = R.rank, R.world, R.local

    B, Lh, P = workload(args)
    period_ms = 1e3 * B / SR
    per_stream_ir = args.workload == "c4"
    ladder = not per_stream_ir and args.streams <= 0
    if per_stream_ir:                                  # strong scaling: the job's streams are cut into contiguous ranges
        lo, hi = sharding.stream_range(rank, world, args.streams_total)
        S_alloc = hi - lo
    else:
        lo = 0
        S_alloc = args.streams_max if ladder else args.streams
    bins = B + 1
    if per_stream_ir:
        e = eng.Engine(B, P, S_alloc, S_alloc, device=local)
        irs = [synth.decaying_ir(2000 + j, Lh, j) for j in range(8)]          # 8 distinct IRs cycled: every stream still owns its spectra
        for s_ in range(S_alloc):
            e.set_ir(s_, irs[(lo + s_) % 8])
            e.bind(s_, s_ + 1, s_)
    else:
        h = synth.decaying_ir(2000, Lh)
        e = eng.Engine(B, P, S_alloc, 1, device=local)
        e.set_ir(0, h)
    if args.two_launch:
        e.set_fused_step(False)
    tile = e.tile_channels
    stream = torch.cuda.Stream()                       # the kernels and the timing events share this stream
    torch.cuda.set_stream(stream)
    e.set_stream(stream.cuda_stream)

    # synthetic input: NBUF distinct white-noise blocks per stream, resident in HBM, cycled step by step (a run at fewer active
    # streams reads the dense prefix of a buffer)
    NBUF = 4
    gen = torch.Generator(device="cuda").manual_seed(1003 + rank)
    d_in = (torch.rand((NBUF, S_alloc, B), device="cuda", generator=gen, dtype=torch.float32) * 2 - 1).contiguous()
    d_out = torch.empty((S_alloc, B), device="cuda", dtype=torch.float32)
    counter = [0]

    def step():
        e.process_device(d_in[counter[0] % NBUF].data_ptr(), d_out.data_ptr(), 1)
        counter[0] += 1

    def timed_steps(n):
        """n consecutive steps with per-step device timing; -> (step_ms, kernel_ms, host time the first one started)"""
        R.barrier()
        e.set_timing(True)
        t0 = time.perf_counter()
        for _ in range(n):
            step()
        sm_, mm_ = e.timings()
        e.set_timing(False)
        return sm_, mm_, t0

    # fill the FDL of every resident stream (steady state needs P blocks of history) + the requested warm-up
    for _ in range(max(args.warmup, 3) + P):
        step()
    R.barrier()

    sampler = ClockSampler(local, args.sample_ms * 1e-3)
    if rank == 0:
        sampler.start()
        time.sleep(0.05)

    # ---- capacity ladder (c3): the largest stream count whose p99 block step over ladder_steps stays inside the period ----
    S = S_alloc
    ladder_log = []
    ladder_failed = False
    if ladder:
        def p99_at(n_streams, n_steps):
            e.set_active_channels(n_streams)
            for _ in range(3):
                step()
            sm_, _, _ = timed_steps(n_steps)
            return R.max(np.percentile(sm_, 99)), R.max(np.percentile(sm_, 50))
        S, ladder_log, ladder_failed = capacity_search(p99_at, S_alloc, period_ms, args.ladder_steps)
        e.set_active_channels(S)
        # the rungs leave each stream's history and the input cycle wherever the search stopped: start again from silence
        # and refill the FDL, so that the timed steps compute the same outputs on every run with these arguments
        e.reset()
        counter[0] = 0
        for _ in range(P):
            step()
    for _ in range(3):
        step()

    # ---- the timed region of the contract: K steps, barrier + synchronize on both sides, CUDA events, max over ranks ----
    launches0 = eng.launch_count()
    e.set_timing(True)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    R.barrier()
    mark0 = sampler.mark()
    t_host0 = time.perf_counter()
    ev0.record(stream)
    for _ in range(args.steps):
        step()
    ev1.record(stream)
    R.barrier()
    mark1 = sampler.mark()
    total_ms = ev0.elapsed_time(ev1)
    launches = eng.launch_count() - launches0
    step_ms, mac_ms = e.timings()
    e.set_timing(False)
    clocks = sampler.summary(mark0, mark1) if rank == 0 else None

    total_ms = R.max(total_ms)
    ms_per_step = total_ms / args.steps
    # final host-side gather of the last output block in global stream order (outside the timed region; the only
    # cross-rank data movement of the whole job)
    total_streams = args.streams_total if per_stream_ir else world * S
    gathered = sharding.gather_streams(d_out[:S].cpu().numpy(), total_streams, device="cuda")
    if args.dump_outputs and rank == 0:
        if ladder:                                     # stream c of rank r is row r*S + c of the gather when it ran (c < S)
            r, c = np.divmod(dump_rows(world * S_alloc, B * 4), S_alloc)
            rows = (r * S + c)[c < S]
        else:
            rows = dump_rows(total_streams, B * 4)
        write_outputs(args.dump_outputs, {"block_output": gathered[rows]})
    throughput_channels = total_streams * B / (ms_per_step * 1e-3) / SR
    lat = percentiles(step_ms, period_ms)
    lat["p99_ms"] = R.max(lat["p99_ms"])
    lat["realtime"] = bool(lat["p99_ms"] < period_ms)
    if ladder and not ladder_failed:
        value, value_kind = float(total_streams), "verified_rt_capacity: largest stream count of the ladder whose p99 over %d consecutive steps < %.3f ms, on every rank" % (args.ladder_steps, period_ms)
    elif lat["realtime"] and args.steps >= 100:
        value, value_kind = float(total_streams), "fixed stream count, real time over the %d timed steps (p99 < period)" % args.steps
    else:
        value, value_kind = throughput_channels, "throughput_equivalent S*B/step/48000 (%s: not a verified capacity)" % (
            "no rung of the capacity ladder held p99 under the period" if ladder_failed else "fixed stream count, too few steps or p99 over the period")
    # slow steps next to the clock / power the GPU ran at (rank 0): is an excursion a power-cap event?
    excursions = None
    if rank == 0 and len(step_ms):
        med = float(np.median(step_ms))
        idx = [int(i) for i in np.argsort(step_ms)[::-1][:3] if step_ms[i] > med + 0.5]
        starts = t_host0 + np.concatenate([[0.0], np.cumsum(step_ms[:-1])]) * 1e-3
        excursions = [{"step": i, "ms": float(step_ms[i]), "median_ms": med, "gpu": sampler.near(starts[i] + step_ms[i] * 5e-4)} for i in idx]

    # ---- roofline of the dominant kernel (SURVEY 8d): FDL read per stream + the shared IR once per GPU (c3) or every stream's own IR
    # spectra (c4); the fused step is the WHOLE block step: add the new spectrum's write and the audio in/out ----
    slots, split_in, cluster = e.mac_plan()
    fused = (not args.two_launch) and split_in == 1 and cluster == 1 and (not slots or (eng.get_tuning("mac_persistent") and e.fft_size // 2 >= 256))
    alg_bytes = 2 * S * P * bins * 8 if per_stream_ir else (S + 1) * P * bins * 8
    if fused:
        alg_bytes += S * (bins * 8 + 2 * B * 4)
    mac_avg_ms = float(np.mean(mac_ms)) if len(mac_ms) else float("nan")
    peak, peak_src = measured_peak_gbs()
    achieved = alg_bytes / (mac_avg_ms * 1e-3) / 1e9
    M = e.fft_size // 2
    persistent = fused and M >= 256 and eng.get_tuning("mac_persistent")
    if persistent:
        kname = "k_mac_p<%d,%s> (persistent, one launch per block step: forward FFT + TMA-streamed FDL/IR multiply-accumulate + inverse FFT + overlap-add)" % (M, "PERROW" if slots else "shared IR")
    elif slots:
        kname = "k_mac_slots<%d,INV> (per-stream-IR FDL multiply-accumulate + inverse FFT + overlap-add)" % M
    elif fused and M >= 256 and eng.get_tuning("mac_tma"):
        kname = "k_mac_tma<%d> (one CTA per tile, one launch per block step)" % M
    else:
        kname = ("k_mac<%d,INV,FUSE> (register-staged, one launch per block step)" if fused else "k_mac<%d,INV> (FDL multiply-accumulate + inverse FFT + overlap-add)") % M
    roof = {"bound": "hbm", "kernel": kname, "achieved": achieved, "peak": peak,
            "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src, "frac_of_nominal_8000": achieved / 8000.0,
            "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": mac_avg_ms, "kernel_share_of_step": mac_avg_ms / float(np.mean(step_ms)),
            "traffic": None}
    prof = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(prof):
        try:
            tj = json.load(open(prof))
            # the static ncu figure applies only to the very kernel and shape it was captured on (bytes scale with the stream count)
            if tj.get("block") == B and tj.get("partitions") == P and tj.get("kernel", "").split("<")[0] == kname.split("<")[0] and not per_stream_ir:
                roof["traffic"] = tj["dram_bytes_per_launch"] * S / tj["streams"]
                roof["traffic_source"] = "ncu --set full at %d streams (%s), scaled by stream count" % (tj["streams"], tj.get("file", "profiles/"))
        except Exception:
            pass

    # ---- e2e: host (pinned) buffers through irb_engine_submit / _wait, copies inside the timed region ----
    e2e = None
    if not args.no_e2e:
        e2e = e2e_leg(args, R, eng, e, S, B, total_streams, period_ms, per_stream_ir, tile)

    # ---- self-check after the timed region, at the bench's own size (the GPU full): (1) the block step as measured against its
    # two-launch form on EVERY channel, bit for bit; (2) random channels against the CPU reference (oracle/_ref) ----
    selfcheck = None
    if not args.no_selfcheck:
        selfcheck = self_check(args, R, eng, e, S, B, Lh, per_stream_ir, lo)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_reference_sample(args, args.cpu_seconds)
        cpu.pop("seconds", None)
        cpu.pop("probe", None)
    sampler.stop()

    ok = selfcheck is None or selfcheck["ok"]
    if rank == 0:
        metric, unit = metric_of(args)
        wl = ("configs[3]: %d streams with per-stream %.0f s IRs (%d taps, %d partitions), block %d, sharded by stream over %d GPU(s)"
              % (total_streams, args.ir_seconds, Lh, P, B, world)) if per_stream_ir else \
             ("configs[2] shape: %d independent mono streams per GPU sharing one %.1f s IR (%d taps, %d partitions), block %d" % (S, args.ir_seconds, Lh, P, B))
        line = {"metric": metric, "value": value if ok else None, "unit": unit, "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
                "higher_is_better": True, "scaling": "strong" if per_stream_ir else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": wl, "value_kind": value_kind,
                           "streams_per_gpu": S, "streams_resident_per_gpu": S_alloc, "block": B, "ir_taps": Lh, "partitions": P, "fft_size": e.fft_size,
                           "state_bytes_per_gpu": int(e.state_bytes), "l2_policy": "inputs larger than L2 (FDL %.2f GB per GPU in use)" % (S * P * B * 8 / 1e9),
                           "mac_plan": [bool(slots), split_in, cluster], "tuning": args.tune,
                           "sharding": "contiguous stream ranges by rank, IR replicated, no data-path collective; host gather of outputs",
                           "gathered_output_shape": list(gathered.shape), "channel_samples_per_s": throughput_channels * SR,
                           "throughput_equivalent_channels": throughput_channels, "capacity_ladder": ladder_log},
                "latency": lat, "excursions": excursions, "roofline": roof, "cpu_baseline": cpu, "e2e": e2e, "selfcheck": selfcheck, "gpu_launches": int(launches), "clocks": clocks}
        if not ok:
            line["invalid"] = "selfcheck failed: the measured block step does not reproduce its two-launch form / the CPU reference"
        print(json.dumps(line), flush=True)
    e.close()
    R.close()
    if not ok:
        sys.exit(3)


def e2e_leg(args, R, eng, e, S, B, total_streams, period_ms, per_stream_ir, tile):
    """Host buffers in and out: continuous feed (submit/wait pipeline), block-by-block round trip, the copy-only ceiling of the
    same sizes on the same ranks, and the largest stream count whose block-by-block round trip stays inside the block period."""
    rank, world = R.rank, R.world
    K2 = args.e2e_steps or min(args.steps, 32)
    K2 = max(4, min(K2, (2 << 30) // (S * B * 4)))          # at most ~2 GB of pinned host memory per direction
    if per_stream_ir:
        K2 = min(K2, 8)
    hin = eng.pinned_empty((K2, S, B))
    hout = eng.pinned_empty((K2, S, B))
    rng = np.random.default_rng(1003 + rank)
    hin[:] = rng.random((K2, S, B), dtype=np.float32) * 2 - 1
    e.set_stream(None)
    e.process(hin[:4], hout[:4])                      # warm-up of the copy path
    R.barrier()
    REP = 4                                           # the feed is continuous: REP back-to-back submissions of K2 blocks, one wait
    t0 = time.perf_counter()
    for _ in range(REP):
        e.submit(hin, hout)                           # copies and kernels enqueued; the pipeline stays full across submissions
    e.wait()                                          # every output block is back on the host
    dt = (time.perf_counter() - t0) / REP
    dt = R.max(dt)
    # strict block-by-block round trip (what a live host callback sees)
    nb1 = min(K2, 16)
    R.barrier()
    rts = []
    for i in range(nb1):
        t0 = time.perf_counter()
        e.process(hin[i], hout[i])
        rts.append(time.perf_counter() - t0)
    dt1 = R.max(float(np.mean(rts)))
    checksum = float(np.abs(hout[nb1 - 1]).sum())
    blk_bytes = S * B * 4
    out = {"value": total_streams * B * K2 / dt / SR, "unit": UNIT, "h2d_bytes_per_step": blk_bytes, "d2h_bytes_per_step": blk_bytes,
           "steps": K2, "ms_per_step": 1e3 * dt / K2, "api": "%d x irb_engine_submit(host in, host out, n_blocks=%d) + irb_engine_wait, pinned buffers, wall clock" % (REP, K2),
           "blockwise_roundtrip_ms": 1e3 * dt1, "blockwise_realtime": bool(1e3 * dt1 < period_ms), "checksum": checksum}
    # ---- largest stream count whose block-by-block host round trip stays inside the period at this number of ranks ----
    if not per_stream_ir:
        def roundtrip_at(n):
            e.set_active_channels(n)
            x, y = hin.reshape(-1)[:nb1 * n * B].reshape(nb1, n, B), hout.reshape(-1)[:nb1 * n * B].reshape(nb1, n, B)
            e.process(x[0], y[0])
            R.barrier()
            ts = []
            for i in range(nb1):
                t0 = time.perf_counter()
                e.process(x[i], y[i])
                ts.append(time.perf_counter() - t0)
            return R.max(float(np.max(ts[1:]))) * 1e3
        rt_S, trail = 0, []
        if 1e3 * dt1 < period_ms * 0.97:
            rt_S = S
            trail.append({"streams": S, "roundtrip_ms": 1e3 * dt1})
        else:
            cand = int(S * period_ms / (1e3 * dt1) * 0.97) // 2048 * 2048
            for _ in range(6):
                cand = max(tile, min(cand, S)) // tile * tile
                ms = roundtrip_at(cand)
                trail.append({"streams": cand, "roundtrip_max_ms": ms})
                if ms < period_ms:
                    rt_S = cand
                    break
                cand = int(cand * min(0.95, period_ms / ms * 0.98)) // 2048 * 2048
            e.set_active_channels(S)
        out["rt_streams_per_gpu"] = rt_S
        out["rt_streams_search"] = trail
        out["rt_streams_note"] = "largest stream count per GPU whose one-block-per-call host round trip (irb_engine_process, copies included) stays under the %.3f ms period with all %d ranks running" % (period_ms, world)
    # ---- the same continuous feed with the INPUT in write-combined pinned memory (the host only writes it) ----
    try:
        hwc = eng.pinned_empty((K2, S, B), write_combined=True)
        hwc[:] = hin
        e.process(hwc[:4], hout[:4])
        R.barrier()
        t0 = time.perf_counter()
        for _ in range(REP):
            e.submit(hwc, hout)
        e.wait()
        dtw = R.max((time.perf_counter() - t0) / REP)
        out["write_combined_input"] = {"value": total_streams * B * K2 / dtw / SR, "ms_per_step": 1e3 * dtw / K2}
        eng.pinned_free(hwc)
        del hwc
    except Exception as ex:
        out["write_combined_input"] = {"error": str(ex)}
    eng.pinned_free(hin)
    eng.pinned_free(hout)
    del hin, hout
    # ---- copy-only ceiling: the same bytes per block, H2D and D2H at once, on every rank at the same time, no kernels ----
    try:
        probe = eng.CopyProbe(blk_bytes, 0, device=R.local)
        probe.run(2, 3)
        res = {}
        for name, direction in (("h2d", 1), ("d2h", 2), ("both", 3)):
            R.barrier()
            secs = R.max(probe.run(8, direction))
            res[name] = world * blk_bytes * 8 * (2 if direction == 3 else 1) / secs / 1e9
        probe.close()
        used = world * 2 * blk_bytes / (dt / K2) / 1e9
        out.update({"host_copy_ceiling_gbs": res["both"], "host_copy_h2d_only_gbs": res["h2d"], "host_copy_d2h_only_gbs": res["d2h"],
                    "host_copy_used_gbs": used, "frac_of_copy_ceiling": used / res["both"],
                    "host_copy_note": "aggregate over %d rank(s): %d-byte pinned transfers per direction and block, both directions at once, no kernels; "
                                      "the submit/wait leg moves the same bytes per step" % (world, blk_bytes)})
    except Exception as ex:                               # the probe is an aid: never fail the bench for it
        out["host_copy_ceiling_gbs"] = None
        out["host_copy_note"] = "probe failed: %s" % ex
    return out


def self_check(args, R, eng, e, S, B, Lh, per_stream_ir, lo):
    from irbaboon_b200 import synth
    KC = 4
    rng = np.random.default_rng(77 + R.rank)
    xin = (rng.random((KC, S, B), dtype=np.float32) * 2 - 1).astype(np.float32)
    e.set_stream(None)
    e.reset()
    ya = e.process(xin).copy()
    e.reset()
    e.set_fused_step(bool(args.two_launch))             # the other form of the block step
    yb = e.process(xin).copy()
    e.set_fused_step(not args.two_launch)
    out = {"blocks": KC, "channels_compared": int(S), "against": "fused step" if args.two_launch else "two-launch step (k_fwd, then the MAC kernel)",
           "bit_identical": bool(np.array_equal(ya, yb))}
    # random channels against the reference's own convolvePeriodic on the same input (first KC blocks from a reset engine)
    worst, n_ref, kind = 0.0, 0, None
    try:
        import oracle
        ref = oracle.Reference() if oracle.have_reference() else oracle.Oracle()
        kind = "oracle/_ref (reference object code)" if oracle.have_reference() else "oracle port"
        chans = sorted(set(int(c) for c in np.random.default_rng(5).integers(0, S, 8)) | {0, S - 1})
        irs = [synth.decaying_ir(2000 + j, Lh, j) for j in range(8)] if per_stream_ir else None
        for c in chans:
            h = irs[(lo + c) % 8] if per_stream_ir else synth.decaying_ir(2000, Lh)
            x = np.ascontiguousarray(xin[:, c, :]).reshape(-1)
            want = ref.convolve_periodic(x, h, B)[0, :KC * B]
            got = ya[:, c, :].reshape(-1)
            fs = max(1.0, float(np.abs(want).max()))
            worst = max(worst, float(np.abs(got - want).max()) / fs)
            n_ref += 1
    except Exception as ex:
        kind = "unavailable: %s" % ex
    out.update({"reference_channels": n_ref, "reference": kind, "max_abs_over_full_scale": worst, "tolerance": 1e-5, "reference_ok": bool(n_ref == 0 or worst <= 1e-5)})
    good = out["bit_identical"] and out["reference_ok"]
    out["ok"] = R.max(0.0 if good else 1.0) == 0.0      # every rank
    return out


# ---------------------------------------------------------------------------------------------------------
def run_c5(args, R, eng):
    """BASELINE configs[4]: a batch of 2^20-sample ESS captures deconvolved by spectral division (fp::convolution::deconvolve,
    smoothing off).  A step = one irb_deconvolve_batch call over the rank's batch.  value: captures/s from the CUDA-event time
    of the call's kernels (host<->device copies excluded); e2e: wall clock around the call, pinned host buffers in and out."""
    from irbaboon_b200 import synth
    torch = R.torch
    n, nb = 1 << 20, args.captures
    if args.dump_outputs and DUMP_BYTES // R.world < n * 4:
        raise SystemExit("bench.py: --dump-outputs fits one 2^20-sample capture per rank for at most %d ranks" % (DUMP_BYTES // (n * 4)))
    eng.set_device(R.local)
    sweep, base = c5_inputs(4)
    caps = eng.pinned_empty((nb, n))
    res = eng.pinned_empty((nb, n))
    for j in range(nb):
        caps[j] = base[j % 4] + synth.white_noise(4000 + j + 100000 * R.rank, 0, n) * np.float32(1e-3)
    d_caps = torch.from_numpy(np.asarray(caps)).cuda()
    d_res = torch.empty_like(d_caps)
    for _ in range(max(3, args.warmup)):
        eng.deconvolve_batch_device(d_caps.data_ptr(), nb, n, sweep, d_res.data_ptr(), SR, args.smoothing)
    sampler = ClockSampler(R.local, args.sample_ms * 1e-3)
    if R.rank == 0:
        sampler.start()
    R.barrier()
    launches0 = eng.launch_count()
    dev_ms, wall = [], []
    t_all = time.perf_counter()
    for _ in range(args.steps):                            # captures and results resident in HBM
        eng.deconvolve_batch_device(d_caps.data_ptr(), nb, n, sweep, d_res.data_ptr(), SR, args.smoothing)
        dev_ms.append(eng.last_compute_ms())
    R.barrier()
    t_all = R.max(time.perf_counter() - t_all)
    launches = eng.launch_count() - launches0
    clocks = sampler.summary() if R.rank == 0 else None
    sampler.stop()
    res_dev = d_res.cpu().numpy()
    if args.dump_outputs:                                  # every rank deconvolves its own batch
        rows = dump_rows(nb, n * 4, DUMP_BYTES // R.world)
        write_outputs(args.dump_outputs, {"impulse_responses" + ("_rank%d" % R.rank if R.world > 1 else ""): res_dev[rows]})
    for _ in range(2):                                     # e2e: pinned host captures in, pinned host IRs out
        eng.deconvolve_batch(caps, sweep, SR, args.smoothing, out=res)
    R.barrier()
    for _ in range(3):
        t0 = time.perf_counter()
        eng.deconvolve_batch(caps, sweep, SR, args.smoothing, out=res)
        wall.append(time.perf_counter() - t0)
    same_bits = bool(np.array_equal(res_dev, np.asarray(res)))
    dev = R.max(float(np.mean(dev_ms))) * 1e-3
    w = R.max(float(np.mean(wall)))
    total = nb * R.world
    peak, peak_src = measured_peak_gbs()
    alg = nb * 2 * n * 4                                  # SURVEY 8d: read the capture, write the IR (the sweep's spectrum is shared)
    three_pass = nb * 3 * 2 * (n // 2) * 8                # what the three-kernel scheme moves when nothing stays in L2
    # spot check against the reference on three captures of the batch
    chk = {"captures": [], "max_abs_over_full_scale": 0.0, "device_entry_equals_host_entry_bitwise": same_bits}
    try:
        import oracle
        ref = oracle.Reference() if oracle.have_reference() else oracle.Oracle()
        for j in sorted({0, nb // 2, nb - 1}):
            want = ref.deconvolve(np.array(caps[j]), sweep, SR, args.smoothing)[0]
            fs = max(1.0, float(np.abs(want).max()))
            chk["captures"].append(j)
            chk["max_abs_over_full_scale"] = max(chk["max_abs_over_full_scale"], float(np.abs(res[j] - want).max()) / fs)
            chk["relative_l2"] = max(chk.get("relative_l2", 0.0), float(np.linalg.norm(np.asarray(res[j], np.float64) - want) / np.linalg.norm(want)))
        chk["note"] = "relative L2 is reported, not gated: dividing by a sweep spectrum that falls to 2e-4 of its peak puts the reference itself 2e-5 from the float64 result (tests/test_gpu_fullsize.py calibrates the bound)"
        chk["ok"] = chk["max_abs_over_full_scale"] <= 1e-5 and same_bits
    except Exception as ex:
        chk["ok"], chk["note"] = same_bits, "reference unavailable: %s" % ex
    cpu = None
    if R.rank == 0 and R.world == 1 and not args.no_cpu_baseline:
        cpu = cpu_reference_sample(args, args.cpu_seconds)
        cpu.pop("seconds", None); cpu.pop("probe", None)
    ok = R.max(0.0 if chk["ok"] else 1.0) == 0.0
    if R.rank == 0:
        metric, unit = metric_of(args)
        line = {"metric": metric, "value": total / dev if ok else None, "unit": unit, "n_gpus": R.world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": 1e3 * t_all / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": "configs[4]: %d captures per GPU of a 2^20-sample exponential sine sweep (+ room IR, + noise) deconvolved by spectral division, N = 2^20" % nb,
                           "captures_per_gpu": nb, "fft_points": n, "smoothing": bool(args.smoothing), "value_kind": "irb_deconvolve_batch_device: captures and results resident in HBM, CUDA-event time of the whole call",
                           "l2_policy": "inputs larger than L2 (%.1f GB per batch)" % (nb * n * 4 / 1e9), "tuning": args.tune},
                "roofline": {"bound": "hbm", "kernel": ("k_line_fft / k_spec_* (transforms, split, divide, merge) + k_avg_passes (three log-average passes as a wavefront, one CTA per capture: "
                                                        "bound by the reference's sequential running sum and the per-bin rebuild arithmetic, not by HBM): the batch's device time as a whole") if args.smoothing else
                             "k_line_fft<512> (columns) + k_rowpair<1024> (rows, divide, inverse rows) + k_line_fft<512,INV>: the batch's kernel time as a whole",
                             "achieved": alg / dev / 1e9, "peak": peak, "unit": "GB/s", "frac": alg / dev / 1e9 / peak, "peak_source": peak_src,
                             "algorithmic_bytes_per_launch": alg, "kernel_ms": dev * 1e3, "three_pass_bytes": three_pass, "frac_at_three_pass_bytes": three_pass / dev / 1e9 / peak,
                             "traffic": None},
                "cpu_baseline": cpu,
                "e2e": {"value": total / w, "unit": unit, "h2d_bytes_per_step": nb * n * 4, "d2h_bytes_per_step": nb * n * 4, "ms_per_step": 1e3 * w,
                        "api": "irb_deconvolve_batch(pinned host captures, host sweep) -> pinned host IRs, wall clock, mean of 3 calls"},
                "selfcheck": chk, "gpu_launches": int(launches), "clocks": clocks}
        if not ok:
            line["invalid"] = "selfcheck failed"
        print(json.dumps(line), flush=True)
    eng.pinned_free(caps); eng.pinned_free(res)
    R.close()
    if not ok:
        sys.exit(3)


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
