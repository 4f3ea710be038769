"""bench.py's contract.  CPU: the reference arm prints ONE JSON line with the agreed keys, the product arm refuses to run
without a CUDA device (no CPU fallback), arguments are checked and --dump-outputs samples a fixed set of rows.  GPU: the
dumped outputs repeat from run to run."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line(built):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-seconds", "2"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "channels" and d["higher_is_better"] is True and d["value"] > 0
    assert d["metric"].startswith("48kHz RT channels per B200")
    assert d["e2e"] == {"value": d["value"], "unit": "channels", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["config"]["block"] == 512 and d["config"]["partitions"] == 188 and d["gpu_launches"] == 0


def test_product_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode != 0 and "no CPU fallback" in (p.stderr + p.stdout)


# ---- the capacity ladder (SURVEY 8d channels_RT) as a pure function ----------------------------------------------
def _bench_module():
    import importlib.util
    spec = importlib.util.spec_from_file_location("irb_bench", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def _fake_gpu(ms_per_stream, fixed_ms, slow_every=0, slow_ms=2.2, seed=0):
    """p99_at of a GPU whose step time is linear in the stream count, with an isolated slow step every `slow_every` steps."""
    import numpy as np
    calls = []
    rng = np.random.default_rng(seed)

    def p99_at(streams, steps):
        t = fixed_ms + ms_per_stream * streams + rng.normal(0, 0.003, steps)
        if slow_every:
            t[rng.integers(0, slow_every, 1)[0]::slow_every] += slow_ms
        calls.append((streams, steps))
        return float(np.percentile(t, 99)), float(np.percentile(t, 50))
    return p99_at, calls


def test_capacity_ladder_finds_the_largest_real_time_rung():
    b = _bench_module()
    period = 1e3 * 512 / 48000.0
    # 7.1 TB/s-like device: 0.1105 us per stream -> 96.5 k streams fit the period exactly
    p99_at, calls = _fake_gpu(1.105e-4, 0.0)
    S, log, failed = b.capacity_search(p99_at, 98304, period, 300)
    assert not failed and S % 2048 == 0 and S == 94208                       # 96 256 would need 10.64 ms + margin: the first rung below the 2 % guard
    assert calls[0] == (98304, 40) and all(c[1] == 300 for c in calls[1:]) and log[-1]["realtime"]
    # everything resident already runs in real time: verified at the full count, nothing above it is claimed
    p99_at, calls = _fake_gpu(0.9e-4, 0.0)
    S, log, failed = b.capacity_search(p99_at, 98304, period, 300)
    assert (S, failed) == (98304, False) and calls == [(98304, 40), (98304, 300)]
    # a rung that misses only on p99 is verified a second time before the search moves down (both attempts are in the trail)
    state = {"n": 0}
    def flaky(streams, steps):
        state["n"] += 1
        base = 1.105e-4 * streams
        return (base + (2.2 if state["n"] == 2 else 0.01), base)            # the first full verification catches stray slow steps
    S, log, failed = b.capacity_search(flaky, 98304, period, 300)
    assert (S, failed) == (94208, False) and [(r["streams"], r.get("attempt")) for r in log] == [(98304, None), (94208, 1), (94208, 2)]
    # isolated +2.2 ms steps, four in 300: the rungs near the limit fail on p99 and the search walks down rung by rung
    p99_at, calls = _fake_gpu(1.105e-4, 0.0, slow_every=70)
    S, log, failed = b.capacity_search(p99_at, 98304, period, 300)
    assert not failed and 2048 <= S <= 77824 and 1.105e-4 * S + 2.2 < period and [r["streams"] for r in log[1:]] == sorted((r["streams"] for r in log[1:]), reverse=True)


def test_capacity_ladder_never_aborts():
    b = _bench_module()
    period = 1e3 * 512 / 48000.0
    p99_at, calls = _fake_gpu(1.0e-4, 20.0)                                # a disturbed box: no stream count can be real-time
    S, log, failed = b.capacity_search(p99_at, 98304, period, 300)
    assert failed and S == 2048 and len(calls) <= 26                        # falls to the last rung and reports it as unverified
    p99_at, calls = _fake_gpu(4.0e-4, 0.0)                                 # a GPU four times slower: jumps to the estimate, then verifies
    S, log, failed = b.capacity_search(p99_at, 98304, period, 300)
    assert not failed and 22528 <= S <= 26624 and len(calls) <= 6


def test_bench_rejects_zero_steps_and_dumps_from_the_reference_arm():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert p.returncode == 2 and "error:" in p.stderr, (extra, p.stderr[-2000:])


def test_dump_rows_fixed_sample_within_budget():
    import numpy as np
    b = _bench_module()
    assert np.array_equal(b.dump_rows(8192, 4096), np.arange(8192))                     # c4 at one GPU: 32 MB, every stream
    rows = b.dump_rows(98304, 2048)
    assert len(rows) * 2048 <= b.DUMP_BYTES < 64 << 20 and len(rows) == b.DUMP_BYTES // 2048
    assert np.all(np.diff(rows) > 0) and rows[-1] < 98304 and np.array_equal(rows, b.dump_rows(98304, 2048))
    # the capacity ladder keeps the sampled streams below the count it stopped at: two stops share the leading rows
    a, c = rows[rows < 94208], rows[rows < 92160]
    assert np.array_equal(a[:len(c)], c)
    assert len(b.dump_rows(256, 4 << 20)) == 12                                             # c5: 12 of 256 captures


@pytest.mark.gpu
def test_dumped_outputs_repeat_across_runs(tmp_path):
    """Two runs with the same arguments, capacity ladder included, time exactly --steps block steps and dump the same outputs."""
    import numpy as np
    args = ["--steps", "5", "--warmup", "2", "--streams-max", "4096", "--ladder-steps", "20", "--no-cpu-baseline", "--no-e2e", "--no-selfcheck"]
    outs = []
    for k in range(2):
        d = tmp_path / str(k)
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args + ["--dump-outputs", str(d)], capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert p.returncode == 0, p.stderr[-2000:]
        line = json.loads(p.stdout.strip().splitlines()[-1])
        assert line["steps"] == 5 and line["gpu_launches"] == 5
        y = np.load(d / "block_output.npy")
        assert y.dtype == np.float32 and y.shape == (line["config"]["streams_per_gpu"], 512)
        outs.append(y)
    n = min(len(outs[0]), len(outs[1]))
    assert n >= 2048 and np.isfinite(outs[0]).all() and np.abs(outs[0]).max() > 0
    assert np.array_equal(outs[0][:n], outs[1][:n])


def test_clock_sampler_degrades_without_a_gpu():
    """No NVML / no CUDA device (this container): the sampler constructs, starts, stops and reports that it saw nothing --
    the bench line then says so instead of inventing clocks."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    b = _bench_module()
    s = b.ClockSampler(0, 0.005)
    s.start()
    s.stop()
    out = s.summary()
    assert out["sm_mhz"] is None and out["reasons"] == ["no samples"] and s.near(0.0) is None
