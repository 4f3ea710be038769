"""numpy statement of the batched IR chop (include/irb_b200.h, irb_ir_chop_batch_device), shared by the chop tests.

The walk is written the way the device computes it, as flags and a run-length scan: position j of the backward walk is
s_j = (q - j) mod n, loud_j := not (level(x[s_j]) - level(peak) < threshold), and walked = (the first j with j - (last loud
position <= j) >= consecutive) + 1, or ir_length when there is none.  tests/test_ir_chop_abi.py pins it to the facade's
sequential fp::ir::IRchop.  The levels come from tests/cpp/chop_rule.cpp: the facade's (glibc logf) or the device rule's."""
import ctypes
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_f32p = ctypes.POINTER(ctypes.c_float)


def build_helper(out_dir):
    """compile tests/cpp/chop_rule.cpp against the facade library (which must be built) into out_dir; -> ctypes.CDLL"""
    fp = os.path.join(ROOT, "irbaboon_b200", "fp")
    so = os.path.join(str(out_dir), "libchop_rule.so")
    subprocess.check_call(["g++", "-std=c++14", "-O2", "-fopenmp", "-fPIC", "-shared", "-o", so, os.path.join(ROOT, "tests", "cpp", "chop_rule.cpp"),
                           "-I" + fp, "-I" + os.path.join(ROOT, "include"), "-L" + fp, "-lfp_b200", "-L" + os.path.dirname(fp), "-lirb_b200",
                           "-Wl,-rpath," + fp, "-Wl,-rpath," + os.path.dirname(fp)])
    h = ctypes.CDLL(so)
    for name in ("chop_levels_facade", "chop_levels_rule"):
        getattr(h, name).argtypes = [_f32p, ctypes.c_longlong, _f32p]
    h.chop_ln10f.restype = h.chop_glibc_ln10f.restype = ctypes.c_float
    h.chop_log_sweep.argtypes = [ctypes.POINTER(ctypes.c_longlong), ctypes.POINTER(ctypes.c_uint32), ctypes.c_int]
    h.chop_find_level_flips.argtypes = [ctypes.c_uint32, _f32p, ctypes.c_int]
    h.chop_captures_to_irs.argtypes = [_f32p, ctypes.c_int, ctypes.c_int, _f32p, ctypes.c_int, ctypes.c_double, ctypes.c_int, ctypes.c_float, ctypes.c_int,
                                       ctypes.c_int, _f32p]
    return h


def levels(helper, x, rule):
    """dB levels of |x| (float32): the device rule (rule=True) or the facade's linTodB"""
    x = np.ascontiguousarray(x, np.float32).reshape(-1)
    out = np.empty_like(x)
    (helper.chop_levels_rule if rule else helper.chop_levels_facade)(x.ctypes.data_as(_f32p), x.size, out.ctypes.data_as(_f32p))
    return out


def peak(x):
    """(max |x| from 0 with NaN ignored, first index carrying it or 0)"""
    a = np.abs(np.asarray(x, np.float32))
    m = np.float32(np.nanmax(a)) if np.any(~np.isnan(a)) else np.float32(0)
    m = max(m, np.float32(0))
    hit = np.flatnonzero(a == m)
    return m, int(hit[0]) if hit.size else 0


def loud_flags(x, ir_length, threshold_db, lv, peak_db):
    """loud_j for j in [0, ir_length) of the backward walk from the peak (lv: levels of every sample of x)"""
    n = len(x)
    _, q = peak(x)
    s = (q - np.arange(ir_length)) % n
    with np.errstate(invalid="ignore"):
        quiet = (lv[s] - np.float32(peak_db)).astype(np.float32) < np.float32(threshold_db)
    return ~quiet


def walk(loud, consecutive):
    """walked: first j with a run of >= consecutive quiet positions ending at j, plus one; len(loud) when none; 0 for consecutive <= 0"""
    Lw = len(loud)
    if consecutive <= 0:
        return 0
    if consecutive > Lw:
        return Lw
    last = np.maximum.accumulate(np.where(loud, np.arange(Lw), -1))
    hit = np.flatnonzero(np.arange(Lw) - last >= consecutive)
    return int(hit[0]) + 1 if hit.size else Lw


def chop(helper, x, ir_length, threshold_db, consecutive, rule=True, normalize=False, goal_lin=np.float32(1.0)):
    """-> (out[ir_length] float32, q, start): fp::ir::IRchop (+ tools::normalize) by the statement above"""
    x = np.asarray(x, np.float32)
    n = len(x)
    pk, q = peak(x)
    lv = levels(helper, x, rule)
    peak_db = levels(helper, np.array([pk], np.float32), rule)[0]
    walked = walk(loud_flags(x, ir_length, threshold_db, lv, peak_db), consecutive)
    start = (q - walked) % n
    out = x[(start + np.arange(ir_length)) % n].copy()
    f32 = np.float32
    with np.errstate(invalid="ignore", over="ignore"):
        n_out = ir_length // 4
        if n_out:
            step = f32(1.0 / n_out)
            i = np.arange(n_out)
            g = (1.0 - (i.astype(f32) * step).astype(np.float64)).astype(f32)
            o0 = ir_length - 1 - n_out
            out[o0:o0 + n_out] = out[o0:o0 + n_out] * g
        n_in = walked // 4
        if n_in:
            step = f32(1.0 / n_in)
            out[:n_in] = out[:n_in] * (np.arange(n_in).astype(f32) * step)
        if normalize:
            a = np.abs(out)
            mag = f32(np.nanmax(a)) if np.any(~np.isnan(a)) else f32(0)
            mag = max(mag, f32(0))
            with np.errstate(divide="ignore"):
                gain = f32(goal_lin) / mag
            out = (out * gain).astype(f32)
    return out.astype(f32), q, start


def decisions_agree(helper, x, ir_length, threshold_db):
    """True when the facade's levels and the device rule's give the same peak level and the same loud/quiet flag at every position
    the walk can visit: the row does not sit on a glibc-vs-correctly-rounded decision flip"""
    x = np.asarray(x, np.float32)
    pk, _ = peak(x)
    p = np.array([pk], np.float32)
    pf, pr = levels(helper, p, False)[0], levels(helper, p, True)[0]
    if not (pf == pr or (np.isnan(pf) and np.isnan(pr))):
        return False
    return bool(np.array_equal(loud_flags(x, ir_length, threshold_db, levels(helper, x, False), pf),
                               loud_flags(x, ir_length, threshold_db, levels(helper, x, True), pr)))


def cases(seed=0):
    """[(name, row float32, ir_length, threshold_db, consecutive)]: wrap at both ends, ties for the peak, consecutive 0, 1 and
    > ir_length, ir_length < 4 and == n, silent rows, NaN / Inf rows, and many random decaying IRs"""
    rng = np.random.default_rng(seed)
    f32 = np.float32

    def ir_row(n, q, floor_db=-90.0, pre=0, decay=None):
        r = (rng.standard_normal(n) * 10.0 ** (floor_db / 20.0)).astype(f32)
        decay = decay or max(4.0, n / 16)
        t = np.arange(n - q)
        r[q:] += np.clip(rng.standard_normal(n - q) * np.exp(-t / decay), -1.4, 1.4).astype(f32)
        r[q] = f32(1.5)
        if pre:                                          # a loud stretch before the peak the walk has to pass
            r[max(0, q - pre - 10):q - 10] += (0.01 * rng.standard_normal(min(pre, q - 10))).astype(f32)
        return r

    out = []
    for n, q, L, thr, c in [(4096, 2000, 1024, -60.0, 50), (4096, 5, 1024, -60.0, 50), (4096, 4090, 1024, -60.0, 50), (4096, 3000, 2048, -60.0, 50),
                            (4096, 30, 2048, -40.0, 20), (1000, 999, 500, -60.0, 10), (1000, 0, 1000, -60.0, 3), (4096, 2000, 1024, -60.0, 0),
                            (4096, 2000, 1024, -60.0, 1), (4096, 2000, 100, -60.0, 101), (4096, 2000, 100, -60.0, 100), (4096, 2000, 3, -60.0, 2),
                            (4096, 2000, 2, -60.0, 1), (4096, 2000, 1, -60.0, 1), (4096, 7, 4096, -60.0, 50), (16, 3, 16, -60.0, 2), (1, 0, 1, -60.0, 1)]:
        out.append(("ir_n%d_q%d_L%d_c%d" % (n, q, L, c), ir_row(n, q) if n > 1 else np.array([0.25], f32), L, thr, c))
    out.append(("loud_stretch", ir_row(8192, 4000, pre=600), 2048, -60.0, 50))
    out.append(("never_quiet", (rng.standard_normal(4096)).astype(f32), 1000, -60.0, 50))
    tie = ir_row(4096, 3000)
    tie[1200] = f32(1.5)
    tie[3500] = f32(-1.5)
    out.append(("tie", tie, 1024, -60.0, 50))
    neg = ir_row(4096, 100)
    neg[100] = f32(-1.5)
    neg[2500] = f32(1.5)
    out.append(("tie_negative_first", neg, 1024, -60.0, 50))
    out.append(("zeros", np.zeros(4096, f32), 1024, -60.0, 50))
    out.append(("zeros_threshold_above_0", np.zeros(4096, f32), 1024, 1.0, 50))
    out.append(("all_nan", np.full(4096, np.nan, f32), 1024, -60.0, 50))
    nan = ir_row(4096, 2000)
    nan[1990:1995] = np.nan
    nan[2100] = np.nan
    out.append(("some_nan", nan, 1024, -60.0, 50))
    inf = ir_row(4096, 2000)
    inf[2500] = np.inf
    out.append(("inf", inf, 1024, -60.0, 50))
    ninf = ir_row(4096, 2000)
    ninf[100] = -np.inf
    ninf[101] = np.inf
    out.append(("two_inf", ninf, 1024, -60.0, 50))
    for k in range(40):
        n = int(rng.integers(16, 6000))
        q = int(rng.integers(0, n))
        L = int(rng.integers(1, n + 1))
        out.append(("random%d" % k, ir_row(n, q, floor_db=float(rng.uniform(-120, -30)), decay=float(rng.uniform(2, n))), L,
                    float(rng.choice([-80.0, -60.0, -40.0, -20.0])), int(rng.choice([0, 1, 2, 5, 50, 200, L, L + 1]))))
    return out
