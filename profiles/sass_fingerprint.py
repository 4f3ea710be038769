"""Compare the compiled kernels of two builds of libirb_b200.so instruction by instruction.

Usage: python profiles/sass_fingerprint.py OLD.so NEW.so [--exact irb_spectral.cu,irb_benchaids.cu]

For every `Function :` in `cuobjdump -sass` of both libraries it compares a fingerprint:
  * the multiset of opcodes, predicates removed and modifiers kept (`LDS.128`, `SYNCS.ARRIVE.TRANS64` ...);
  * the instruction count;
  * REG, STACK, SHARED and LOCAL from `cuobjdump -res-usage`.
A refactor that moves code into inline helpers should leave every fingerprint as it was: register numbers and the operand
order of commutative instructions may change, the work a kernel does may not.  Kernels of the translation units named by
--exact must in addition have identical SASS text and encodings once the instruction addresses are removed.

Prints one line per function and a summary; exits 1 when a function is missing on one side or any check fails.
"""
import argparse
import collections
import os
import re
import subprocess
import sys

CUOBJDUMP = os.environ.get("CUOBJDUMP", "/usr/local/cuda/bin/cuobjdump")
_INSN = re.compile(r"^\s*/\*[0-9a-f]{4,}\*/\s+(.*?)\s*;\s*(/\*.*\*/)?\s*$")
_ENC = re.compile(r"^\s*(/\* 0x[0-9a-f]+ \*/)\s*$")
_RES = re.compile(r"\b(REG|STACK|SHARED|LOCAL):(\d+)")


def _run(*args):
    return subprocess.run([CUOBJDUMP, *args], check=True, capture_output=True, text=True).stdout


def _unit(line):
    # "identifier = /path/a.cu /path/b.cu" -> the translation unit of this ELF (the first ELF of a link names them all)
    names = line.split("=", 1)[1].split()
    return os.path.basename(names[0]) if len(names) == 1 else None


def sass(lib):
    """{(unit, function): ([instruction text], [text + encoding])}; a static kernel may exist in several units."""
    funcs, unit, cur = {}, None, None
    for line in _run("-sass", lib).splitlines():
        if line.startswith("identifier ="):
            unit = _unit(line)
            continue
        m = re.match(r"^\s*Function : (\S+)", line)
        if m:
            cur = funcs.setdefault((unit, m.group(1)), ([], []))
            continue
        if cur is None:
            continue
        m = _INSN.match(line)
        if m:
            cur[0].append(m.group(1))
            cur[1].append(m.group(1) + " " + (m.group(2) or ""))
            continue
        m = _ENC.match(line)
        if m and cur[1]:
            cur[1][-1] += " " + m.group(1)
    return funcs


def resources(lib):
    res, unit, cur = {}, None, None
    for line in _run("-res-usage", lib).splitlines():
        if line.startswith("identifier ="):
            unit = _unit(line)
            continue
        m = re.match(r"^\s*Function (\S+):\s*$", line)
        if m:
            cur = (unit, m.group(1))
            continue
        if cur and "REG:" in line:
            res[cur] = {k: int(v) for k, v in _RES.findall(line)}
            cur = None
    return res


def opcode(insn):
    insn = re.sub(r"^@!?U?P\w+\s+", "", insn)      # predicate guard
    return insn.split()[0]


def fingerprint(insns, res):
    return collections.Counter(opcode(i) for i in insns), len(insns), tuple(res.get(k, -1) for k in ("REG", "STACK", "SHARED", "LOCAL"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("old")
    ap.add_argument("new")
    ap.add_argument("--exact", default="irb_spectral.cu,irb_benchaids.cu", help="translation units whose SASS must be identical")
    args = ap.parse_args()
    exact_units = set(u for u in args.exact.split(",") if u)
    old, new = sass(args.old), sass(args.new)
    rold, rnew = resources(args.old), resources(args.new)
    bad = 0
    only_old, only_new = sorted(set(old) - set(new)), sorted(set(new) - set(old))
    for u, f in only_old:
        print(f"MISSING in new  {u} {f}")
    for u, f in only_new:
        print(f"MISSING in old  {u} {f}")
    bad += len(only_old) + len(only_new)
    n_same_text = n_fail = 0
    for key in sorted(set(old) & set(new)):
        unit, f = key
        ho, no, ro = fingerprint(old[key][0], rold.get(key, {}))
        hn, nn, rn = fingerprint(new[key][0], rnew.get(key, {}))
        same_text = old[key][1] == new[key][1]
        n_same_text += same_text
        ok = ho == hn and no == nn and ro == rn and (same_text or unit not in exact_units)
        n_fail += not ok
        diff = ""
        if ho != hn:
            d = (hn - ho) + (ho - hn)
            diff = " opcodes " + ",".join(f"{k}:{ho[k]}->{hn[k]}" for k in sorted(d))
        print(f"{'ok  ' if ok else 'DIFF'} {unit} {f} insns {no}->{nn} REG/STACK/SHARED/LOCAL {'/'.join(map(str, ro))}->{'/'.join(map(str, rn))}"
              f" sass {'identical' if same_text else 'differs'}{diff}")
    n = len(set(old) & set(new))
    print(f"summary: {n} functions in both, {len(only_old)} only in old, {len(only_new)} only in new; "
          f"{n - n_fail} pass, {n_fail} fail; {n_same_text} with identical SASS; "
          f"identical SASS required for {','.join(sorted(exact_units)) or 'none'}")
    return 1 if bad + n_fail else 0


if __name__ == "__main__":
    sys.exit(main())
