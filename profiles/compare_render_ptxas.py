"""Compiler output of the library's CUDA sources (build.SOURCES) at two source trees: ptxas registers, spills and stack per kernel,
and which kernels compile to the same SASS.  Host only (nvcc + cuobjdump, no GPU): the check a refactor owes before any run.

    python profiles/compare_render_ptxas.py BASE_CSRC NEW_CSRC [--out FILE]

BASE_CSRC / NEW_CSRC are csrc directories (e.g. one extracted with `git archive <rev> dd2360-raytracing_b200/csrc include`; the
include/ directory must sit two levels above csrc, as in the repository).  Both are compiled with the flags of build.py, once
plain and once with -DRT_COUNTERS.  Exit status 1 if a kernel of both trees uses more registers, spill bytes or stack in NEW.
"""
from __future__ import annotations

import argparse
import os
import re
import subprocess
import sys
import tempfile
from concurrent.futures import ThreadPoolExecutor

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "dd2360-raytracing_b200"))
import build as rt_build  # noqa: E402

ENTRY = re.compile(r"Compiling entry function '(\w+)'")
STACK = re.compile(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads")
REGS = re.compile(r"Used (\d+) registers")


def compile_source(csrc: str, src: str, extra: list[str], tmp: str) -> tuple[dict, dict]:
    """-> ({kernel: (regs, spill stores, spill loads, stack)}, {kernel: [SASS lines without addresses]}) of one source"""
    obj = os.path.join(tmp, src.replace(".cu", ".o"))
    cmd = [rt_build._nvcc(), *rt_build.NVCC_FLAGS, *extra, "-Xptxas", "-v", "-c", os.path.join(csrc, src), "-o", obj]
    log = subprocess.run(cmd, check=True, capture_output=True, text=True).stderr
    res, cur, stack = {}, None, (0, 0, 0)
    for line in log.splitlines():
        if m := ENTRY.search(line):
            cur, stack = m.group(1), (0, 0, 0)
        elif (m := STACK.search(line)) and cur:
            stack = (int(m.group(2)), int(m.group(3)), int(m.group(1)))
        elif (m := REGS.search(line)) and cur:
            res[cur] = (int(m.group(1)), *stack)
            cur = None
    sass, name = {}, None
    for line in subprocess.run(["cuobjdump", "-sass", obj], check=True, capture_output=True, text=True).stdout.splitlines():
        if m := re.match(r"\s*Function : (\w+)", line):
            name = m.group(1)
            sass[name] = []
        elif name and (m := re.match(r"\s*/\*[0-9a-f]{4,}\*/\s*(.*?)\s*/\*", line)):
            sass[name].append(m.group(1))
    return res, sass


def demangle(names: list[str]) -> dict:
    out = subprocess.run(["cu++filt"], input="\n".join(names), check=True, capture_output=True, text=True).stdout.splitlines()
    out = [d.replace("(bool)1", "true").replace("(bool)0", "false").replace("(int)", "") for d in out]
    return {n: re.sub(r"^void |\(.*$", "", d).replace("rt::", "").replace("coop::", "").replace("h16::", "") for n, d in zip(names, out)}


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("base")
    ap.add_argument("new")
    ap.add_argument("--out")
    a = ap.parse_args()
    lines, worse = [], False
    for label, extra in (("plain build", []), ("-DRT_COUNTERS build", ["-DRT_COUNTERS"])):
        with tempfile.TemporaryDirectory() as t0, tempfile.TemporaryDirectory() as t1, ThreadPoolExecutor() as ex:
            jobs = [(src, ex.submit(compile_source, a.base, src, extra, t0), ex.submit(compile_source, a.new, src, extra, t1))
                    for src in rt_build.SOURCES]
            results = [(src, f0.result(), f1.result()) for src, f0, f1 in jobs]
        for src, (r0, s0), (r1, s1) in results:
            names = sorted(set(r0) | set(r1))
            dm = demangle(names)
            same = [n for n in names if n in s0 and n in s1 and s0[n] == s1[n]]
            lines.append(f"{label}, {src}: {len(same)} of {len(r0)} kernels SASS-identical")
            differ = [n for n in names if n not in same]
            if differ:
                lines.append(f"  {'kernel':58s} {'regs':>9s} {'spill st':>11s} {'spill ld':>11s} {'stack':>11s}   (base -> new)")
            for n in differ:
                b, c = r0.get(n), r1.get(n)
                cells = [f"{'-' if b is None else b[k]:>4} -> {'-' if c is None else c[k]:<4}" for k in range(4)]
                flag = ""
                if b and c and any(c[k] > b[k] for k in range(4)):
                    flag, worse = "  WORSE", True
                lines.append(f"  {dm[n]:58s} {cells[0]:>9s} {cells[1]:>11s} {cells[2]:>11s} {cells[3]:>11s}{flag}")
            lines.append("  SASS-identical: " + ", ".join(dm[n] for n in same))
            lines.append("")
    text = "\n".join(lines)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text)
    return 1 if worse else 0


if __name__ == "__main__":
    sys.exit(main())
