"""Static instruction counts of one pair-kernel instantiation (no GPU needed):

    python scripts/pair_sass.py                      # st_pair_kernel<25, true> of this tree
    python scripts/pair_sass.py --src OTHER_TREE     # the same for another checkout (e.g. a git worktree of the parent)
    python scripts/pair_sass.py --json out.json

Compiles csrc/b200aa.cu to a cubin with the library's nvcc flags, reads registers / stack / spills from `-Xptxas -v`
and disassembles the kernel with inline line info (`nvdisasm -gi`).  Prints one JSON object:
  total       every SASS instruction of the function (all paths)
  steady      instructions between the step loop's head and its back-edge (the shortest loop in the SASS that holds the
              code of the `for (int q ...)` body) on the path the 800 / 400 benchmark takes every step: int16 samples,
              one-sided sign masks, shared halves, no |X| dump, no tile flush.  Instructions whose inline chain passes
              through one of those excluded source lines are not counted; everything else in the loop is, including
              what ptxas recomputes there (lane, shared-memory bases).
  ops / steady_ops   counts of a few opcodes of interest in both sets
The step loop and the off-path lines are found by matching source text in pair_kernel.cuh, so the script follows edits.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OPS = ("S2R", "S2UR", "CS2R", "POPC", "VOTE", "REDUX", "SHFL", "LDS", "STS", "LDL", "STL", "BAR", "WARPSYNC")


def _nvcc():
    return os.environ.get("NVCC") or "/usr/local/cuda/bin/nvcc"


def _tool(name):
    return os.path.join(os.path.dirname(_nvcc()), name) if os.path.isabs(_nvcc()) else name


def line_of(lines, pattern, start=0):
    for i in range(start, len(lines)):
        if pattern in lines[i]:
            return i + 1
    raise SystemExit("pattern not found in pair_kernel.cuh: %r" % pattern)


def steady_lines(src):
    """(first, last) lines of the kernel and of its step loop, and the off-path line ranges."""
    lines = open(src).read().split("\n")
    k0 = line_of(lines, "st_pair_kernel(const PairParams pp)")
    loop0 = line_of(lines, "for (int q = q0 - ((fresh", k0)
    loop1 = line_of(lines, "__syncwarp();                    // the copy above has read the buffer", loop0)
    off = []
    # float32 samples (load and conversion)
    ld = line_of(lines, "} else {", line_of(lines, "auto load_pair", k0))
    off.append((ld, ld + 4))
    cv = line_of(lines, "} else {", line_of(lines, "if (is16) {", line_of(lines, "load_pair(q, wa, wb);", k0)))
    off.append((cv, cv + 3))
    # first step of a run (whole frame a)
    f0 = line_of(lines, "// first step of a run: all of a", loop0)
    f1 = line_of(lines, "zprev = fb_ - lb_;", f0)
    off.append((f0, f1))
    # two-sided sign masks (a sample may equal the clip mean)
    ts = line_of(lines, "if (two_sided) td_pair<R, false, true>", loop0)
    off.append((ts, ts))
    # |X| dump
    d0 = line_of(lines, "if (pp.dbg) {", loop0)
    off.append((d0, d0 + 9))
    # tile flush inside the loop (every fourth step)
    fl = line_of(lines, "if (tile_n == 8) B200AA_PAIR_FLUSH(cb);", loop0)
    off.append((fl, fl))
    return (k0, line_of(lines, "#undef B200AA_PAIR_FLUSH", k0)), loop0, loop1, off


def compile_cubin(src_root, out_dir):
    csrc = os.path.join(src_root, "pyaudioanalysis_b200", "csrc")
    cubin = os.path.join(out_dir, "b200aa.cubin")
    cmd = [_nvcc(), "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-cubin",
           "-Xptxas", "-v", "-o", cubin, os.path.join(csrc, "b200aa.cu")]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise SystemExit("nvcc failed")
    return cubin, res.stderr


def ptxas_stats(log, mangled):
    m = re.search(r"Function properties for %s\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads\n"
                  r".*?Used (\d+) registers" % re.escape(mangled), log)
    if not m:
        raise SystemExit("no ptxas record for " + mangled)
    return {"registers": int(m.group(4)), "stack": int(m.group(1)), "spill_stores": int(m.group(2)), "spill_loads": int(m.group(3))}


def disasm(cubin, mangled):
    sym = subprocess.run(["readelf", "-sW", cubin], capture_output=True, text=True).stdout
    idx = None
    for ln in sym.split("\n"):
        f = ln.split()
        if len(f) >= 8 and f[-1] == mangled and f[3] == "FUNC":
            idx = f[0].rstrip(":")
    if idx is None:
        raise SystemExit("symbol not found: " + mangled)
    return subprocess.run([_tool("nvdisasm"), "-gi", "-fun", idx, cubin], capture_output=True, text=True).stdout


def parse(text, kernel_file):
    """[(address, opcode, inline chain of kernel_file lines, innermost first)], backward branches [(target, source)]"""
    ins_re = re.compile(r"^/\*([0-9a-f]{4,})\*/\s+(?:@!?U?P\w+\s+)?([A-Z][A-Z0-9_]*)([^;]*);")
    rows, labels, pending, chain = [], {}, [], []
    for ln in text.split("\n"):
        s = ln.strip()
        if s.startswith("//## File"):
            chain = [int(n) for f, n in re.findall(r'"([^"]+)", line (\d+)', s) if f.endswith(kernel_file)]
            continue
        m = re.match(r"^(\.L_x_\d+):", s)
        if m:
            pending.append(m.group(1))
            continue
        m = ins_re.match(s)
        if m:
            a = int(m.group(1), 16)
            for lab in pending:
                labels[lab] = a
            pending = []
            rows.append((a, m.group(2), m.group(3), chain))
    back = []
    for a, op, rest, _ in rows:
        m = re.search(r"`\((\.L_x_\d+)\)", rest)
        if op == "BRA" and m and labels[m.group(1)] <= a:
            back.append((labels[m.group(1)], a))
    return rows, back


def count(text, kernel_file, kernel, loop0, loop1, off):
    rows, back = parse(text, kernel_file)
    # nvdisasm names one level of inlining only: code two calls deep (an intrinsic in a helper) carries no kernel line.
    # It belongs to the kernel line of the code around it, so that line is carried forward and appended to the chain.
    ctx = None
    for i, (a, op, rest, chain) in enumerate(rows):
        if chain and kernel[0] <= chain[-1] <= kernel[1]:
            ctx = chain[-1]
        elif ctx is not None:
            rows[i] = (a, op, rest, chain + [ctx])
    in_loop = lambda c: bool(c) and loop0 <= c[-1] <= loop1
    n_loop = sum(1 for r in rows if in_loop(r[3]))
    # the step loop: the shortest backward-branch span that holds (nearly) all instructions of its source lines
    spans = [(b - t, t, b) for t, b in back if sum(1 for r in rows if t <= r[0] <= b and in_loop(r[3])) >= 0.9 * n_loop]
    _, head, tail = min(spans)
    ops = {o: 0 for o in OPS}
    sops = {o: 0 for o in OPS}
    steady = 0
    for a, op, _, chain in rows:
        if op in ops:
            ops[op] += 1
        if not head <= a <= tail or any(x <= c <= y for c in chain for x, y in off):
            continue
        steady += 1          # includes what ptxas rematerialises inside the loop (lane, shared-memory bases)
        if op in sops:
            sops[op] += 1
    return len(rows), steady, ops, sops, (head, tail)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--src", default=ROOT, help="repository tree to compile")
    ap.add_argument("--R", type=int, default=25)
    ap.add_argument("--shared", type=int, default=1)
    ap.add_argument("--json", help="also write the result here")
    ap.add_argument("--sass", help="also write the kernel's disassembly (with inline line info) here")
    a = ap.parse_args()
    mangled = "_ZN6b200aa14st_pair_kernelILi%dELb%dEEEvNS_10PairParamsE" % (a.R, a.shared)
    src = os.path.join(a.src, "pyaudioanalysis_b200", "csrc", "pair_kernel.cuh")
    kernel, loop0, loop1, off = steady_lines(src)
    with tempfile.TemporaryDirectory() as td:
        cubin, log = compile_cubin(a.src, td)
        st = ptxas_stats(log, mangled)
        text = disasm(cubin, mangled)
    if a.sass:
        with open(a.sass, "w") as f:
            f.write(text)
    total, steady, ops, sops, span = count(text, "pair_kernel.cuh", kernel, loop0, loop1, off)
    res = {"kernel": "st_pair_kernel<%d, %s>" % (a.R, "true" if a.shared else "false"), **st,
           "total": total, "steady": steady, "ops": ops, "steady_ops": sops,
           "step_loop_lines": [loop0, loop1], "step_loop_sass": [hex(span[0]), hex(span[1])], "off_path_lines": off}
    print(json.dumps(res))
    if a.json:
        with open(a.json, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
