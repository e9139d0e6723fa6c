"""Local-memory (stack / spill) instructions of the grid kernel, by time-step phase.

    python tools/grid_local_memory.py [--cubin FILE] [--kernel SUBSTR ...]

Compiles csrc/sv_grid.cu to a cubin with the library's flags (or reads --cubin), prints ptxas's stack frame and spill
bytes of every sv_grid_kernel instantiation, then disassembles the selected instantiations (default: the SV gradient
smoother, one problem and team) with line information and counts the STL / LDL sites per phase.  Each site counts once
(static count); how often it runs is not measured here.  A phase is the source between two PROF_MARK calls of the time
loop and is named after the comment of the mark that closes it; an inlined helper counts in the phase of its call site.
Needs nvcc, cuobjdump and nvdisasm (CUDA toolkit); no GPU.
"""
import argparse
import os
import re
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "..", "pmmh-qn_b200", "csrc", "sv_grid.cu")
sys.path.insert(0, os.path.join(HERE, "..", "pmmh-qn_b200"))
from _build import NVCC_FLAGS  # noqa: E402

HEADLINE = ["ILi1024ELb0ENS_15SvLeverageModelELb1ELb0E", "ILi1024ELb0ENS_15SvLeverageModelELb1ELb1E"]


def compile_cubin(out):
    nvcc = os.environ.get("NVCC", "nvcc")
    flags = [f for f in NVCC_FLAGS if f not in ("-shared", "-Xcompiler", "-fPIC")]
    cmd = [nvcc] + flags + ["-Xptxas", "-v", "-cubin", "-o", out, SRC]
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout)
        raise SystemExit("nvcc failed")
    return res.stdout


def ptxas_table(log):
    """{mangled kernel name: (registers, stack, spill stores, spill loads)} of the sv_grid_kernel instantiations."""
    out, name, frame = {}, None, None
    for line in log.splitlines():
        m = re.search(r"Compiling entry function '(\w+)'", line)
        if m:
            name, frame = m.group(1), None
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and name:
            frame = tuple(int(v) for v in m.groups())
        m = re.search(r"Used (\d+) registers", line)
        if m and name and frame is not None:
            if "sv_grid_kernel" in name:
                out[name] = (int(m.group(1)),) + frame
            name = None
    return out


def short(name):
    m = re.search(r"sv_grid_kernelILi(\d+)ELb(\d)ENS_\d+(\w+?)ELb(\d)ELb(\d)E", name)
    gt, hess, model, smo, team = m.groups()
    return f"<{gt}, {'true' if hess == '1' else 'false'}, {model}, {'true' if smo == '1' else 'false'}, " \
           f"{'true' if team == '1' else 'false'}>"


def phases():
    """[(last source line, phase name)] of the time loop, in source order, and the loop's line range."""
    lines = open(SRC).read().splitlines()
    start = next(i for i, l in enumerate(lines, 1) if "for (int t = 1; t < NOBS; ++t)" in l)
    marks = []
    for i, l in enumerate(lines, 1):
        m = re.search(r"PROF_MARK\((\d+)\);\s*//\s*(.*)", l)
        if m and i > start:
            marks.append((i, f"{m.group(1)}: {m.group(2).strip()}"))
    end = next(i for i, l in enumerate(lines, 1) if i > marks[-1][0] and l.strip() == "}")
    return marks, start, end


def classify(line, marks, start, end):
    if line is None or line < start or line > end:
        return "outside the time loop"
    for last, name in marks:
        if line <= last:
            return name
    return "end of the step"


def local_sites(cubin, kernel):
    dis = subprocess.run(["nvdisasm", "-gi", cubin], stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                         text=True).stdout
    marks, start, end = phases()
    counts, inside, line = {}, False, None
    fn = re.compile(r'//## File "([^"]*)", line (\d+)(?: inlined at "([^"]*)", line (\d+))?')
    for l in dis.splitlines():
        if l.startswith("\t.section"):
            inside = ".text." in l and kernel in l
            line = None
            continue
        if not inside:
            continue
        m = fn.search(l)
        if m:
            # the annotation without "inlined at" is the outermost frame, which comes last
            if m.group(3) is None and m.group(1).endswith("sv_grid.cu"):
                line = int(m.group(2))
            continue
        op = re.search(r"\b(STL|LDL)(\.\w+)*\b", l)
        if op and "/*" in l:
            ph = classify(line, marks, start, end)
            st = counts.setdefault(ph, [0, 0])
            st[0 if op.group(1) == "STL" else 1] += 1
    return counts, marks


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--cubin", help="a cubin of sv_grid.cu built with -lineinfo (default: compile one)")
    ap.add_argument("--kernel", action="append", help="substring of the mangled name (default: the SV gradient smoother)")
    args = ap.parse_args()
    with tempfile.TemporaryDirectory() as tmp:
        cubin = args.cubin
        if cubin is None:
            cubin = os.path.join(tmp, "sv_grid.cubin")
            table = ptxas_table(compile_cubin(cubin))
            print("| instantiation | registers | stack frame (B) | spill stores (B) | spill loads (B) |")
            print("|---|---|---|---|---|")
            for name in sorted(table, key=short):
                print(f"| {short(name)} | " + " | ".join(str(v) for v in table[name]) + " |")
            print()
        for k in args.kernel or HEADLINE:
            counts, marks = local_sites(cubin, k)
            print(f"local-memory sites of sv_grid_kernel{k}:")
            print("| phase (closing PROF_MARK) | STL | LDL |")
            print("|---|---|---|")
            order = [n for _, n in marks] + ["end of the step", "outside the time loop"]
            for ph in order:
                if ph in counts:
                    print(f"| {ph} | {counts[ph][0]} | {counts[ph][1]} |")
            loop = [v for ph, v in counts.items() if ph != "outside the time loop"]
            print(f"| time loop total | {sum(v[0] for v in loop)} | {sum(v[1] for v in loop)} |")
            print()


if __name__ == "__main__":
    main()
