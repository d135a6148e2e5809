"""Per-kernel `ptxas -v` summary of an nvcc log: one line per kernel (demangled name, stack, spills, registers, barriers,
static shared memory), sorted by name, so that two builds can be compared with diff.

    python profiles/ptxas_table.py pgmorl_b200/build/k3_ppo.o.log > before.txt
"""
import re
import subprocess
import sys


def table(log):
    rows, name = [], None
    for line in open(log):
        m = re.search(r"Compiling entry function '(\w+)'", line)
        if m:
            name = m.group(1)
            continue
        m = re.search(r"Function properties for (\w+)", line)
        if m:
            name = m.group(1)
            continue
        if name and "bytes stack frame" in line:
            spill = line.split("ptxas info    :")[-1].strip() if "ptxas info" in line else line.strip()
            rows.append([name, spill, None])
        elif name and "Used" in line and "registers" in line and rows and rows[-1][0] == name:
            rows[-1][2] = line.split("ptxas info    :")[-1].strip()
    names = subprocess.run(["c++filt"], input="\n".join(r[0] for r in rows), capture_output=True, text=True).stdout.split("\n")
    out = []
    for (mangled, spill, used), dem in zip(rows, names):
        if used is None:
            continue
        dem = re.sub(r"^void pgm::", "", dem.strip())
        dem = re.sub(r"\(pgm::\w+\)$", "", dem).replace(" ", "")
        out.append(f"{dem:48s} {spill} | {used}")
    return sorted(set(out))


if __name__ == "__main__":
    print("\n".join(table(sys.argv[1])))
