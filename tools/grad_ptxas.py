"""ptxas resources of every jk_grad_kernel instantiation, as a markdown table (profiles/grad/ptxas_jk_grad*.md).

Compiles joltqc_b200/csrc/jk_grad_inst.cu once per bra class with the library's flags and -Xptxas -v
(no GPU needed) and prints one row per (class, NSPIN) instantiation: registers, stack frame, spill stores,
spill loads.

    python tools/grad_ptxas.py --nspin 1 [--check profiles/grad/ptxas_jk_grad.md]
    python tools/grad_ptxas.py --nspin 2 > profiles/grad/ptxas_jk_grad_uhf.md

--check compares the rows with a committed table and exits non-zero on any difference.
"""
import argparse
import os
import re
import subprocess
import sys
import tempfile
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from joltqc_b200 import build as B  # noqa: E402

ENTRY = re.compile(r"Compiling entry function '(\S+)'")
RES = re.compile(r"Used (\d+) registers")
STACK = re.compile(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads")
# _ZN3jqc14jk_grad_kernelILi2ELi1ELi1ELi0ELb1ELi128ELi1EEEvNS_8GradArgsE: LI, LJ, LK, LL, SMALL, NT[, NSPIN]
TARGS = re.compile(r"jk_grad_kernelILi(\d)ELi(\d)ELi(\d)ELi(\d)ELb([01])ELi(\d+)E(?:Li(\d)E)?E")


def compile_unit(ij):
    i, j = ij
    with tempfile.TemporaryDirectory() as tmp:
        cmd = [B.NVCC] + B.FLAGS + ["-Xptxas", "-v", f"-DJQC_LI={i}", f"-DJQC_LJ={j}", "-c",
                                    os.path.join(B.CSRC, "jk_grad_inst.cu"), "-o", os.path.join(tmp, "o.o")]
        r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode:
        raise RuntimeError(r.stderr)
    return r.stderr


def parse(text):
    rows = {}
    cur = None
    for line in text.splitlines():
        m = ENTRY.search(line)
        if m:
            t = TARGS.search(m.group(1))
            cur = None
            if t:
                li, lj, lk, ll, small, _, nspin = t.groups()
                cur = (f"({li}{lj}\\|{lk}{ll})", "unrolled" if small == "1" else "rolled", int(nspin or 1))
                rows[cur] = [None, 0, 0, 0]
            continue
        if cur is None:
            continue
        m = STACK.search(line)
        if m:
            rows[cur][1:] = [int(x) for x in m.groups()]
        m = RES.search(line)
        if m:
            rows[cur][0] = int(m.group(1))
    return rows


def table_rows(rows, nspin):
    out = []
    for (cls, var, ns), (reg, stack, st, ld) in sorted(rows.items()):
        if ns == nspin:
            out.append(f"| {cls} | {var} | {reg} | {stack} | {st} | {ld} |")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nspin", type=int, default=1, choices=(1, 2))
    ap.add_argument("--check", help="committed table to compare the rows with")
    ap.add_argument("--jobs", type=int, default=os.cpu_count())
    args = ap.parse_args()
    with ThreadPoolExecutor(args.jobs) as ex:
        texts = list(ex.map(compile_unit, sorted(B.BRA, key=lambda c: -(c[0] + c[1]))))
    rows = {}
    for t in texts:
        rows.update(parse(t))
    mine = table_rows(rows, args.nspin)
    if args.check:
        with open(args.check) as f:
            ref = [ln.strip() for ln in f if re.match(r"\| \(\d\d", ln)]
        diff = [(a, b) for a, b in zip(ref, mine) if a != b]
        if len(ref) != len(mine) or diff:
            for a, b in diff:
                print(f"committed: {a}\nnow:       {b}")
            print(f"{len(ref)} committed rows, {len(mine)} now, {len(diff)} differ")
            sys.exit(1)
        print(f"{len(mine)} rows identical to {args.check}")
        return
    n_unrolled = sum(1 for r in mine if "| unrolled |" in r)
    print("| class (ij\\|kl) | variant | registers | stack frame (B) | spill stores (B) | spill loads (B) |")
    print("|---|---|---|---|---|---|")
    print("\n".join(mine))
    print(f"\n{len(mine)} instantiations ({len(mine) - n_unrolled} rolled, {n_unrolled} unrolled).")


if __name__ == "__main__":
    main()
