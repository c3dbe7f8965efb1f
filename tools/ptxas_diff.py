"""Per-kernel registers, spill bytes and stack frame from two `nvcc -Xptxas -v` logs (e.g. two `build(verbose=True,
force=True)` runs, before and after a change), as a table.  Usage: ptxas_diff.py BEFORE_LOG AFTER_LOG."""
import re
import subprocess
import sys


def parse(text):
    out, fn = {}, None
    for line in text.splitlines():
        m = re.search(r"Compiling entry function '(\S+)'|Function properties for (\S+)", line)
        if m:
            fn = m.group(1) or m.group(2)
            out.setdefault(fn, {})
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and fn:
            out[fn].update(stack=int(m.group(1)), spill_st=int(m.group(2)), spill_ld=int(m.group(3)))
        m = re.search(r"Used (\d+) registers", line)
        if m and fn:
            out[fn]["regs"] = int(m.group(1))
    return {k: v for k, v in out.items() if "regs" in v}


def demangle(names):
    r = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True)
    return r.stdout.split("\n")[: len(names)] if r.returncode == 0 else names


def normalise(table):
    """Key by demangled name (anonymous-namespace ids differ between trees); a kernel that gained a `bool Prog`
    template argument is matched to its old name through its `false` instantiation."""
    names = list(table)
    out = {}
    for n, d in zip(names, demangle(names)):
        d = d.replace(", false>", ">").replace("<false>", "").removeprefix("void ")
        out[d] = table[n]
    return out


def main(before, after):
    b, a = normalise(parse(open(before).read())), normalise(parse(open(after).read()))
    names = sorted(set(b) | set(a))
    grew = 0
    print(f"{'kernel':120s} {'regs':>9s} {'spill st/ld':>15s} {'stack':>11s}")
    for n in names:
        d = n
        x, y = b.get(n), a.get(n)
        f = lambda e, k: "-" if e is None else str(e.get(k, 0))
        if x and y and (y["regs"] > x["regs"] or y.get("spill_st", 0) > x.get("spill_st", 0) or y.get("spill_ld", 0) > x.get("spill_ld", 0)):
            grew += 1
        mark = "" if x and y and x == y else ("  new" if not x else ("  removed" if not y else "  changed"))
        print(f"{d[:120]:120s} {f(x,'regs'):>4s}>{f(y,'regs'):<4s} {f(x,'spill_st')+'/'+f(x,'spill_ld'):>7s}>{f(y,'spill_st')+'/'+f(y,'spill_ld'):<7s} "
              f"{f(x,'stack'):>5s}>{f(y,'stack'):<5s}{mark}")
    print(f"kernels whose registers or spills grew: {grew}")
    return grew


if __name__ == "__main__":
    sys.exit(1 if main(sys.argv[1], sys.argv[2]) else 0)
