"""Static instruction budget of a kernel's loops, from `cuobjdump -sass` of an sm_100a cubin.

    python tools/sass_loop_budget.py CUBIN_OR_SASS FUNCTION_SUBSTRING

Every backward branch closes a loop; the loop body is the range [branch target, branch].  For each loop this prints
its address range, its instruction count, the count per opcode class and how many STTM / STS / LDS / UTC*MMA it holds
(which identify the warp role that runs it).  Out-of-line retry paths of mbarrier waits lie outside these ranges (a
backward branch whose range holds an EXIT is such a path and is skipped), so the counts are the instructions issued
per iteration when no wait has to spin."""
import collections
import re
import subprocess
import sys

INSN = re.compile(r"/\*([0-9a-f]{4,})\*/\s+(@!?U?P\w+\s+)?([A-Z][A-Z0-9_]*)(\.[A-Z0-9_.]+)?\s*([^;]*);")
BRA_TARGET = re.compile(r"0x([0-9a-f]+)")


def load_sass(path):
    if path.endswith(".sass") or path.endswith(".txt"):
        return open(path).read()
    return subprocess.run(["cuobjdump", "-sass", path], check=True, capture_output=True, text=True).stdout


def function_insns(sass, name):
    out, inside = [], False
    for line in sass.splitlines():
        if "Function :" in line:
            inside = name in line
            continue
        if inside:
            m = INSN.search(line)
            if m:
                out.append((int(m.group(1), 16), m.group(3), (m.group(4) or ""), m.group(5)))
    return out


def main():
    path, name = sys.argv[1], sys.argv[2]
    insns = function_insns(load_sass(path), name)
    if not insns:
        raise SystemExit(f"no function matching {name!r} in {path}")
    by_addr = {a: i for i, (a, *_) in enumerate(insns)}
    print(f"{name}: {len(insns)} instructions")
    for i, (addr, op, _mod, args) in enumerate(insns):
        if not op.startswith("BRA"):
            continue
        t = BRA_TARGET.search(args)
        if not t or int(t.group(1), 16) >= addr:
            continue
        body = insns[by_addr[int(t.group(1), 16)] : i + 1]
        ops = collections.Counter(op for _a, op, _m, _x in body)
        if ops["EXIT"]:
            continue  # an out-of-line wait retry jumping back into straight-line code, not a loop
        marks = {k: sum(v for o, v in ops.items() if o.startswith(k)) for k in ("STTM", "STS", "LDS", "UTC")}
        print(f"loop [0x{body[0][0]:04x}, 0x{addr:04x}]: {len(body)} instructions; "
              + ", ".join(f"{k} {v}" for k, v in marks.items() if v))
        print("   " + " ".join(f"{o}:{c}" for o, c in ops.most_common()))


if __name__ == "__main__":
    main()
