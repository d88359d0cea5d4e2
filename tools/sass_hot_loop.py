"""SASS instruction counts of a sweep kernel's hot loops (profiles/r05_a): every straight-line block of the kernel that
holds packed FADD2 (one per two ray-triangle pairs of the interval test, or one per triangle of the closest-hit sweep's
segment verdict), with its instruction counts per triangle.

    cuobjdump -sass esctp1raytracer_b200/csrc/tracer_cuda.o | python tools/sass_hot_loop.py <mangled kernel name> [triangles per block]
"""
import collections
import re
import sys


def kernel_lines(lines, name):
    out, inside = [], False
    for ln in lines:
        if ln.strip().startswith("Function :"):
            inside = ln.split(":", 1)[1].strip() == name
            continue
        if inside:
            out.append(ln)
    return out


def blocks(lines):
    """split at branch targets (.L_x_ labels) and after branches"""
    cur = []
    for ln in lines:
        if re.match(r"\s*\.L_x_\d+:", ln):
            if cur:
                yield cur
            cur = []
            continue
        m = re.search(r"/\*[0-9a-f]+\*/\s+(@!?U?P\w+\s+)?([A-Z][A-Z0-9_.]*)", ln)
        if not m:
            continue
        cur.append((m.group(2), ln.strip()))
        if m.group(2).split(".")[0] in ("BRA", "EXIT", "RET", "CALL", "BRX", "JMP"):
            yield cur
            cur = []
    if cur:
        yield cur


def main():
    name = sys.argv[1]
    per = int(sys.argv[2]) if len(sys.argv) > 2 else 16
    lines = kernel_lines(sys.stdin.read().splitlines(), name)
    if not lines:
        sys.exit("kernel not found: " + name)
    total = collections.Counter(op for b in blocks(lines) for op, _ in b)
    print("## %s: FP instruction counts (whole kernel)" % name)
    for op, n in sorted(total.items(), key=lambda x: -x[1]):
        if op.split(".")[0] in ("FFMA", "FADD", "FADD2", "FMUL", "FMNMX", "FMNMX3", "FFMA2", "FMUL2"):
            print("#  %6d %s" % (n, op))
    hot = [b for b in blocks(lines) if sum(op == "FADD2" for op, _ in b) >= per]
    for b in sorted(hot, key=lambda b: -sum(op == "FADD2" for op, _ in b)):
        c = collections.Counter(op for op, _ in b)
        fadd2 = c["FADD2"]
        if fadd2 == per and c["FMNMX3"] == 2 * per:  # segment verdict: one FADD2 per triangle, no per-pair work
            print("## hot-loop block at %s: %d instructions, %d FADD2 = one per triangle (segment verdict) x %d triangles"
                  % (b[0][1].split("*/")[0] + "*/", len(b), fadd2, per))
        else:
            print("## hot-loop block at %s: %d instructions, %d FADD2 = %d rays per thread x %d triangles"
                  % (b[0][1].split("*/")[0] + "*/", len(b), fadd2, 2 * fadd2 // per, per))
        print("#  per triangle: " + ", ".join("%g %s" % (n / per, op) for op, n in sorted(c.items(), key=lambda x: -x[1])
                                             if op.split(".")[0] in ("FFMA", "FADD", "FADD2", "FMNMX3", "FMNMX", "LDS", "FSETP", "SEL",
                                                                     "IADD3", "LOP3")))
        if fadd2 != per:
            print("#  per FADD2 (two pairs): %g FMNMX3 besides the 2 per triangle of the set-up" % ((c["FMNMX3"] - 2 * per) / fadd2))
    if hot:
        first = max(hot, key=lambda b: sum(op == "FADD2" for op, _ in b))
        print("## the widest block's first %d instructions (about one triangle)" % (len(first) // per))
        for _, ln in first[: len(first) // per]:
            print("        " + ln)


if __name__ == "__main__":
    main()
