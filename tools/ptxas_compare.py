"""Per-kernel registers, spills, stack and shared memory of two -Xptxas -v logs (the Makefile keeps them in
raytracerwin_b200/csrc/build/ptxas*.log), matched by mangled name with nvcc's per-build hash of anonymous namespaces
removed (it depends on the source's path, so trees built in different directories compare too).  Prints every kernel
of the first log with its line in the second and whether it changed or is gone, then kernels only the second log has.

   python tools/ptxas_compare.py OLD.log NEW.log
"""
import re
import sys


def parse(path):
    out, cur = {}, None
    for line in open(path):
        m = re.search(r"Compiling entry function '(\S+)'", line)
        if m:
            cur = re.sub(r"(_cu_|_GLOBAL__N__)[0-9a-f]{8}", r"\1", m.group(1))
            out[cur] = []
        elif cur and ("Used" in line or "spill" in line) and "Function properties" not in line:
            out[cur].append(re.sub(r"^ptxas info\s*:\s*", "", line.strip()))
    return {k: "; ".join(v) for k, v in out.items()}


def main(old, new):
    A, B = parse(old), parse(new)
    changed = removed = 0
    for k in A:
        if k not in B:
            removed += 1
            print(f"removed {k}: {A[k]}")
            continue
        same = A[k] == B[k]
        changed += not same
        print(f"{'same   ' if same else 'CHANGED'} {k}: {A[k]}" + ("" if same else f"  ->  {B[k]}"))
    for k in B:
        if k not in A:
            print(f"new     {k}: {B[k]}")
    print(f"{len(A)} kernels compared, {changed} changed, {removed} removed, {sum(k not in A for k in B)} new")
    return changed + removed


if __name__ == "__main__":
    sys.exit(1 if main(sys.argv[1], sys.argv[2]) else 0)
