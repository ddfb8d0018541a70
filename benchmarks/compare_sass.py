"""Compare the kernels of two builds of libouzelum_b200.so without a GPU: for a change that must not alter the code of the
kernels it keeps.  `python benchmarks/compare_sass.py BEFORE.so AFTER.so`

For every kernel (by mangled name) it reports whether it exists in both builds, whether REG / SHARED / STACK / LOCAL from
`cuobjdump -res-usage` agree, and whether the opcode sequences from `cuobjdump -sass` agree (mnemonics with their modifiers,
in order; predicates and operands stripped, so moved kernel-parameter offsets in the constant bank do not count).
Exit status 1 if a kernel present in both differs.
"""
import os
import re
import subprocess
import sys

CUOBJDUMP = os.path.join(os.path.dirname(os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")), "cuobjdump")
RES_KEYS = ("REG", "SHARED", "STACK", "LOCAL")


def res_usage(lib):
    out = subprocess.run([CUOBJDUMP, "-res-usage", lib], capture_output=True, text=True, check=True).stdout
    res, name = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function (\S+):$", line)
        if m:
            name = m.group(1)
        elif name and "REG:" in line:
            fields = dict(kv.split(":", 1) for kv in line.split())
            res[name] = tuple(fields[k] for k in RES_KEYS)
            name = None
    return res


def opcodes(lib):
    out = subprocess.run([CUOBJDUMP, "-sass", lib], capture_output=True, text=True, check=True).stdout
    ops, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)$", line)
        if m:
            cur = ops.setdefault(m.group(1), [])
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\w+\s+)?([A-Z][A-Z0-9_.]*)", line)
        if m and cur is not None:
            cur.append(m.group(1))
    return ops


def main(before, after):
    rb, ra = res_usage(before), res_usage(after)
    ob, oa = opcodes(before), opcodes(after)
    gone = sorted(set(ob) - set(oa))
    new = sorted(set(oa) - set(ob))
    common = sorted(set(ob) & set(oa))
    bad = 0
    print(f"kernels: {len(ob)} before, {len(oa)} after, {len(common)} in both")
    for k in gone:
        print(f"  only before: {k}")
    for k in new:
        print(f"  only after:  {k}")
    for k in common:
        same_res, same_ops = rb.get(k) == ra.get(k), ob[k] == oa[k]
        if not (same_res and same_ops):
            bad += 1
            print(f"  DIFFERS {k}: resources {rb.get(k)} -> {ra.get(k)}, opcodes {len(ob[k])} -> {len(oa[k])}"
                  f"{'' if same_ops else ' (sequence differs)'}")
    print(f"{len(common) - bad} of {len(common)} common kernels have the same {'/'.join(RES_KEYS)} and opcode sequence")
    return 1 if bad else 0


if __name__ == "__main__":
    if len(sys.argv) != 3:
        sys.exit(__doc__)
    sys.exit(main(sys.argv[1], sys.argv[2]))
