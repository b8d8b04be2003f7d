#!/usr/bin/env python3
"""SASS summary of the hot kernels in libb2rt.so (cuobjdump -sass): instruction count, opcode histogram, the 128-bit
read-only global loads, local-memory traffic instructions and the registers / stack / shared memory of each kernel.
DESIGN.md's instruction-count arguments are made from this file.
Usage: python profiles/sass_summary.py [out.json]   (no GPU needed)"""
import collections
import json
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "mini-opencl-raytracer_b200", "libb2rt.so")
# the hit policy of trace_persistent is its first template argument: 0 closest, 1 any-hit, 2 multi (traverse.cuh HIT_*)
KERNELS = {
    "trace_persistent<closest, no counters, CAP 64>": "trace_persistentILi0ELb0ELi64E",
    "trace_persistent<any-hit, no counters, CAP 64>": "trace_persistentILi1ELb0ELi64E",
    "trace_persistent<multi, no counters, CAP 64>": "trace_persistentILi2ELb0ELi64E",
    "trace_tail_kernel<closest, no counters>": "trace_tail_kernelILb0ELb0E",
    # frame instantiations (STREAM = false) under the row names they had before the kernels took the STREAM argument
    "wf_shade_kernel": "wf_shade_kernelILb0E",
    "wf_generate_kernel": "wf_generate_kernelILb0E",
    "render_mega_kernel<wide, CAP 64>": "render_mega_kernelILb0ELi64ELb0E",
    "wf_shade_kernel<radiance stream>": "wf_shade_kernelILb1E",
    "wf_generate_kernel<radiance stream>": "wf_generate_kernelILb1E",
    "render_mega_kernel<wide, CAP 64, radiance stream>": "render_mega_kernelILb0ELi64ELb1E",
    "render_mega_kernel<binary, CAP 64, radiance stream>": "render_mega_kernelILb1ELi64ELb1E",
    "point_persistent<no counters, CAP 64>": "point_persistentILb0ELi64E",
    "point_binary_kernel<CAP 64>": "point_binary_kernelILi64E",
}


def main(out):
    sass = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True, check=True).stdout
    res = subprocess.run(["cuobjdump", "-res-usage", LIB], capture_output=True, text=True, check=True).stdout
    usage = {}
    for m in re.finditer(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+) SHARED:(\d+) LOCAL:(\d+)", res):
        usage[m.group(1)] = {"registers": int(m.group(2)), "stack_bytes": int(m.group(3)), "shared_bytes": int(m.group(4))}
    arch = re.search(r"arch = (sm_\w+)", sass)
    blocks = re.split(r"\n\s*Function : ", sass)
    summary = {"library": os.path.relpath(LIB, ROOT), "arch": arch.group(1) if arch else None, "kernels": {}}
    for title, key in KERNELS.items():
        body = next((b for b in blocks if b.split("\n", 1)[0].find(key) >= 0), None)
        if body is None:
            continue
        name = body.split("\n", 1)[0].strip()
        ops = collections.Counter()
        for line in body.splitlines():
            m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", line)
            if m:
                ops[m.group(1)] += 1
        base = collections.Counter()
        for op, c in ops.items():
            base[op.split(".")[0]] += c
        summary["kernels"][title] = {
            "symbol": name, **usage.get(name, {}),
            "instructions": sum(ops.values()),
            "LDG.E.128.CONSTANT": sum(c for op, c in ops.items() if op.startswith("LDG.E.128.CONSTANT")),
            "LDG_other": sum(c for op, c in ops.items() if op.startswith("LDG") and not op.startswith("LDG.E.128.CONSTANT")),
            "STG": base.get("STG", 0), "local_memory_ops (LDL+STL)": base.get("LDL", 0) + base.get("STL", 0),
            "tensor_core_or_tma_ops": sum(c for op, c in ops.items() if op.startswith(("UTC", "UTMA", "HMMA", "IMMA", "QMMA"))),
            "top_opcodes": dict(base.most_common(16)),
        }
    with open(out, "w") as f:
        json.dump(summary, f, indent=1)
    print(json.dumps(summary, indent=1))


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r2_sass_summary.json"))
