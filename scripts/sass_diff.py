#!/usr/bin/env python3
"""Compare the SASS and resource usage of two builds, kernel by kernel.

    python -m vfclik_b200.build --out=/tmp/a/libvfk_parent.so     # objects in build/obj/libvfk_parent/
    python -m vfclik_b200.build --out=/tmp/b/libvfk_change.so     # objects in build/obj/libvfk_change/
    python scripts/sass_diff.py build/obj/libvfk_parent build/obj/libvfk_change

For every kernel of every object file present in either directory it prints one line: `same` when the instruction sequence
is identical once addresses, branch targets and encodings are stripped (`diff` otherwise), the instruction count on each
side, and REG / STACK / SHARED / LOCAL from `cuobjdump -res-usage` on each side.  A summary follows, with every kernel
whose STACK or LOCAL grew.  Runs cuobjdump only; no GPU is needed.
"""
import argparse
import os
import re
import shutil
import subprocess
import sys

RES_KEYS = ("REG", "STACK", "SHARED", "LOCAL")
INSN = re.compile(r"^\s+/\*[0-9a-f]{4,}\*/\s+(.*?)\s*;")
BRANCH = re.compile(r"^(@!?U?P\w+\s+)?(BRA|BRX|BSSY|CALL|JMP|JMX|RET|BREAK|BPT)\b")


def tool(name):
    path = shutil.which(name) or os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", name)
    if not os.path.exists(path):
        sys.exit("%s not found (put the CUDA toolkit's bin/ on PATH or set CUDA_HOME)" % name)
    return path


def run(*cmd):
    return subprocess.run(cmd, check=True, stdout=subprocess.PIPE, text=True).stdout


def sass(obj):
    """{mangled name: [instruction text]} with addresses and encodings dropped and branch targets replaced."""
    out, cur = {}, None
    for line in run(tool("cuobjdump"), "-sass", obj).splitlines():
        if "Function : " in line:
            cur = out.setdefault(line.split("Function : ", 1)[1].strip(), [])
            continue
        m = INSN.match(line)
        if m and cur is not None:
            text = " ".join(m.group(1).split())
            if BRANCH.match(text):
                text = re.sub(r"0x[0-9a-f]+", "<target>", text)
            cur.append(text)
    return out


def resources(obj):
    """{mangled name: {REG, STACK, SHARED, LOCAL}}"""
    out, cur = {}, None
    for line in run(tool("cuobjdump"), "-res-usage", obj).splitlines():
        line = line.strip()
        if line.startswith("Function "):
            cur = line[len("Function "):].rstrip(":")
        elif cur and line.startswith("REG:"):
            fields = dict(f.split(":", 1) for f in line.split())
            out[cur] = {k: int(fields[k]) for k in RES_KEYS}
            cur = None
    return out


def demangle(names):
    if not names:
        return {}
    lines = subprocess.run([tool("cu++filt")], input="\n".join(names), check=True, stdout=subprocess.PIPE, text=True).stdout
    return dict(zip(names, lines.splitlines()))


def load(directory):
    """{(object file, mangled name): (instructions, resources)}"""
    kernels = {}
    for f in sorted(os.listdir(directory)):
        if not f.endswith(".o"):
            continue
        path = os.path.join(directory, f)
        code, res = sass(path), resources(path)
        for name, insns in code.items():
            kernels[(f, name)] = (insns, res.get(name, {}))
    return kernels


def fmt_res(r):
    return " ".join("%s %s" % (k, r.get(k, "?")) for k in RES_KEYS)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("a", help="object directory of the first build (the reference)")
    ap.add_argument("b", help="object directory of the second build")
    ap.add_argument("--changed", action="store_true", help="list only the kernels whose instructions or resources differ")
    args = ap.parse_args()
    A, B = load(args.a), load(args.b)
    keys = sorted(set(A) | set(B))
    names = demangle(sorted({k[1] for k in keys}))
    same = diff = res_changed = 0
    grew, only = [], []
    for key in keys:
        label = "%s %s" % (key[0], names.get(key[1], key[1]))
        if key not in A or key not in B:
            only.append(key)
            print("only in %s: %s" % ("b" if key in B else "a", label))
            continue
        (ia, ra), (ib, rb) = A[key], B[key]
        identical = ia == ib
        same += identical
        diff += not identical
        res_changed += ra != rb
        if any(rb.get(k, 0) > ra.get(k, 0) for k in ("STACK", "LOCAL")):
            grew.append(label)
        if args.changed and identical and ra == rb:
            continue
        print("%-4s insns %6d -> %6d  | %s -> %s | %s" % ("same" if identical else "diff", len(ia), len(ib), fmt_res(ra), fmt_res(rb),
                                                        label))
    print("\n%d kernels in a, %d in b, %d only on one side; %d identical instruction sequences, %d differ; %d with changed "
          "resources" % (len(A), len(B), len(only), same, diff, res_changed))
    for label in grew:
        print("STACK or LOCAL grew: %s" % label)


if __name__ == "__main__":
    main()
