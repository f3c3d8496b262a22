"""Developer helper: compare the SASS of two builds of liboptistate_kf.so function by function, and the -Xptxas -v registers and
spills of the direct-load kernels (kf_seq_kernel, kf_seq_direct.cu) of the two trees.  For a refactor that must leave the
generated code alone: every function that should not change is reported identical or listed with its instruction counts.

    python tools/sass_diff.py OLD_ROOT NEW_ROOT [--out FILE]

Each ROOT is a source tree whose optistate_b200/_lib/liboptistate_kf.so has been built (python -m optistate_b200._build).
Instruction addresses and encodings are dropped before comparing; the code itself carries no build paths."""
import argparse
import os
import re
import subprocess
import sys
import tempfile

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC"]


def sass_functions(path):
    """{function: [instructions]} of a library or cubin; the hash in the names of anonymous namespaces follows from the source
    path, so it is dropped"""
    out = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True, check=True).stdout
    out = re.sub(r"_GLOBAL__N__[0-9a-f_]+", "_GLOBAL__N_", out)
    funcs = {}
    for chunk in re.split(r"\n\s*Function : ", out)[1:]:
        name, body = chunk.split("\n", 1)
        ins = []
        for line in body.split("\n"):
            m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(.*?)\s*;?\s*(?:/\*.*)?$", line)
            if m:
                ins.append(re.sub(r"\s+", " ", m.group(1)))
        funcs[name.strip()] = ins
    return funcs


def demangle(names):
    out = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout.strip().split("\n")
    return dict(zip(names, out))


def ptxas_direct(root):
    """registers and spill bytes of every entry of kf_seq_direct.cu"""
    with tempfile.TemporaryDirectory() as tmp:
        src = os.path.join(root, "optistate_b200", "csrc", "kf_seq_direct.cu")
        r = subprocess.run(["nvcc", *NVCC_FLAGS, "-Xptxas", "-v", "-c", "-o", os.path.join(tmp, "a.o"), src],
                           capture_output=True, text=True, check=True)
    res, cur = {}, None
    for line in r.stderr.split("\n"):
        m = re.search(r"Compiling entry function '(\S+)'", line)
        if m:
            cur = m.group(1)
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and cur:
            res.setdefault(cur, {})["spill"] = (int(m.group(1)), int(m.group(2)))
        m = re.search(r"Used (\d+) registers", line)
        if m and cur:
            res.setdefault(cur, {})["reg"] = int(m.group(1))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("old")
    ap.add_argument("new")
    ap.add_argument("--out")
    a = ap.parse_args()
    lib = lambda root: os.path.join(root, "optistate_b200", "_lib", "liboptistate_kf.so")
    old, new = sass_functions(lib(a.old)), sass_functions(lib(a.new))
    dem = demangle(sorted(set(old) | set(new)))
    lines, changed = [], []
    same = [n for n in old if n in new and old[n] == new[n]]
    only = sorted(set(old) ^ set(new))
    for n in sorted(set(old) & set(new), key=lambda n: dem[n]):
        if old[n] != new[n]:
            changed.append(n)
    tma = [n for n in old if "kf_seq_tma_kernel" in n]
    lines.append(f"functions: {len(old)} old, {len(new)} new; identical {len(same)}; changed {len(changed)}; in one build only {len(only)}")
    lines.append(f"kf_seq_tma_kernel instantiations: {len(tma)}, identical {sum(1 for n in tma if n in same)}")
    lines.append(f"functions outside kf_seq_kernel: {sum(1 for n in old if 'kf_seq_kernel' not in n)}, "
                 f"identical {sum(1 for n in same if 'kf_seq_kernel' not in n)}")
    for n in only:
        lines.append(f"  only in {'old' if n in old else 'new'}: {dem[n]}")
    lines.append("")
    lines.append("changed functions (instructions old -> new):")
    for n in changed:
        lines.append(f"  {len(old[n]):6d} -> {len(new[n]):6d}  {dem[n]}")
    lines.append("")
    po, pn = ptxas_direct(a.old), ptxas_direct(a.new)
    pdem = demangle(sorted(set(po) | set(pn)))
    lines.append("kf_seq_kernel (-Xptxas -v): registers, spill stores / loads bytes, old -> new")
    for n in sorted(set(po) | set(pn), key=lambda n: pdem[n]):
        o, w = po.get(n, {}), pn.get(n, {})
        short = re.sub(r"\(okf::.*", "", pdem[n]).replace("void ", "").replace("okf::", "")
        lines.append(f"  {short:60s} reg {o.get('reg')} -> {w.get('reg')}   spill {o.get('spill')} -> {w.get('spill')}")
    text = "\n".join(lines) + "\n"
    if a.out:
        open(a.out, "w").write(text)
    sys.stdout.write(text)


if __name__ == "__main__":
    main()
