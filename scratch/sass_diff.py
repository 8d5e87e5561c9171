"""Function-by-function comparison of two builds of the library, without a GPU.

    python scratch/sass_diff.py OLD.sass NEW.sass [OLD_ptxas.log NEW_ptxas.log]

The .sass files are `cuobjdump -sass libpytracer_b200.so`; the logs are the build output with
RT_EXTRA_FLAGS="-Xptxas -v".  Prints, per kernel, whether its SASS is identical (addresses stripped), and the
registers and spill bytes of every kernel whose SASS or resources differ."""
import re
import subprocess
import sys


def functions(path):
    out, name, body = {}, None, []
    for line in open(path):
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            if name:
                out[name] = body
            name, body = m.group(1), []
        elif name:
            s = " ".join(re.sub(r"/\*[0-9a-f]{4,}\*/", "", line).split())  # instruction addresses; column widths
            if s and not s.startswith("/* 0x"):
                body.append(s)
    if name:
        out[name] = body
    return out


def resources(path):
    res, name = {}, None
    for line in open(path):
        m = re.search(r"Function properties for (\S+)", line)
        if m:
            name = m.group(1)
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and name:
            res.setdefault(name, {})["spill"] = f"{m.group(1)}/{m.group(2)} B"
        m = re.search(r"Compiling entry function '(\S+)'", line)
        if m:
            name = m.group(1)
        m = re.search(r"Used (\d+) registers", line)
        if m and name:
            res.setdefault(name, {})["regs"] = int(m.group(1))
    return res


def demangle(n):
    return subprocess.run(["c++filt", n], capture_output=True, text=True).stdout.strip()


old, new = functions(sys.argv[1]), functions(sys.argv[2])
ro, rn = (resources(sys.argv[3]), resources(sys.argv[4])) if len(sys.argv) > 4 else ({}, {})
same = [n for n in old if n in new and old[n] == new[n]]
print(f"{len(same)} of {len(old)} kernels identical; only in old: {sorted(set(old) - set(new))}; "
      f"only in new: {sorted(set(new) - set(old))}")
for n in sorted(set(old) & set(new)):
    if old[n] != new[n] or ro.get(n) != rn.get(n):
        print(f"differs: {demangle(n)}: {len(old[n])} -> {len(new[n])} instructions; "
              f"registers / spill stores/loads {ro.get(n)} -> {rn.get(n)}")
