"""Compare the kernels of two sm_100a builds of auv_kernels.cu: ptxas resource lines and SASS.

    nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -cubin -Xptxas -v \
         -o X.cubin gym_auv_b200/csrc/auv_kernels.cu 2> X_ptxas.txt          (for the parent and the branch)
    python tools/sass_compare.py parent.cubin parent_ptxas.txt branch.cubin branch_ptxas.txt

Kernels are matched by their demangled name with a trailing ``, false>`` template argument removed
(a defaulted template parameter appended to a kernel renames its existing instantiations).  SASS is
compared after constant-bank operands ``c[0x0][0x...]`` (kernel parameters) are normalised, and after
the comment / address columns are dropped.  Prints one line per kernel and a summary."""
from __future__ import annotations

import re
import subprocess
import sys


def demangle(names):
    out = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout.split("\n")
    return dict(zip(names, out))


def key(dem: str) -> str:
    dem = re.sub(r"\(.*\)$", "", dem)
    return re.sub(r"k_lidar<(\w+), (\w+), (\w+), false>", r"k_lidar<\1, \2, \3>", dem)


def ptxas(path):
    res, cur = {}, None
    for line in open(path):
        m = re.search(r"Compiling entry function '(\w+)'", line)
        if m:
            cur = m.group(1)
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and cur:
            res.setdefault(cur, {})["spill"] = (int(m.group(1)), int(m.group(2)))
        m = re.search(r"Used (\d+) registers.*?(?:(\d+) bytes smem)?", line)
        if m and cur:
            res.setdefault(cur, {})["regs"] = int(m.group(1))
            sm = re.search(r"(\d+) bytes smem", line)
            res[cur]["smem"] = int(sm.group(1)) if sm else 0
    return res


def sass(cubin):
    txt = subprocess.run(["cuobjdump", "-sass", cubin], capture_output=True, text=True, check=True).stdout
    fns, cur = {}, None
    for line in txt.split("\n"):
        m = re.match(r"\s+Function : (\w+)", line)
        if m:
            cur = m.group(1)
            fns[cur] = []
            continue
        if cur is None:
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(.*?);", line)
        if m:
            ins = re.sub(r"c\[0x0\]\[0x[0-9a-f]+\]", "c[0x0][P]", m.group(1))
            fns[cur].append(ins)
    return fns


def main(a_cubin, a_ptxas, b_cubin, b_ptxas):
    pa, pb = ptxas(a_ptxas), ptxas(b_ptxas)
    sa, sb = sass(a_cubin), sass(b_cubin)
    da, db = demangle(sorted(set(pa) | set(sa))), demangle(sorted(set(pb) | set(sb)))
    ka = {key(da[n]): n for n in da}
    kb = {key(db[n]): n for n in db}
    same = changed = 0
    for k in sorted(set(ka) | set(kb)):
        na, nb = ka.get(k), kb.get(k)
        rb = pb.get(nb, {}) if nb else {}
        res = f"{rb.get('regs')} registers, {rb.get('smem', 0)} bytes smem, spill stores/loads " \
              f"{'/'.join(map(str, rb.get('spill', (0, 0))))} bytes"
        if na is None:
            print(f"{k}: {res}  (new)")
            continue
        if nb is None:
            print(f"{k}: removed")
            continue
        ra = pa.get(na, {})
        same_res = (ra.get("regs"), ra.get("smem", 0), ra.get("spill", (0, 0))) == \
                   (rb.get("regs"), rb.get("smem", 0), rb.get("spill", (0, 0)))
        same_sass = sa.get(na) == sb.get(nb)
        if same_res and same_sass:
            same += 1
        else:
            changed += 1
        print(f"{k}: {res}  ptxas {'same' if same_res else 'CHANGED from ' + str(ra)}, "
              f"SASS {'identical' if same_sass else 'DIFFERS'} ({len(sb.get(nb, []))} instructions, "
              f"parameter offsets normalised)")
    print(f"# existing entry functions: {same} identical, {changed} changed")


if __name__ == "__main__":
    main(*sys.argv[1:5])
