"""Per-kernel SASS of two builds: every kernel of the BASE build must be instruction-identical in the NEW one.

    python scripts/sass_compare.py <base build dir> <new build dir>      (directories of *.cu.o, e.g. depthdensifier_b200/build)

Kernels that gained a trailing `kRagged` template argument and a trailing `const int64_t* layout` parameter (K3, K4) are
matched to their old names with `kRagged = false`; kernels only the new build has are listed as NEW."""
import re, subprocess, sys
def funcs(obj):
    out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", obj], capture_output=True, text=True, check=True).stdout
    d, cur = {}, None
    for ln in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", ln)
        if m:
            cur = subprocess.run(["c++filt", m.group(1)], capture_output=True, text=True).stdout.strip(); d[cur] = []; continue
        if cur and re.match(r"\s*/\*[0-9a-f]{4,}\*/", ln):
            d[cur].append(re.sub(r"\s+", " ", ln.strip()))
    return d
def norm(name):  # new uniform instantiation -> the parent's name
    return re.sub(r", false>\(", ">(", name).replace(", long const*)", ")")
base, new = sys.argv[1], sys.argv[2]
tot = same = 0
for src in ["align.cu.o", "filter.cu.o", "fuse.cu.o", "fuse_sort.cu.o", "api.cu.o", "geometry.cu.o", "pchip.cu.o", "masks.cu.o"]:
    a = funcs(f"{base}/{src}")
    b = {}
    for k, v in funcs(f"{new}/{src}").items():
        b.setdefault(norm(k) if k.endswith(", long const*)") and ", false>(" in k else k, v)
    for name, ins in a.items():
        tot += 1
        if b.get(name) == ins: same += 1
        else: print("DIFF", src, name, len(ins), len(b.get(name, [])))
    for name in b:
        if name not in a: print("NEW ", src, name, len(b[name]))
print(f"{same}/{tot} base kernels instruction-identical")
sys.exit(0 if same == tot else 1)
