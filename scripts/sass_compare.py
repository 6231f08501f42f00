"""Per-kernel SASS of two builds: every kernel of the BASE build must be instruction-identical in the NEW one.

    python scripts/sass_compare.py <base build dir> <new build dir>      (directories of *.cu.o, e.g. depthdensifier_b200/build)

Kernels are matched by name.  A `kRagged = false` instantiation (trailing `kRagged` template argument and `const int64_t*
layout` parameter: K3, K4) whose name the base build lacks is compared with the base kernel of its pre-ragged name, so a
base from before the ragged layout can be checked too; kernels only the new build has are listed as NEW, and base kernels
the new build no longer has (a deleted source or kernel) as GONE.  Every *.cu.o of either directory is read.  The exit status checks the kernels both builds have."""
import os, re, subprocess, sys
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
def norm(name):  # new uniform instantiation -> the pre-ragged name
    return re.sub(r", false>\(", ">(", name).replace(", long const*)", ")")
base, new = sys.argv[1], sys.argv[2]
tot = same = gone = 0
for src in sorted({f for d in (base, new) for f in os.listdir(d) if f.endswith(".cu.o")}):
    a, b = (funcs(f"{d}/{src}") if os.path.exists(f"{d}/{src}") else {} for d in (base, new))
    pre_ragged = {norm(k): k for k in b if k not in a and k.endswith(", long const*)") and ", false>(" in k}
    matched = set()
    for name, ins in a.items():
        twin = name if name in b else pre_ragged.get(name)
        if twin is None:
            print("GONE", src, name, len(ins)); gone += 1; continue
        tot += 1
        matched.add(twin)
        if b.get(twin) == ins: same += 1
        else: print("DIFF", src, name, len(ins), len(b.get(twin, [])))
    for name in b:
        if name not in matched: print("NEW ", src, name, len(b[name]))
print(f"{same}/{tot} base kernels instruction-identical, {gone} gone")
sys.exit(0 if same == tot else 1)
