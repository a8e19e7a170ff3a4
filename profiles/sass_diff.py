"""Per-function SASS comparison of two object files (addresses and comments stripped)."""
import re, subprocess, sys
def funcs(obj):
    out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", obj], capture_output=True, text=True, check=True).stdout
    res, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            # anonymous-namespace names carry a per-compilation hash: drop it so both builds name a kernel alike
            cur = re.sub(r"_GLOBAL__N__[0-9a-f]+_", "_GLOBAL__N__", m.group(1)); res[cur] = []; continue
        if cur and re.match(r"\s*/\*[0-9a-f]{4}\*/", line):
            ins = re.sub(r"/\*[0-9a-f]{4}\*/", "", line).split(";")[0].strip()
            res[cur].append(ins)
    return res
# usage: sass_diff.py parent.o branch.o [pattern] [OLD=NEW ...]: each OLD=NEW renames the branch's functions
# (a kernel that gained a template argument whose default keeps the parent's code)
a, b = funcs(sys.argv[1]), funcs(sys.argv[2])
pat = sys.argv[3] if len(sys.argv) > 3 else ""
for sub in sys.argv[4:]:
    old, new = sub.split("=", 1)
    b = {k.replace(old, new): v for k, v in b.items()}
common = sorted(k for k in a if k in b and pat in k)
same = [k for k in common if a[k] == b[k]]
diff = [k for k in common if a[k] != b[k]]
print(f"parent functions {len(a)}, branch functions {len(b)}, compared (matching '{pat}') {len(common)}, identical {len(same)}, different {len(diff)}")
print("only in parent:", sorted(set(a) - set(b)))
print("only in branch:", sorted(k for k in set(b) - set(a)))
for k in diff: print("DIFF", k)
