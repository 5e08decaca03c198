"""Per-kernel SASS comparison of two builds of libnmfk_b200.so (cuobjdump -sass, instructions only, addresses dropped).

    python tools/sass_compare.py OLD.so NEW.so [-v]

Kernels are matched by demangled name; a kernel of OLD that gained a trailing defaulted template flag (bool DIV = false) is
matched with its <..., false> instantiation in NEW.  -v also lists the kernels that are new in NEW.
"""
import re, subprocess, sys
def demangle(names):
    return subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout.splitlines()
def funcs(lib):
    out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", lib], capture_output=True, text=True).stdout
    d = {}; cur = None
    for line in out.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m: cur = m.group(1); d.setdefault(cur, []); continue
        if cur and re.search(r"/\*[0-9a-f]{4,}\*/", line):
            d[cur].append(re.sub(r"/\*[0-9a-f]{4,}\*/", "", line).rstrip())
    return dict(zip(demangle(list(d)), d.values()))
a = funcs(sys.argv[1]); b = funcs(sys.argv[2])
bd = {x: x for x in b}
ad = {x: x for x in a}
same, changed, missing, matched = 0, [], [], set()
for f, dem in ad.items():
    g = f if f in b else None
    if g is None:  # <..., X>(args) -> <..., X, false>(args)
        alt = re.sub(r">\((.*)\)$", r", false>(\1)", dem)
        g = bd.get(alt)
    if g is None: missing.append(dem); continue
    matched.add(g)
    (same := same + 1) if a[f] == b[g] else changed.append(dem)
print("parent kernels: %d, identical SASS: %d, changed: %d, missing: %d, new in this build: %d" %
      (len(a), same, len(changed), len(missing), len(b) - len(matched)))
for x in changed: print("CHANGED", x)
for x in missing: print("MISSING", x)
if "-v" in sys.argv:
    for x in [g for g in b if g not in matched]: print("NEW", x)
