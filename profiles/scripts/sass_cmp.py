"""Compare per-kernel SASS of two cuobjdump -sass listings, ignoring the anonymous-namespace hash in the names and the
instruction addresses; the new listing's default RES=false kernels carry an extra `Lb0E` template argument."""
import re, sys
def funcs(path):
    out, cur = {}, None
    for line in open(path):
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = re.sub(r"_GLOBAL__N__[0-9a-f]+_", "_GLOBAL__N__X_", m.group(1)); out[cur] = []; continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s*(.*?);", line)
        if cur and m:
            out[cur].append(m.group(1).strip())
    return out
a, b = funcs(sys.argv[1]), funcs(sys.argv[2])
for k, v in a.items():
    k2 = k.replace("ELi1EEEvNS0_", "ELi1ELb0EEEvNS0_") if "k_conv_umma" in k else k
    w = b.get(k2)
    tag = re.search(r"k_conv_\w+?E", k).group(0)
    print(f"{'IDENTICAL' if w == v else 'DIFFERENT'}  {len(v):6d} vs {len(w) if w else 0:6d} instructions  {k2}")
new = [k for k in b if "Lb1E" in k]
print(f"{len(new)} residual (RES=true) kernels, new")
