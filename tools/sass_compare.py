"""Compare per-kernel SASS (addresses, immediates and constant-bank offsets masked) and ptxas resource lines of two builds.

    python tools/sass_compare.py [--same-names] BASE_DIR NEW_DIR candidates_tc pack exact local

Each directory holds <name>.sass (cuobjdump -sass <name>.o) and <name>.ptxas.txt (nvcc -Xptxas -v output) per translation
unit.  Kernels are matched by demangled name; a trailing `, false>` template argument of the new tc_candidates_kernel (the
K-streamed flag) and pack_operands_kernel<5> are mapped to the parent's names, unless --same-names (both builds have the same
template arguments: kernels are matched by their names as they are)."""
import re, subprocess, sys, collections
args = sys.argv[1:]
same_names = "--same-names" in args
if same_names:
    args.remove("--same-names")
base, new = args[0], args[1]
def demangle(names):
    out = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout.splitlines()
    return dict(zip(names, out))
def sass(path):
    funcs, cur = collections.OrderedDict(), None
    for line in open(path):
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1); funcs[cur] = []; continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(.*?);", line)
        if m and cur:
            ins = re.sub(r"0x[0-9a-f]+", "IMM", m.group(1))
            ins = re.sub(r"c\[IMM\]\[(IMM|URZ)\]", "c[IMM][IMM]", ins).strip()   # constant-bank offsets: relocated string addresses
            funcs[cur].append(ins)
    return funcs
def ptxas(path):
    res, cur = {}, None
    lines = open(path).read().splitlines()
    for i, l in enumerate(lines):
        m = re.match(r"ptxas info\s+: Function properties for (\S+)", l)
        if m:
            cur = m.group(1); res[cur] = [lines[i + 1].strip()]
        m = re.match(r"ptxas info\s+: Used (.*)", l)
        if m and cur:
            res[cur].append("Used " + m.group(1)); cur = None
    return res
def norm(n, new=False):
    n = n.replace("(anonymous namespace)::", "")
    n = re.sub(r"^void ", "", n)
    n = re.sub(r"\(.*", "", n)
    if same_names:
        return n
    if new:
        n = re.sub(r"tc_candidates_kernel<(.*), false>$", r"tc_candidates_kernel<\1>", n)
    n = n.replace("pack_operands_kernel<5>", "pack_operands_kernel")
    return n
for obj in args[2:]:
    print("## %s.cu" % obj)
    b, n = sass("%s/%s.sass" % (base, obj)), sass("%s/%s.sass" % (new, obj))
    pb, pn = ptxas("%s/%s.ptxas.txt" % (base, obj)), ptxas("%s/%s.ptxas.txt" % (new, obj))
    db, dn = demangle(list(b) + list(pb)), demangle(list(n) + list(pn))
    nb = {norm(db[k]): k for k in b}; nn = {norm(dn[k], True): k for k in n}
    pnb = {norm(db[k]): v for k, v in pb.items()}; pnn = {norm(dn[k], True): v for k, v in pn.items()}
    same = 0
    for name in sorted(nb):
        if name not in nn:
            print("MISSING in new: %s" % name); continue
        x, y = b[nb[name]], n[nn[name]]
        rb, rn = pnb.get(name), pnn.get(name)
        ok = x == y and rb == rn
        same += ok
        print("%-100s instr %5d -> %5d %s | %s" % (name[:100], len(x), len(y), "SASS identical" if x == y else "SASS DIFFERS",
                                                 ("; ".join(rn or []) if rb == rn else "RESOURCES DIFFER: %s -> %s" % (rb, rn))))
    extra = sorted(set(nn) - set(nb))
    print("existing instantiations identical: %d of %d; new instantiations: %d" % (same, len(nb), len(extra)))
    for e in extra:
        print("  new: %-100s instr %5d | %s" % (e[:100], len(n[nn[e]]), "; ".join(pnn.get(e, []))))
