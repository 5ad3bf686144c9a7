"""Compare the SASS of every solve-kernel instantiation of two builds of libcmpc.so, matching them by
their template arguments without the trailing BODY flag; print resource usage of each BODY twin."""
import re, subprocess, sys
CUDA = "/usr/local/cuda/bin/"

def funcs(lib):
    out = subprocess.run([CUDA + "cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    parts = re.split(r"\n\s+Function : (\S+)\n", out)
    res = {}
    for i in range(1, len(parts), 2):
        body = parts[i + 1].split("\n\t\t.......")[0]
        # drop addresses/comments: keep instruction text only
        ins = [re.sub(r"/\*[0-9a-f]{4,}\*/", "", l).strip() for l in body.splitlines() if "/*" in l]
        res[parts[i]] = "\n".join(ins)
    return res

def demangle(names):
    out = subprocess.run([CUDA + "cu++filt"], input="\n".join(names), capture_output=True, text=True).stdout
    return dict(zip(names, out.splitlines()))

def key(dm, drop_last):
    m = re.match(r"void cmpc::(solve_kernel|solve_riccati_kernel)<(.*)>\(cmpc::SolveParams\)", dm)
    if not m:
        return None, None
    args = [a.strip() for a in m.group(2).split(",")]
    body = None
    if drop_last:
        body = args[-1]
        args = args[:-1]
    return m.group(1) + "<" + ", ".join(args) + ">", body

base, new = funcs(sys.argv[1]), funcs(sys.argv[2])
db, dn = demangle(list(base)), demangle(list(new))
bk = {key(db[n], False)[0]: n for n in base if key(db[n], False)[0]}
nk = {}
for n in new:
    k, b = key(dn[n], True)
    if k:
        nk[(k, b)] = n
same = diff = 0
for k, n in sorted(bk.items()):
    m = nk.get((k, "(bool)0"))
    if m is None:
        print("MISSING", k); diff += 1; continue
    if base[n] == new[m]:
        same += 1
    else:
        diff += 1; print("DIFFERS", k)
    if (k, "(bool)1") not in nk:
        print("NO BODY TWIN", k)
print(f"{same} of {len(bk)} parent instantiations have identical SASS, {diff} differ or are missing; "
      f"{sum(1 for (_, b) in nk if b == "(bool)1")} BODY twins")
