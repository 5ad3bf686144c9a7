"""Compare the SASS of every solve-kernel instantiation of two builds of libcmpc.so.  Instantiations are matched by
their template arguments without the trailing feature flags (BODY, CONTACT, WEIGHTS; a build that predates a flag
has it false): the plain (0,0,0), BODY (1,0,0) and BODY + CONTACT (1,1,0) kernels of the second build against the
first build's, and the WEIGHTS twins (1,0,1) and (1,1,1) of the second build counted.
Usage: sass_twin_diff.py <base libcmpc.so> <new libcmpc.so>"""
import re, subprocess, sys
CUDA = "/usr/local/cuda/bin/"
CORE_ARGS = {"solve_kernel": 7, "solve_riccati_kernel": 2}   # template arguments before the feature flags

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

def key(dm):
    """(kernel<core arguments>, (BODY, CONTACT, WEIGHTS)) of a solve-kernel instantiation, or None"""
    m = re.match(r"void cmpc::(solve_kernel|solve_riccati_kernel)<(.*)>\(cmpc::SolveParams\)", dm)
    if not m:
        return None
    args = [a.strip() for a in m.group(2).split(",")]
    core = CORE_ARGS[m.group(1)]
    flags = tuple(int(a == "(bool)1") for a in args[core:])
    return m.group(1) + "<" + ", ".join(args[:core]) + ">", (flags + (0, 0, 0))[:3]

def table(lib):
    code = funcs(lib)
    dm = demangle(list(code))
    return {k: code[n] for n in code for k in [key(dm[n])] if k}

base, new = table(sys.argv[1]), table(sys.argv[2])
counts = {}
for flags, name in (((0, 0, 0), "plain"), ((1, 0, 0), "BODY"), ((1, 1, 0), "BODY+CONTACT")):
    ks = sorted(k for k in base if k[1] == flags)
    same = 0
    for k in ks:
        if k not in new:
            print("MISSING", name, k[0])
        elif base[k] != new[k]:
            print("DIFFERS", name, k[0])
        else:
            same += 1
    counts[name] = (same, len(ks))
twins = {f: sorted(k[0] for k in new if k[1] == f) for f in ((1, 1, 0), (1, 0, 1), (1, 1, 1))}
for k in sorted(k[0] for k in new if k[1] == (1, 0, 0)):
    for f, name in (((1, 1, 0), "CONTACT"), ((1, 0, 1), "WEIGHTS"), ((1, 1, 1), "CONTACT+WEIGHTS")):
        if k not in twins[f]:
            print("NO", name, "TWIN", k)
print("; ".join(f"{name}: {counts[name][0]} of {counts[name][1]}" for name in counts) +
      f" base instantiations have identical SASS; {len(twins[(1, 0, 1)])} BODY+WEIGHTS and "
      f"{len(twins[(1, 1, 1)])} BODY+CONTACT+WEIGHTS twins")
