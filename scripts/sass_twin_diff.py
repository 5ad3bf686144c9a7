"""Compare the SASS of two builds of libcmpc.so.

By default every solve-kernel instantiation, matched by its template arguments without the trailing feature flags
(BODY, CONTACT, WEIGHTS, FORCE, STAGE; a build that predates a flag has it false), with one count per feature set:
plain (0,0,0,0,0), BODY (1,0,0,0,0), BODY+CONTACT (1,1,0,0,0), BODY+WEIGHTS (1,0,1,0,0), BODY+CONTACT+WEIGHTS
(1,1,1,0,0), BODY+WEIGHTS+FORCE (1,0,1,1,0), BODY+CONTACT+WEIGHTS+FORCE (1,1,1,1,0), BODY+WEIGHTS+FORCE+STAGE
(1,0,1,1,1) and BODY+CONTACT+WEIGHTS+FORCE+STAGE (1,1,1,1,1).  With --all, every function of the two
libraries (score, condense, store, plant, assembly kernels too), matched by its mangled name, the solve kernels by
their template arguments and feature flags as above.
Prints MISSING for a function of OLD that NEW lacks, DIFFERS for one whose SASS changed and NEW for one only NEW has;
exits 1 on any MISSING or DIFFERS.
Usage: sass_twin_diff.py [--all] OLD.so NEW.so"""
import re, subprocess, sys
CUDA = "/usr/local/cuda/bin/"
CORE_ARGS = {"solve_kernel": 7, "solve_riccati_kernel": 2}   # template arguments before the feature flags
NFLAGS = 5
SETS = (((0, 0, 0, 0, 0), "plain"), ((1, 0, 0, 0, 0), "BODY"), ((1, 1, 0, 0, 0), "BODY+CONTACT"),
        ((1, 0, 1, 0, 0), "BODY+WEIGHTS"), ((1, 1, 1, 0, 0), "BODY+CONTACT+WEIGHTS"),
        ((1, 0, 1, 1, 0), "BODY+WEIGHTS+FORCE"), ((1, 1, 1, 1, 0), "BODY+CONTACT+WEIGHTS+FORCE"),
        ((1, 0, 1, 1, 1), "BODY+WEIGHTS+FORCE+STAGE"), ((1, 1, 1, 1, 1), "BODY+CONTACT+WEIGHTS+FORCE+STAGE"))

def funcs(lib):
    """mangled name -> SASS instruction text, one entry per copy (a function compiled into two modules has two)"""
    out = subprocess.run([CUDA + "cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    parts = re.split(r"\n\s+Function : (\S+)\n", out)
    res = {}
    for i in range(1, len(parts), 2):
        body = parts[i + 1].split("\n\t\t.......")[0]
        # drop addresses/comments: keep instruction text only
        ins = [re.sub(r"/\*[0-9a-f]{4,}\*/", "", l).strip() for l in body.splitlines() if "/*" in l]
        res.setdefault(parts[i], []).append("\n".join(ins))
    return res

def demangle(names):
    out = subprocess.run([CUDA + "cu++filt"], input="\n".join(names), capture_output=True, text=True).stdout
    return dict(zip(names, out.splitlines()))

def key(dm):
    """(kernel<core arguments>, (BODY, CONTACT, WEIGHTS, FORCE, STAGE)) of a solve-kernel instantiation, or None"""
    m = re.match(r"void cmpc::(solve_kernel|solve_riccati_kernel)<(.*)>\(cmpc::SolveParams\)", dm)
    if not m:
        return None
    args = [a.strip() for a in m.group(2).split(",")]
    core = CORE_ARGS[m.group(1)]
    flags = tuple(int(a == "(bool)1") for a in args[core:])
    return m.group(1) + "<" + ", ".join(args[:core]) + ">", (flags + (0,) * NFLAGS)[:NFLAGS]

def solve_kernels(code):
    dm = demangle(list(code))
    return {k: code[n] for n in code for k in [key(dm[n])] if k}

def compare(base, new, label):
    """prints MISSING / DIFFERS / NEW lines; returns (identical, compared, new only)"""
    same = 0
    for k in sorted(base):
        if k not in new:
            print("MISSING", label(k))
        elif base[k] != new[k]:
            print("DIFFERS", label(k))
        else:
            same += 1
    added = sorted(k for k in new if k not in base)
    for k in added:
        print("NEW", label(k))
    return same, len(base), len(added)

def summary(name, same, n, added):
    return f"{name}: {same} of {n} identical" + (f" ({added} new)" if added else "")

args = sys.argv[1:]
everything = "--all" in args
old_lib, new_lib = [a for a in args if a != "--all"]
old_code, new_code = funcs(old_lib), funcs(new_lib)
failed = False
lines = []
if everything:
    # solve kernels under their (kernel, flags) key, so that a build with a new trailing flag still matches
    def by_key(code):
        dm = demangle(list(code))
        return {(lambda k: f"{k[0]} {k[1]}" if k else n)(key(dm[n])): v for n, v in code.items()}
    same, n, added = compare(by_key(old_code), by_key(new_code), lambda k: k)
    failed = same != n
    lines.append(summary("all functions", same, n, added))
else:
    old, new = solve_kernels(old_code), solve_kernels(new_code)
    for flags, name in SETS:
        same, n, added = compare({k: v for k, v in old.items() if k[1] == flags},
                                 {k: v for k, v in new.items() if k[1] == flags}, lambda k: f"{name} {k[0]}")
        failed |= same != n
        lines.append(summary(name, same, n, added))
print("; ".join(lines))
sys.exit(1 if failed else 0)
