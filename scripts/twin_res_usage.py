"""Resource usage (cuobjdump -res-usage) of every solve kernel of libcmpc.so next to its BODY twin, its BODY+CONTACT
twin, its two WEIGHTS twins, its two FORCE twins and its two STAGE twins, matched by the template arguments without the trailing feature
flags (a build that predates a flag has it false)."""
import re, subprocess, sys
CUDA = "/usr/local/cuda/bin/"
CORE_ARGS = {"solve_kernel": 7, "solve_riccati_kernel": 2}
out = subprocess.run([CUDA + "cuobjdump", "-res-usage", sys.argv[1]], capture_output=True, text=True, check=True).stdout
rows = re.findall(r"Function (\S+):\n\s*(REG:\d+ STACK:\d+ SHARED:\d+ LOCAL:\d+)", out)
names = [r[0] for r in rows]
dm = subprocess.run([CUDA + "cu++filt"], input="\n".join(names), capture_output=True, text=True).stdout.splitlines()
tab = {}
for (n, res), d in zip(rows, dm):
    m = re.match(r"void cmpc::(solve_kernel|solve_riccati_kernel)<(.*)>\(cmpc::SolveParams\)", d)
    if not m:
        continue
    args = [a.strip().replace("(int)", "").replace("(bool)", "") for a in m.group(2).split(",")]
    core = CORE_ARGS[m.group(1)]
    flags = ",".join((args[core:] + ["0"] * 5)[:5])
    tab.setdefault(m.group(1) + "<" + ",".join(args[:core]) + ">", {})[flags] = res
for k in sorted(tab):
    print(k)
    for f, name in (("0,0,0,0,0", "plain"), ("1,0,0,0,0", "BODY"), ("1,1,0,0,0", "BODY+CONTACT"),
                    ("1,0,1,0,0", "BODY+WEIGHTS"), ("1,1,1,0,0", "BODY+CONTACT+WEIGHTS"),
                    ("1,0,1,1,0", "BODY+WEIGHTS+FORCE"), ("1,1,1,1,0", "BODY+CONTACT+WEIGHTS+FORCE"),
                    ("1,0,1,1,1", "BODY+WEIGHTS+FORCE+STAGE"), ("1,1,1,1,1", "BODY+CONTACT+WEIGHTS+FORCE+STAGE")):
        print(f"  {name:34s} {tab[k].get(f, '-')}")
