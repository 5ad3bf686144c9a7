"""Resource usage (cuobjdump -res-usage) of every solve kernel of libcmpc.so next to its BODY twin."""
import re, subprocess, sys
CUDA = "/usr/local/cuda/bin/"
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
    tab.setdefault(m.group(1) + "<" + ",".join(args[:-1]) + ">", {})[args[-1]] = res
for k in sorted(tab):
    print(f"{k:42s} plain: {tab[k].get('0', '-'):40s} BODY: {tab[k].get('1', '-')}")
