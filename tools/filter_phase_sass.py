"""Static SASS instructions between the clock64 stamps of the production Wiener kernel (k_filter<true, false, 32>)
of a -DB4D_PROFILE_STEP build: the counts that go next to the per-phase cycles the launcher prints ("P" / "PMEAN").
    python tools/filter_phase_sass.py b4d_filter.o   (an object or a library built with make EXTRA=-DB4D_PROFILE_STEP)
Static counts: a phase with a full-group fast path and a batched path for partial groups lists both."""
import os
import re
import subprocess
import sys

CUOBJDUMP = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")
sass = subprocess.run([CUOBJDUMP, "-sass", sys.argv[1]], capture_output=True, text=True, check=True).stdout
body = [f for f in sass.split("Function : ") if "k_filterILb1ELb0ELi32ELb0E" in f.split("\n")[0]][0]
ins = re.findall(r"/\*([0-9a-f]{4,})\*/\s+([^;]*);", body)
clk = [i for i, (_, t) in enumerate(ins) if "SR_CLOCKLO" in t]
print(sys.argv[1], "instructions", len(ins), "clock reads at", clk)
for a, b in zip(clk, clk[1:]):
    ops = {}
    for _, t in ins[a + 1:b]:
        op = re.sub(r"^@!?U?P\w+\s+", "", t).split()[0].split(".")[0]
        ops[op] = ops.get(op, 0) + 1
    top = sorted(ops.items(), key=lambda x: -x[1])[:7]
    print("%5d..%5d %5d  %s" % (a, b, b - a - 1, " ".join("%s:%d" % kv for kv in top)))
