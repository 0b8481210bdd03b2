"""SASS evidence for profiles/: per-kernel instruction mix of libtgpu.so (cuobjdump -sass) and the lines around the
TMA bulk copies (UBLKCP) / mbarrier waits.  usage: python tools/sass_summary.py [libtgpu.so] > profiles/rNN_sass_summary.txt"""
import collections
import re
import subprocess
import sys

lib = sys.argv[1] if len(sys.argv) > 1 else "pressurepoissonsolver_b200/libtgpu.so"
out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True).stdout
kern, kernels = None, collections.OrderedDict()
for line in out.splitlines():
    m = re.match(r"\s*Function : (\S+)", line)
    if m:
        kern = m.group(1)
        kernels[kern] = []
        continue
    m = re.match(r"\s*/\*([0-9a-f]{4,})\*/\s+(.*?);", line)
    if m and kern:
        kernels[kern].append(m.group(2).strip())
demangle = subprocess.run(["c++filt"] + list(kernels), capture_output=True, text=True).stdout.splitlines()
names = dict(zip(kernels, demangle))
WANT = ("smooth3d16_kernel", "smooth3d32c_kernel", "iface_rhs32_kernel", "smooth2d32_kernel", "apply_tma_kernel", "apply3d32_tma_kernel",
        "face_residual_restrict", "push_faces_kernel")
KEYS = ("DFMA", "DADD", "DMUL", "LDS", "STS", "LDG", "STG", "LDGSTS", "UBLKCP", "SYNCS", "BAR", "SHFL", "MUFU", "LDL", "STL", "LDC", "CCTL", "MEMBAR", "ERRBAR", "ATOM", "RED")
print("# SASS instruction mix per kernel (cuobjdump -sass %s); columns: total instructions, then the count of each opcode family" % lib)
print("# UBLKCP = cp.async.bulk (TMA 1-D bulk copy), SYNCS = mbarrier operations, LDGSTS = cp.async, LDL/STL = local-memory (spill) traffic")
for k, ins in kernels.items():
    n = names.get(k, k)
    if not any(w in n for w in WANT):
        continue
    short = re.sub(r"\(.*", "", n).replace("void tgpu::", "")
    c = collections.Counter()
    for i in ins:
        op = re.sub(r"^@!?U?P\d+\s+", "", i).split()[0].split(".")[0]
        for key in KEYS:
            if op == key or (key == "LDG" and op in ("LDG", "LD")) or (key == "STG" and op in ("STG", "ST")):
                c[key] += 1
    print("%-62s %6d  %s" % (short[:62], len(ins), " ".join("%s=%d" % (key, c[key]) for key in KEYS if c[key])))
print()
print("# excerpt: the TMA bulk copy and its mbarrier in apply_tma_kernel<3, 16, 0>")
for k, ins in kernels.items():
    if "apply_tma_kernel<3, 16, 0>" in names.get(k, ""):
        for idx, i in enumerate(ins):
            if "UBLKCP" in i or "SYNCS" in i:
                print("  %5d  %s" % (idx, i))
        break
