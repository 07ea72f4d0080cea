"""Instruction histogram of the tcgen05 / TMA / TMEM opcodes per kernel in libsow_b200.so (cuobjdump -sass; no GPU needed).

    python tools/sass_histogram.py > profiles/r02_sass_histogram.txt
UTCHMMA = tcgen05.mma (kind::f16), UTMALDG / UTMASTG = TMA tensor load / store, UTMAPF = TMA L2 prefetch, UBLKCP / UBLKPF = bulk
copy / prefetch, LDTM / STTM = tcgen05.ld / st (TMEM), UTCBAR = tcgen05.commit, UTCATOMSWS = TMEM alloc, SYNCS = mbarrier,
UCGABAR = cluster barrier, MAPA / ST.E...CLUSTER via 'MAPA', DMMA = fp64 mma.sync (Cholesky-QR above rank 16), LDGSTS = cp.async,
ACQBULK / PREEXIT = griddepcontrol.wait / launch_dependents (programmatic dependent launch).  2CTA = instructions of the CTA-pair
(cta_group::2) forms: UTCHMMA.2CTA, UTMALDG.2D.2CTA, UTCBAR.2CTA.MULTICAST, UTCATOMSWS.2CTA (also counted under their opcode).
"""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "sow_b200", "csrc", "libsow_b200.so")
OPS = ["UTCHMMA", "UTCQMMA", "UTCIMMA", "UTMALDG", "UTMASTG", "UTMAPF", "UBLKCP", "UBLKPF", "LDTM", "STTM", "UTCBAR", "UTCATOMSWS",
       "SYNCS", "UCGABAR", "MAPA", "UMAPA", "HMMA", "DMMA", "FFMA", "DFMA", "LDGSTS", "ACQBULK", "PREEXIT"]


def main():
    out = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True, check=True).stdout
    kernels = collections.OrderedDict()
    cur = None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
            kernels[cur] = collections.Counter()
            continue
        if cur is None:
            continue
        m = re.search(r"^\s*/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", line)
        if m:
            op = m.group(1).split(".")[0]
            kernels[cur]["_total"] += 1
            if ".2CTA" in m.group(1):
                kernels[cur]["2CTA"] += 1
            for known in OPS:
                if op == known or (known in ("UCGABAR", "MAPA", "UMAPA") and op.startswith(known)):
                    kernels[cur][known] += 1
                    break
    dem = subprocess.run(["c++filt"] + list(kernels), capture_output=True, text=True).stdout.splitlines()
    print("# cuobjdump -sass sow_b200/csrc/libsow_b200.so: per-kernel counts of tensor-core / TMA / TMEM / barrier opcodes")
    print("# (" + ", ".join(OPS) + ", 2CTA; 'instr' = all SASS instructions of the kernel)")
    tot = collections.Counter()
    for (name, c), d in zip(kernels.items(), dem):
        short = re.sub(r"\(.*", "", d).replace("void ", "")
        cells = " ".join(f"{op}={c[op]}" for op in OPS + ["2CTA"] if c[op])
        print(f"{short:<70s} instr={c['_total']:<6d} {cells}")
        tot.update(c)
    print("# TOTAL " + " ".join(f"{op}={tot[op]}" for op in OPS + ["2CTA"] if tot[op]))


if __name__ == "__main__":
    main()
