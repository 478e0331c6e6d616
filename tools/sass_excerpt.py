"""Instruction census of the shipped kernels (cuobjdump -sass of the built library) -> profiles/r03_sass_excerpt.txt."""
import collections
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SO = os.path.join(ROOT, "mav_trajectory_generation_b200", "libmtg_b200.so")
WANT = collections.OrderedDict([
    ("twisted_tmem_v5_kernelILi10ELi4ELi3ELi2ELb0ELi2ELi16EE", "K1v5 compiled for K = 16 (C5, C3: one tile buffer, early refill, unrolled sweeps) <N=10,r=4,D=3>"),
    ("twisted_tmem_v5_kernelILi10ELi4ELi3ELi2ELb0ELi0ELi8EE", "K1v5 compiled for K = 8 (C2: double buffered, unrolled sweeps) <10,4,3>"),
    ("twisted_tmem_v5_kernelILi8ELi3ELi3ELi3ELb0ELi0ELi4EE", "K1v5 compiled for K = 4 (C4) <N=8,r=3,D=3>"),
    ("twisted_tmem_v5_kernelILi10ELi4ELi3ELi2ELb0ELi2ELi0EE", "K1v5 run-time shape at K = 14, 16 (TMA inputs, one tile buffer, early refill) <N=10,r=4,D=3>"),
    ("twisted_tmem_v5_kernelILi10ELi4ELi3ELi2ELb0ELi0ELi0EE", "K1v5 run-time shape at K <= 12 (TMA inputs, double buffered) <10,4,3>"),
    ("twisted_tmem_v5_kernelILi8ELi3ELi3ELi3ELb0ELi0ELi0EE", "K1v5 run-time shape <N=8,r=3,D=3>"),
    ("twisted_tmem_kernelILi10ELi4ELi3ELb0ELb0E", "K1v3 per-tile <10,4,3>"),
    ("twisted_tmem_kernelILi10ELi4ELi3ELb0ELb1E", "K1v3 cost-only (fused Mellinger) <10,4,3>"),
    ("twisted_tmem_v4_kernelILi10ELi4ELi3ELb0E", "K1v4 persistent <10,4,3>"),
    ("twisted_chunked_kernelILi10ELi4ELi3E", "K3 chunked large-K <10,4,3>"),
    ("masked_block_kernelILi10ELi3E", "K4 masked block <N=10,DG=3>"),
    ("range_eval_kernelILi10E", "evaluateRange evaluation <N=10>"),
    ("cost_kernelILi10ELi4E", "computeCost <N=10,r=4>")])
KEYS = ["IMAD", "WARPSYNC", "ENDCOLLECTIVE", "BRA", "R2UR", "FSEL", "STTM", "LDTM", "UTCATOMSWS", "UTMASTG", "UBLKCP", "SYNCS", "UTMACMDFLUSH", "LDGSTS", "LDGDEPBAR", "DEPBAR", "DFMA", "DMUL",
        "DADD", "MUFU.RCP64H", "MUFU.RSQ64H", "STL", "LDL", "UTCHMMA", "UTCQMMA", "ATOMG", "SHFL", "FENCE.VIEW.ASYNC", "STS", "LDS",
        "LDG", "STG"]


def main():
    sass = subprocess.run(["cuobjdump", "-sass", SO], capture_output=True, text=True).stdout
    funcs = re.split(r"\n\s*Function : ", sass)
    out = ["# SASS evidence of the shipped library (cuobjdump -sass libmtg_b200.so, sm_100a, CUDA 12.9), round 3; tools/sass_excerpt.py\n",
           "# tcgen05.st/ld -> STTM/LDTM, tcgen05.alloc -> UTCATOMSWS, TMA tensor store -> UTMASTG, cp.async.bulk (TMA bulk load) -> UBLKCP,\n"
           "# mbarrier -> SYNCS, cp.async -> LDGSTS; no UTC*MMA (tensor cores are off on this path by design); STL/LDL = local-memory spills.\n\n"]
    found = set()
    for f in funcs[1:]:
        name = f.split("\n", 1)[0]
        for k, label in WANT.items():
            if k in name and k not in found:
                found.add(k)
                lines = [l for l in f.split("\n") if "/*" in l and ";" in l]
                ops = collections.Counter()
                for l in lines:
                    mo = re.search(r"\*/\s+(@!?U?P\d+\s+)?([A-Z0-9_.]+)", l)
                    if mo:
                        op = mo.group(2)
                        for key in KEYS:
                            if op == key or op.startswith(key + ".") or op.startswith(key):
                                if key in ("LDG", "STG", "STS", "LDS") and not (op == key or op.startswith(key + ".")):
                                    continue
                                ops[key] += 1
                                break
                out.append(f"== {label}\n   {name[:130]}\n   instructions: {len(lines)}\n   " +
                           "  ".join(f"{k}={ops[k]}" for k in KEYS if ops[k] or k in ("STL", "LDL", "UTCHMMA")) + "\n")
                for l in [l.strip() for l in lines if any(x in l for x in ("STTM", "LDTM", "UTMASTG", "UTCATOMSWS", "UBLKCP", "SYNCS"))][:6]:
                    out.append("     " + re.sub(r"\s+", " ", l)[:120] + "\n")
                out.append("\n")
    open(os.path.join(ROOT, "profiles", "r03_sass_excerpt.txt"), "w").write("".join(out))
    print("".join(out)[:1500])


if __name__ == "__main__":
    main()
