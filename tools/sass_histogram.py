"""Opcode histogram of the step kernels' SASS (cuobjdump -sass of the in-tree library): how many global loads /
stores, shuffles, integer and floating-point instructions a thread executes on the straight path, and proof
that the hot kernels carry no local-memory traffic outside their boundary slow path.

  python tools/sass_histogram.py > profiles/rNN_sass_histogram.txt
MEASUREMENT INFRASTRUCTURE (runs here: no GPU needed)."""
import collections
import re
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
LIB = ROOT / "lattice_boltzmann_method_gpu_b200" / "liblbm_b200.so"
# FAST arithmetic, BGK collision (COLL 0), no moments, no sum |u|; dense: speculative pull, in-place even / odd step
WANT = ["k_step_dense<double, false, 0, false, false, true, 1>", "k_step_dense<double, false, 0, false, false, true, 2>",
        "k_step_dense<float, false, 0, false, false, true, 1>", "k_step_dense<float, false, 0, false, false, true, 2>",
        "k_sparse_aa_even<double, false, 0, false, false, false>", "k_sparse_aa_odd<double, false, 0, false, false, false>",
        "k_sparse_aa_even<float, false, 0, false, false, false>", "k_sparse_aa_odd<float, false, 0, false, false, false>",
        "k_step_sparse<double, false, 0, false, false>", "k_sparse_aa_persist<float, false, 0>"]
GROUPS = [("LDG", r"^LDG"), ("STG", r"^STG"), ("LDL/STL (local)", r"^(LDL|STL)"), ("SHFL", r"^SHFL"), ("LDC/ULDC (constant bank)", r"^(LDC|ULDC|LDCU)"),
          ("integer (IADD3 IMAD LOP3 SHF LEA ISETP SEL VIADD ...)", r"^(IADD|IMAD|LOP3|SHF|LEA|ISETP|SEL|VIADD|IABS|MOV|PRMT|UIADD|UMOV|ULOP|USHF|UIMAD|R2P|P2R|PLOP|UISETP|ULEA|USEL)"),
          ("fp32 (FFMA FADD FMUL MUFU)", r"^(FFMA|FADD|FMUL|MUFU|FSETP|FSEL)"), ("fp64 (DFMA DADD DMUL)", r"^(DFMA|DADD|DMUL|DSETP)"),
          ("branches / barriers", r"^(BRA|BSSY|BSYNC|EXIT|CALL|RET|BAR|WARPSYNC|NANOSLEEP|YIELD)")]


def main():
    raw = subprocess.run(["cuobjdump", "-sass", str(LIB)], capture_output=True, text=True).stdout
    names = subprocess.run(["c++filt"], input="\n".join(re.findall(r"Function : (\S+)", raw)), capture_output=True, text=True).stdout.split("\n")
    chunks = raw.split("Function : ")[1:]
    print("static SASS instruction counts per kernel (whole function, slow paths included); sm_100a, nvcc 12.9 -O3")
    print()
    for want in WANT:
        for nm, body in zip(names, chunks):
            if want in nm:
                ops = re.findall(r"^\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", body, re.M)
                hist = collections.Counter()
                for op in ops:
                    base = op.split(".")[0]
                    for g, pat in GROUPS:
                        if re.match(pat, base):
                            hist[g] += 1
                            break
                    else:
                        hist["other"] += 1
                print(f"{want}: {len(ops)} instructions")
                for g, _ in GROUPS + [("other", "")]:
                    if hist[g]:
                        print(f"    {g:58s} {hist[g]:5d}")
                break
    return 0


if __name__ == "__main__":
    sys.exit(main())
