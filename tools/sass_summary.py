"""Regenerates profiles/sass/: a per-kernel mnemonic table of libb200fusion.so, full listings of a few
representative kernels, and the complete listing of every kernel (gzip).

    python tools/sass_summary.py r1
"""
import collections
import gzip
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import b200path  # noqa: F401,E402

tag = sys.argv[1] if len(sys.argv) > 1 else "r1"
so = os.path.join(ROOT, "lib", "libb200fusion.so")
out_dir = os.path.join(ROOT, "profiles", "sass")
os.makedirs(out_dir, exist_ok=True)
sass = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True, check=True).stdout
with gzip.open(os.path.join(out_dir, f"{tag}_all_kernels.sass.gz"), "wt", compresslevel=9) as f:
    f.write(sass)
demangle = lambda n: subprocess.run(["c++filt", n], capture_output=True, text=True).stdout.strip()
COLS = ["UTCHMMA", "UTMALDG", "UTMASTG", "UTMAPF", "LDTM", "UTCBAR", "SYNCS", "FFMA2", "FMUL2", "FADD2", "FFMA", "MUFU",
        "HMMA", "LDG", "STG", "LDS", "STS", "LD", "ST", "SHFL", "MATCH", "ATOMS", "ATOMG", "RED", "BAR", "DFMA", "DADD",
        "DMUL"]
kernels = {}
cur = None
for line in sass.splitlines():
    m = re.match(r"\s+Function : (\S+)", line)
    if m:
        cur = m.group(1)
        kernels[cur] = {"ops": collections.Counter(), "lines": []}
        continue
    if cur is None:
        continue
    kernels[cur]["lines"].append(line)
    m = re.match(r"\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z][A-Z0-9_]*)", line)
    if m:
        kernels[cur]["ops"][m.group(1)] += 1
rows = []
for name, k in kernels.items():
    d = demangle(name)
    d = re.sub(r"\(.*$", "", d).replace("b200::", "").replace("(anonymous namespace)::", "")
    rows.append((d, sum(k["ops"].values()), k["ops"], name))
rows.sort()
with open(os.path.join(out_dir, f"{tag}_sass_summary.md"), "w") as f:
    f.write(f"# SASS summary of libb200fusion.so (sm_100a), {tag}\n\n")
    f.write("`cuobjdump -sass <pkg>/libb200fusion.so` (`python tools/sass_summary.py`), one row per kernel: instruction "
            "count and the count of the mnemonics that identify the Blackwell-native paths (UTCHMMA = tcgen05.mma, "
            "LDTM = tcgen05.ld, UTMALDG/UTMASTG = TMA load/store, SYNCS = mbarrier, FFMA2/FMUL2/FADD2 = packed fp32x2; "
            "LD/ST = generic-space accesses, which the hot kernels should not have).  No HMMA (legacy mma.sync) anywhere.  "
            f"The tool writes the complete listing of every kernel to `{tag}_all_kernels.sass.gz` (a build product, not "
            "kept in git); six representative kernels are "
            "stored uncompressed next to this file.\n\n")
    f.write("| kernel | instr | " + " | ".join(COLS) + " |\n|---|---|" + "---|" * len(COLS) + "\n")
    for d, n, ops, _ in rows:
        f.write(f"| `{d}` | {n} | " + " | ".join(str(ops[c]) if ops[c] else "" for c in COLS) + " |\n")
wanted = ("conv_gemm_kernel<256, false, 0, false, 0, 0, false>", "conv_gemm_kernel<128, false, 0, false, 0, 0, true>",
          "conv_wgrad_kernel<256>", "attn_fused_kernel<64>", "dwi_normalize_reg_kernel<4>", "nyul_transform_kernel<false>")
for old in os.listdir(out_dir):
    if old.endswith(".sass"):
        os.remove(os.path.join(out_dir, old))
for d, n, ops, name in rows:
    if any(d.endswith(w) or d == w or d.endswith("void " + w) for w in wanted):
        fn = re.sub(r"[^A-Za-z0-9]+", "_", d).strip("_") + ".sass"
        with open(os.path.join(out_dir, fn), "w") as f:
            f.write("\n".join(kernels[name]["lines"]) + "\n")
print(f"{len(rows)} kernels -> {out_dir}")
