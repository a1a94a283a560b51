"""Dump the SASS of the hot kernels of libemagls_cuda.so, one gzip file per kernel, under profiles/<tag>_sass/
(north_star: SASS committed next to the ncu summaries).  usage: python tools/sass_dump.py r02"""
import gzip
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "emagls_b200", "lib", "libemagls_cuda.so")
tag = sys.argv[1] if len(sys.argv) > 1 else "r02"
out = os.path.join(ROOT, "profiles", f"{tag}_sass")
os.makedirs(out, exist_ok=True)
# (file name, substring of the demangled name) of the instances that run in the default em32 configuration
WANT = [("ozaki_gemm_fwd_EpiPhaseSliceFix6_words_nt80_ew20", ["ozaki_gemm_kernel<6", "EpiPhaseSliceFix<6>", "TileCfg<80, 2, 20>"]),
        ("ozaki_gemm_fwd_EpiPhaseSliceRaw6_nt64", ["ozaki_gemm_kernel<6", "EpiPhaseSliceRaw<6>", "TileCfg<64, 3, 16>"]),
        ("ozaki_gemm_bwd_EpiStoreF64_6_nt80", ["ozaki_gemm_kernel<6", "EpiStoreF64", "TileCfg<80, 2, 16>"]),
        ("tsqr_sep_kernel", ["tsqr_sep_kernel"]), ("svdclip_kernel_occ4", ["svdclip_kernel<4>"]),
        ("chain_bwd_sep_kernel", ["chain_bwd_sep_kernel"]), ("bwd_fused_kernel_T6", ["bwd_fused_kernel<6>"]),
        ("gram_sweep_kernel", ["gram_sweep_kernel"]), ("fused_render16_kernel_pre1", ["fused_render16_kernel<1>"])]
sass = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True).stdout
blocks, cur, name = {}, None, None
for line in sass.splitlines():
    m = re.search(r"Function : (\S+)", line)
    if m:
        name = subprocess.run(["c++filt", m.group(1)], capture_output=True, text=True).stdout.strip()
        cur = blocks.setdefault(name, [])
    if cur is not None:
        cur.append(line)
index = []
for fname, keys in WANT:
    hits = [n for n in blocks if all(k in n for k in keys)]
    if not hits:
        index.append(f"{fname}: NOT FOUND")
        continue
    n = hits[0]
    body = "\n".join(blocks[n]) + "\n"
    with gzip.open(os.path.join(out, fname + ".sass.gz"), "wt") as f:
        f.write("// " + n + "\n" + body)
    ninstr = sum(1 for l in blocks[n] if re.match(r"\s+/\*[0-9a-f]{4,}\*/", l))
    ops = {}
    for l in blocks[n]:
        mm = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_]+)", l)
        if mm:
            ops[mm.group(1)] = ops.get(mm.group(1), 0) + 1
    top = " ".join(f"{k}={v}" for k, v in sorted(ops.items(), key=lambda kv: -kv[1])[:10])
    ev = " ".join(f"{k}={ops[k]}" for k in ("UTCIMMA", "UTCBAR", "LDTM", "UTMALDG", "UTMASTG", "UBLKCP", "SYNCS", "DMMA", "LDGSTS") if k in ops)
    index.append(f"{fname}.sass.gz: {ninstr} instructions | {ev} | {top}\n    {n[:200]}")
open(os.path.join(out, "INDEX.txt"), "w").write(
    "# cuobjdump -sass emagls_b200/lib/libemagls_cuda.so (sm_100a), one file per hot kernel (tools/sass_dump.py)\n" + "\n".join(index) + "\n")
print("\n".join(index))
