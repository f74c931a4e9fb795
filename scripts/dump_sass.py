"""SASS evidence: one instruction-text listing per kernel (gzip) + a mnemonic histogram for every kernel of the built extension.

    python scripts/dump_sass.py            # writes profiles/sass/*.sass.gz and profiles/sass_mnemonics.json

The listings are ``cuobjdump -sass`` with the hex encodings stripped (address + instruction text kept).  What to look for
(B200_PROFILING.md): UTCHMMA (tcgen05.mma, bf16 and tf32 kinds alike), UTMALDG[.IM2COL] (TMA loads), UBLKCP / UBLKRED (bulk copy
engine stores / reductions), LDTM (tcgen05.ld), UTCBAR (tcgen05.commit), LDGMC / multimem (NVLS), ATOM / RED .SYS on peer
pointers (NVLink atomics), LD/ST .SYS (peer loads / stores).
"""
import collections
import gzip
import json
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SO = os.path.join(ROOT, "theanompi_b200", "_tmpi_native.so")
OUT = os.path.join(ROOT, "profiles", "sass")
FULL = ["gemm_tcgen05I13__nv_bfloat16Li128ELi2", "gemm_tcgen05IfLi128ELi1", "fused_twoshot_kernelINS_7SgdRuleELi8", "fused_oneshot_kernelINS_7SgdRuleELi4",
        "fused_twoshot_kernelINS_8AdamRuleELi8", "fused_oneshot_kernelINS_8AdamRuleELi4",
        "easgd_elastic_kernelILi4", "gosgd_pull_merge_kernelILi4", "ticket_acquire_kernel", "ticket_release_kernel", "gosgd_poll_kernel",
        "gosgd_push_end_kernel", "push_region_kernel", "sgd_flat_kernel", "adam_flat_kernel", "bn_colreduce_kernelI13__nv_bfloat16Li1",
        "bn_apply_kernelI13__nv_bfloat16", "lstm_cell_fwd_kernelI13__nv_bfloat16"]


def main():
    txt = subprocess.run(["cuobjdump", "-sass", SO], stdout=subprocess.PIPE, text=True).stdout
    parts = re.split(r"(?=\t\tFunction : )", txt)
    os.makedirs(OUT, exist_ok=True)
    hist = {}
    ins = re.compile(r"/\*([0-9a-f]{4,})\*/\s+(.*?);")
    for p in parts[1:]:
        name = re.match(r"\t\tFunction : (\S+)", p).group(1)
        lines = ["%s  %s" % (m.group(1), m.group(2).strip()) for m in ins.finditer(p)]
        cnt = collections.Counter()
        for l in lines:
            op = l.split(None, 1)[1]
            op = re.sub(r"^@!?U?P\d+\s+", "", op)
            cnt[op.split()[0].split(".")[0] + ("." + ".".join(op.split()[0].split(".")[1:3]) if op.split()[0].startswith(("UTMA", "UBLK", "RED", "ATOM", "LDG", "STG", "UTC")) else "")] += 1
        hist[name] = {"instructions": len(lines), "mnemonics": dict(cnt.most_common(40))}
        if any(k in name for k in FULL):
            short = re.sub(r"[^A-Za-z0-9_]", "_", name)[:120]
            with gzip.open(os.path.join(OUT, short + ".sass.gz"), "wt") as f:
                f.write("// cuobjdump -sass %s  (encodings stripped)\n// Function : %s\n" % (os.path.basename(SO), name))
                f.write("\n".join(lines) + "\n")
    with open(os.path.join(ROOT, "profiles", "sass_mnemonics.json"), "w") as f:
        json.dump(hist, f, indent=1, sort_keys=True)
    key = ("UTCHMMA", "UTMALDG", "UBLKCP", "UBLKRED", "LDTM", "UTCBAR", "LDGMC", "MULTIMEM")
    for name, h in sorted(hist.items()):
        got = {k: v for k, v in h["mnemonics"].items() if k.startswith(key)}
        if got:
            print(name[:90], got)


if __name__ == "__main__":
    main()
