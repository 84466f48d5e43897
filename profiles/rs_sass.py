"""Instruction count of k_rs_score's scoring loop and the kernel's registers, from the compiler alone
(no GPU): compiles csrc/ransac.cu with the library's flags plus -Xptxas -v into a temporary directory,
then reads the SASS of each k_rs_score<CH> with cuobjdump.

The scoring body is the straight-line block of the tile loop that holds every FFMA2: from the loop head
to the first branch after the last FFMA2 (the branch to the in-band queue).  It evaluates CH / 2
hypothesis pairs for APC_TILE_ITEMS = 4 points, so "per pair-point" divides its length by 2 * CH.
The block also holds the per-tile work (next tile's loads, the band limits lo / hi of the 4 points,
the shared-memory loads of the packed planes); "pair-point core" leaves those out and counts only the
instruction classes the evaluation of a pair repeats.

    python profiles/rs_sass.py [--json OUT]
"""
from __future__ import annotations

import collections
import json
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from autodriver_pointcloud_preprocessor_b200 import _build  # noqa: E402

ITEMS = 4
# what the evaluation of a pair repeats: distances and error terms, compares, the band's predicate
# merge, and the accumulation (SEL + IADD3, or a predicated IADD3 / IMAD.IADD)
CORE = ("FFMA2", "FMUL2", "FSETP", "PLOP3", "SEL", "IADD3", "IMAD.IADD")
INS = re.compile(r"\s+/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;")


def opcode(text: str) -> str:
    t = text.split()
    op = t[1] if t[0].startswith("@") else t[0]
    parts = op.split(".")
    return ".".join(parts[:2]) if parts[0] == "IMAD" and len(parts) > 1 else parts[0]


def scoring_body(sass: str) -> list[tuple[int, str]]:
    ins = [(int(m.group(1), 16), m.group(2)) for m in map(INS.match, sass.splitlines()) if m]
    ffma2 = [a for a, t in ins if opcode(t) == "FFMA2"]
    head = None                  # target of the backward branch that closes the tile loop
    for a, t in ins:
        m = re.search(r"BRA\s+(?:`?\(?)0x([0-9a-f]+)", t)
        if m and int(m.group(1), 16) < ffma2[0] and a > ffma2[-1]:
            tgt = int(m.group(1), 16)
            head = tgt if head is None else max(head, tgt)   # other backward branches go to code before the loop
    body = []
    for a, t in ins:
        if a < head:
            continue
        body.append((a, t))
        if a > ffma2[-1] and opcode(t) == "BRA":
            break
    return body


def main() -> None:
    out_json = sys.argv[sys.argv.index("--json") + 1] if "--json" in sys.argv else None
    nvcc = _build._nvcc()
    cuobjdump = os.path.join(os.path.dirname(nvcc), "cuobjdump")
    src = os.path.join(_build.CSRC, "ransac.cu")
    res = {}
    with tempfile.TemporaryDirectory() as tmp:
        obj = os.path.join(tmp, "ransac.o")
        r = subprocess.run([nvcc, *_build.NVCC_FLAGS, "-Xptxas", "-v", "-c", src, "-o", obj],
                           capture_output=True, text=True, check=True)
        ptxas = r.stderr.splitlines()
        syms = subprocess.run([cuobjdump, "-symbols", obj], capture_output=True, text=True, check=True).stdout
        for ch in (20, 16, 10, 8):
            name = next(s for s in re.findall(r"\b(_Z10k_rs_scoreILi\d+EE[^$\s]+)", syms) if f"ILi{ch}EE" in s)
            i = next(k for k, l in enumerate(ptxas) if "Compiling entry" in l and name in l)
            info = "\n".join(ptxas[i + 1:i + 4])
            spill = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", info)
            regs = int(re.search(r"Used (\d+) registers", info).group(1))
            sass = subprocess.run([cuobjdump, "-sass", "-fun", name, obj], capture_output=True, text=True,
                                  check=True).stdout
            body = scoring_body(sass)
            hist = collections.Counter(opcode(t) for _, t in body)
            pp = ch // 2 * ITEMS
            res[f"CH{ch}"] = dict(registers=regs, spill_store_bytes=int(spill.group(1)),
                                  spill_load_bytes=int(spill.group(2)), body_instructions=len(body),
                                  pair_points=pp, per_pair_point=round(len(body) / pp, 2),
                                  core_per_pair_point=round(sum(hist[o] for o in CORE) / pp, 2), opcodes=dict(hist.most_common()))
            c = res[f"CH{ch}"]
            print(f"k_rs_score<{ch}>: {regs} registers, spills {c['spill_store_bytes']}/{c['spill_load_bytes']} B; "
                  f"scoring body {len(body)} instructions / {pp} pair-points = {c['per_pair_point']} "
                  f"(pair-point core {c['core_per_pair_point']})")
            print("   ", ", ".join(f"{k} {v}" for k, v in hist.most_common(14)))
    if out_json:
        with open(out_json, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
