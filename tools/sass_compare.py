"""Compares the SASS of kernels between two builds of liboz_b200.so, instruction by instruction.

Kernels are matched by demangled name with the return type removed, a trailing template argument `, 0` dropped and
then the template arguments `<0>` removed.  A trailing 0 is the reference-scoring instantiation (SCORING_REFERENCE) or the
bf16 one (OUT_BF16 of conv2_table_gather_kernel); a lone `<0>` is the reference-rule instantiation (ozbb::RULES_REFERENCE)
or the bf16 SM-pair GEMM (OP_BF16).  So a kernel that became `template <int RULES>` or `template <int OP>` is compared with
its pre-template self, `tree_step_kernel<R, 0>` with `tree_step_kernel<R>` and `conv2_table_gather_kernel<NJ, W, X, 0>`
with `conv2_table_gather_kernel<NJ, W, X>`.  Before that, the reference-values tree kernel `tree_step_kernel<R, S, 0>`
(VALUES_REFERENCE) becomes `tree_step_kernel<R, S>`, its name before the value convention was a template argument, and
before that the non-exploring tree kernel `tree_step_kernel<R, S, V, 0>` becomes `tree_step_kernel<R, S, V>`, its name
before root exploration was a template argument.
Every instantiation of a listed kernel that
the OLD build has is compared.  Instruction addresses and encodings are ignored; branch and call targets are offsets
inside the kernel's own section, so identical code gives identical text.  Needs cuobjdump and c++filt, no GPU.

usage: python tools/sass_compare.py OLD.so NEW.so [kernel ...]
       (default kernels: tree_step_kernel rules_apply_kernel perft_playout_kernel; the network's kernels, e.g.
        oz_gemm2_kernel oz_gemm_kernel conv2_table_gather_kernel, are matched without their anonymous namespace)
exit status 0 iff every listed kernel is identical.
"""
from __future__ import annotations

import re
import subprocess
import sys

DEFAULT = ["tree_step_kernel", "rules_apply_kernel", "perft_playout_kernel"]


def functions(so: str) -> dict[str, list[str]]:
    txt = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True, check=True).stdout
    out: dict[str, list[str]] = {}
    cur = None
    for line in txt.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = out.setdefault(m.group(1), [])
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(.*?)\s*;", line)
        if m and cur is not None:
            cur.append(re.sub(r"\s+", " ", m.group(1)))
    names = list(out)
    dem = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True, check=True).stdout
    return {normalize(d): out[n] for n, d in zip(names, dem.splitlines())}


def normalize(demangled: str) -> str:
    s = re.sub(r"^void ", "", demangled).replace("(anonymous namespace)::", "")  # oz_net.cu's kernels
    s = re.sub(r"^(tree_step_kernel<\d+, \d+, \d+), 0>\(", r"\1>(", s)  # the non-exploring tree kernel
    s = re.sub(r"^(tree_step_kernel<\d+, \d+), 0>\(", r"\1>(", s)  # the reference-values tree kernel
    s = re.sub(r", 0>\(", ">(", s)
    return s.replace("<0>(", "(")


def main(argv: list[str]) -> int:
    old, new = functions(argv[1]), functions(argv[2])
    kernels = argv[3:] or DEFAULT
    ok = True
    for k in kernels:
        names = sorted(n for n in old if n.startswith(k + "(") or n.startswith(k + "<"))
        if not names:
            print(f"{k}: not found in the old build")
            ok = False
        for name in names:
            label = name.split("(")[0]
            if name not in new:
                print(f"{label}: not found in the new build")
                ok = False
                continue
            a, b = old[name], new[name]
            same = a == b
            ok &= same
            first = next((i for i, (x, y) in enumerate(zip(a, b)) if x != y), min(len(a), len(b)))
            print(f"{label}: {len(a)} vs {len(b)} instructions, " + ("identical" if same else f"first difference at {first}"))
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main(sys.argv))
