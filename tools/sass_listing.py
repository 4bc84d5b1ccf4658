#!/usr/bin/env python
"""profiles/r2_sass_<kernel>.txt: the SASS of the named kernels out of the built library
(cuobjdump -sass l-giremi_b200/liblgmi.so), one instruction per line without the encodings,
preceded by a mnemonic histogram and the tensor-core / TMA / async-copy mnemonics found.

    python tools/sass_listing.py [kernel ...]      # default: k_gram_i8 k_tile_gram_ws k_tile_finish k_pairs_fast"""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "l-giremi_b200", "liblgmi.so")
DEFAULT = ["k_gram_i8", "k_tile_gram_ws", "k_tile_finish", "k_pairs_fast"]
ASYNC = ("UTC", "LDTM", "STTM", "UTMA", "LDGSTS", "SYNCS", "UBLKCP")


def main():
    wanted = sys.argv[1:] or DEFAULT
    text = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True, check=True).stdout
    for part in re.split(r"\n\s*Function : ", text)[1:]:
        mangled = part.split("\n", 1)[0].strip()
        for key in wanted:
            if not re.search(r"\d+%sE" % key, mangled):
                continue
            lines, ops = [], collections.Counter()
            for m in re.finditer(r"^\s+/\*([0-9a-f]{4,5})\*/\s+(.*?;)", part, re.M):
                ins = m.group(2)
                lines.append("/*%s*/ %s" % (m.group(1), ins))
                op = re.sub(r"^@!?U?P\d+\s+", "", ins).split()[0].rstrip(";")
                ops[op] += 1
            found = sorted(op for op in ops if op.startswith(ASYNC))
            out = os.path.join(ROOT, "profiles", "r2_sass_%s.txt" % key)
            with open(out, "w") as fh:
                fh.write("SASS of %s (%s)\nfrom cuobjdump -sass l-giremi_b200/liblgmi.so, sm_100a; flags: l-giremi_b200/build.py\n"
                         % (key, mangled))
                fh.write("%d instructions; tensor-core / TMEM / TMA / async-copy / mbarrier mnemonics: %s\n"
                         % (sum(ops.values()), ", ".join("%s x%d" % (op, ops[op]) for op in found) or "none"))
                fh.write("mnemonic histogram:\n")
                for op, n in ops.most_common():
                    fh.write("  %-34s %6d\n" % (op, n))
                fh.write("\n" + "\n".join(lines) + "\n")
            print(out, sum(ops.values()), found)


if __name__ == "__main__":
    main()
