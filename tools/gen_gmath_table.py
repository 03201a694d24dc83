#!/usr/bin/env python
"""gmath_coeffs.inc -> gmath_table.inc: the coefficient literals as one table (device: __constant__ memory) and the
index of each name; the words of 2/pi as a second table.  Run after tools/gen_gmath_coeffs.py."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "gelato_b200", "csrc")


def main():
    inc = open(os.path.join(CSRC, "gmath_coeffs.inc")).read()
    names = [m.group(1) for m in re.finditer(r"#define (GM_[A-Z0-9_]+) [(]", inc)]
    out = ["/* GENERATED from gmath_coeffs.inc by tools/gen_gmath_table.py -- do not edit by hand.",
           " * The same literals as one table: on the device it lives in __constant__ memory, so that a polynomial",
           " * step is one DFMA with a constant-bank operand (one LDCU.128 per two coefficients) instead of a DFMA plus",
           " * two 32-bit immediate moves per coefficient (ncu r02a: 27 % of the executed instructions were moves). */",
           "#define GM_TAB_N %d" % len(names), "#define GM_TAB_INIT { \\"]
    for i in range(0, len(names), 4):
        out.append("  " + ", ".join(names[i:i + 4]) + (", \\" if i + 4 < len(names) else " \\"))
    out.append("}")
    out += ["#define GMT_%s %d" % (nm[3:], i) for i, nm in enumerate(names)]
    # the words of 2/pi (integers, not operands of the polynomials): a table of their own
    words = [m.group(1) for m in re.finditer(r"#define (GM_2OPI_W[0-9]+) 0x", inc)]
    out += ["#define GM_2OPI_N %d" % len(words), "#define GM_2OPI_INIT { \\"]
    for i in range(0, len(words), 4):
        out.append("  " + ", ".join(words[i:i + 4]) + (", \\" if i + 4 < len(words) else " \\"))
    out.append("}")
    open(os.path.join(CSRC, "gmath_table.inc"), "w").write("\n".join(out) + "\n")


if __name__ == "__main__":
    main()
