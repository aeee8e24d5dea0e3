#!/usr/bin/env python
"""Generates tests/golden/hiddengem_tables/*: the hiddengem output that test_cli_gpu.py expects for its
adversarial-tie tables and its 12,000-bin table.

The expected output is the reference's Viterbi recurrence (src/hiddengem.c:51-147, 246-283) as restated in
oracle/ibdgem_oracle.c (orc_hiddengem), which tests/test_oracle_refruns.py pins byte for byte against the
reference's own hiddengem stdout.  The tables go through the same text round trip as on the command line:
written with %e, parsed back as doubles.  Scores are printed like the reference's %.5Le, subnormal long doubles
included.

Per table, <name>.states.txt holds the Inferred_State column as one line of digits followed by the three
"#% IBDk" lines; long.rows.txt holds every 10th row of the long table's output (segment, three scores, state).

Run from the repository root after `make -C oracle oracle`:  python tests/golden/make_hiddengem_golden.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import oracle  # noqa: E402
from test_cli_gpu import HG_GOLDEN, TIE_PENALTIES, _long_table, _tie_tables  # noqa: E402


def _text_round_trip(l):
    return np.array([[float("%e" % x) for x in row] for row in l])


def _le(x):
    return np.format_float_scientific(np.longdouble(x), precision=5, unique=False, exp_digits=2)


def write(name, l, pen, rows_every=0):
    state, _, score = oracle.hiddengem(_text_round_trip(l), *pen)
    n = len(state)
    counts = ["#%% IBD%d (n = %d): %.2f" % (s, int((state == s).sum()), (state == s).sum() / n * 100) for s in range(3)]
    with open(os.path.join(HG_GOLDEN, name + ".states.txt"), "w") as fh:
        fh.write("".join(str(s) for s in state) + "\n" + "\n".join(counts) + "\n")
    if rows_every:
        with open(os.path.join(HG_GOLDEN, name + ".rows.txt"), "w") as fh:
            for i in range(0, n, rows_every):
                fh.write("%d\t%s\t%s\t%s\t%d\n" % (i + 1, *[_le(score[i, s]) for s in range(3)], state[i]))


def main():
    os.makedirs(HG_GOLDEN, exist_ok=True)
    for k, l in enumerate(_tie_tables()):
        for tag, args in TIE_PENALTIES.items():
            write(f"tie{k}.{tag}", l, [float(a) for a in args[1::2]])
    write("long", _long_table(), [], rows_every=10)
    print("hiddengem golden tables written to", HG_GOLDEN)


if __name__ == "__main__":
    main()
