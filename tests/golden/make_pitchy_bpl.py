"""Regenerates tests/golden/pitchy_bpl_2k.npz and its stability companion (TEST INFRASTRUCTURE).

    python tests/golden/make_pitchy_bpl.py

The generators of make_golden.py (2048 points of the sampler configuration pitchy_bpl, the sequential draw
of the 2k fixtures) and make_stability.py, run on the oracle with the pitchy broken power law
(tests/bpl_oracle).  About 400 s and 850 s on 8 threads.
"""
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))

import bpl_oracle  # noqa: E402
import make_golden  # noqa: E402
import make_stability  # noqa: E402

NAME = "pitchy_bpl_2k"

if __name__ == "__main__":
    make_golden.O = make_stability.O = bpl_oracle
    make_golden.FIXTURES[NAME] = ("pitchy_bpl", 2048)
    make_golden.run(NAME)
    sys.argv = [sys.argv[0], NAME]
    make_stability.main()
