"""Regenerates tests/golden/gc_data.py from a checkout of the OCaml reference (farr/mcmc-ocaml):
    python tests/golden/make_gc_data.py <reference checkout>
The tests only read the output."""
import os
import re
import sys

src = open(os.path.join(sys.argv[1], "bin", "gaussian_cauchy_efficiency.ml")).read()
m = re.search(r"let data = \[\|(.*?)\|\]", src, re.S)
vals = [float(v) for v in m.group(1).replace("\n", " ").split(";") if v.strip()]
assert len(vals) == 100
open(__file__.replace("make_gc_data.py", "gc_data.py"), "w").write(
    '"""The fixed 100-point dataset of bin/gaussian_cauchy_efficiency.ml:33-48 (input data of\n'
    'BASELINE.json config 1), extracted by tests/golden/make_gc_data.py."""\nDATA = ' + repr(vals) + "\n")
