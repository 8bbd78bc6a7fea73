#!/usr/bin/env python
"""Regenerate tests/golden/*.npz from the REFERENCE's own code (oracle/_ref, built where the
reference sources are available); the tests fall back to these files where libhnh_ref.so is absent.
The small multi-rank cases are stored whole; every other reference output the tests compare with
is stored in the reduced form of tests/golden_util.py, which keeps each file small."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref  # noqa: E402
from tests import golden_util as G  # noqa: E402
from tests import mp_util as U  # noqa: E402
from tests import test_algorithms_gpu as TA  # noqa: E402
from tests import test_multirank_gpu as TG  # noqa: E402
from tests.test_multirank_cpu import CASES_2, CASES_4, CASES_8  # noqa: E402

assert ref.build(), "oracle/_ref could not be built (are the reference sources present?)"
os.makedirs(os.path.join(ROOT, "tests", "golden"), exist_ok=True)
U.WRITE_GOLDEN = True

whole = [(2, c) for c in CASES_2 if c["logM"] <= 9] + [(4, c) for c in CASES_4] + \
    [(p, c) for p, cs in TG.CASES.items() for c in cs]
reduced = [(2, c) for c in CASES_2] + [(8, c) for c in CASES_8] + [(p, c) for p, cs in TG.CASES.items() for c in cs] + \
    [(p, c) for p, cs in TG.RECT_CASES.items() for c in cs] + [(4, c) for c in TG.TINY_CASES] + \
    [(1, c) for c in TG.DEVSETUP_CASES[1]]
gpu = [(p, c) for p, cs in TG.CASES.items() for c in cs] + [(p, c) for p, cs in TG.RECT_CASES.items() for c in cs] + \
    [(4, c) for c in TG.TINY_CASES] + [(p, c) for p, cs in TG.DEVSETUP_CASES.items() for c in cs]
seen = set()
for p, c in whole + reduced:
    key = (c["name"], p)
    if key in seen:
        continue
    seen.add(key)
    # the cases with generated names, small enough to be stored whole (the others have names of their own)
    small = (p, c) in whole and c["name"].startswith(c["alg"])
    if not any(c["name"] == g["name"] and p == q for q, g in gpu):
        c = dict(c, script=[])  # only the layout is compared
    ranks, _ = U.reference_for(c, p)
    path = os.path.join(ROOT, "tests", "golden", f"{c['name']}_p{p}.npz")
    if small:
        np.savez_compressed(path, **U.flatten_ref(ranks))
    else:
        G.save(path, U.flatten_ref(ranks, reduced=True, alg=c["alg"]))
    print(path, os.path.getsize(path))

for p, cs in TG.GAT_CASES.items():
    for c in cs:
        TG.gat_reference(c, p)
for p, cs in TG.ALS_CASES.items():
    for c in cs:
        TG.als_reference(c, p)
for name in TA.ALGS:
    TA.p1_als_reference(name)
# the oracle's pins: every test of test_oracle_vs_ref.py writes what it compares with
import pytest  # noqa: E402
sys.exit(pytest.main(["-q", "-p", "no:cacheprovider", os.path.join(ROOT, "tests", "test_oracle_vs_ref.py")]))
