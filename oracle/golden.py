"""Readers of stored vectors under tests/golden that take more than one np.load -- TEST INFRASTRUCTURE ONLY
(tests/, bench.py, tools/)."""
import os

import numpy as np

GOLD = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def allscales_full_bank():
    """The reference's allScales bank (test/case1/allScales, all 2989 templates) as (packed dict of int32 class_begin /
    tmeta / feats, T).  Its features are stored in two files, split at a template boundary, so that every stored file
    stays under 1 MB (tests/golden/make_golden.py)."""
    a, b = (np.load(os.path.join(GOLD, "bank_allScales_full_%s.npz" % part)) for part in "ab")
    packed = dict(class_begin=a["class_begin"], tmeta=a["tmeta"].astype(np.int32),
                  feats=np.concatenate([a["feats"], b["feats"]]).astype(np.int32))
    last = packed["tmeta"][-1, -1]
    if int(last[2] + last[3]) != packed["feats"].shape[0]:
        raise RuntimeError("bank_allScales_full_{a,b}.npz do not belong together")
    return packed, a["T"].tolist()
