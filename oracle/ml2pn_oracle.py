"""TEST INFRASTRUCTURE (oracle): CPU restatement of ``src/ML2PN.py`` -- never imported by the product path.

``calc`` follows ML2PN.py:6-12 and ``scores`` the list handling of ``check`` (ML2PN.py:34-56): python lists of
python floats (the JSON the trainers wrote), numpy float64 reductions.
"""
from __future__ import annotations

import numpy as np


def calc(qos, cons):
    """ML2PN.py:6-12."""
    obj = 0.5 * (np.average(qos[0]) + 1 - np.min(qos[1]))
    for j in range(2):
        v = np.cumprod(qos[2 + j])[-1]
        if v < cons[j][0] or v > cons[j][1]:
            obj += 1
    return obj


def scores(allActions, serCategory, constraints, tag=0, qosNum=4):
    """Per-instance ``calc`` value of the saved picks: ML2PN.py:34-56 without the file I/O.
    ``allActions`` = K lists of [n][F] rows (python floats); ``constraints`` [n][4] = (lo1, hi1, lo2, hi2)."""
    n = len(allActions[0])
    out = []
    for j in range(n):
        sol = [allActions[i][j][tag: tag + qosNum] for i in range(serCategory)]
        sol = [a for a in sol if sum(a) != 3]                                     # ML2PN.py:42
        qos = [[s[i] for s in sol] for i in range(qosNum)]
        c = constraints[j]
        out.append(calc(qos, [[c[0], c[1]], [c[2], c[3]]]))
    return np.asarray(out, dtype=np.float64)
