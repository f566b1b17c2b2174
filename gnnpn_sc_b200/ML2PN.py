"""Drop-in for ``src/ML2PN.py``: score the saved PNHigh picks against the optimum.

``check(dataset, serCategory, epoch)`` reads the same files (``allActions{epoch}.txt`` or the pretrained
stand-in, ``minCostList.data``) and prints ``epoch, mean(minCost / obj)``; the objective of every test
instance is evaluated in one launch of ``gnnpn_ml2pn_score_f64`` (ML2PN.py:6-12 per instance in numpy float64).
Neutral rows (categories the request does not use: ``[0,1,1,1]``, ML2PN.py:42) are dropped through the index table.
"""
from __future__ import annotations

import json
import os

import numpy as np
import torch

from . import ops
from .loadData import loadDataPN


def composition_scores(allActions, serCategory: int, constraints: np.ndarray) -> np.ndarray:
    """Score per instance exactly as ``ML2PN.calc`` (ML2PN.py:6-12) does it, float64 in numpy's operation order:
    ``0.5*(np.average(q0) + 1 - np.min(q1))``, then 1 added per violated global constraint, over the REAL picks of
    the instance (rows whose python ``sum`` is not 3 -- the neutral ``[0,1,1,1]`` of absent categories, ML2PN.py:42).
    ``allActions`` = K lists of [n_test][F] chosen rows; ``constraints`` [n_test, 4] = (lo1, hi1, lo2, hi2).
    One launch of ``gnnpn_ml2pn_score_f64`` for all instances."""
    acts = np.asarray([a for a in allActions[:serCategory]], dtype=np.float64)      # [K, n, F]
    K, n, _ = acts.shape
    rows = np.ascontiguousarray(np.transpose(acts, (1, 0, 2))[:, :, :4])              # [n, K, 4]
    psum = ((0.0 + rows[:, :, 0]) + rows[:, :, 1] + rows[:, :, 2]) + rows[:, :, 3]   # python sum(): left to right
    real = psum != 3
    klen = real.sum(axis=1).astype(np.int32)
    # indices of the real picks, packed to the front of every instance's row of the index table (stable order)
    order = np.argsort(~real, axis=1, kind="stable").astype(np.int64)
    idx = (np.arange(n, dtype=np.int64)[:, None] * K + order).astype(np.int32)
    out = np.zeros(n, dtype=np.float64)
    ok = klen > 0
    if not ok.any():
        return out
    dev = torch.device("cuda")
    _, _, score = ops.ml2pn_score(torch.from_numpy(rows.reshape(n * K, 4)).to(dev), torch.from_numpy(idx).to(dev),
                                  torch.from_numpy(np.asarray(constraints, dtype=np.float64)).to(dev),
                                  torch.from_numpy(np.maximum(klen, 1)).to(dev))
    out[ok] = score.cpu().numpy()[ok]
    return out


def check(dataset, serCategory, epoch, root="."):
    feats, _ = loadDataPN(epoch=-1, dataset=dataset, serviceNumber=1, root=root, rng=False)
    split = len(feats) // 4 * 3
    with open(os.path.join(root, "data", dataset, "minCostList.data")) as f:
        minCost = json.load(f)
    url = (os.path.join(root, "solutions", "pretrained", f"{dataset}-PNHigh.txt") if epoch == -1 else
           os.path.join(root, "solutions", "PNHigh", dataset, f"allActions{epoch}.txt"))
    with open(url) as f:
        allActions = json.load(f)
    cons = np.asarray([inst[0][5:9] for inst in feats[split:]], dtype=np.float64)
    obj = composition_scores(allActions, serCategory, cons)
    ratio = float(np.mean(np.asarray(minCost[split:split + len(obj)]) / obj))
    print(epoch, ratio)
    return ratio
