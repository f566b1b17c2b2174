"""Host-side data layer (gnnpn_sc_b200/loadData.py) against structural invariants."""
import json
import os

import numpy as np
import pytest

from gnnpn_sc_b200 import loadData as ld
from gnnpn_sc_b200 import synth


@pytest.fixture(scope="module")
def tiny(tmp_path_factory):
    root = tmp_path_factory.mktemp("ds")
    ds = synth.ml_dataset(n_instances=12, K=7, S=70, seed=5, min_tasks=3)
    synth.write_dataset(str(root), "tiny", ds)
    rng = np.random.default_rng(0)
    rankings = [rng.permutation(70).tolist() for _ in range(12)]
    os.makedirs(root / "solutions" / "ML" / "tiny", exist_ok=True)
    with open(root / "solutions" / "ML" / "tiny" / "testServices-epoch0.txt", "w") as f:
        json.dump(rankings, f)
    return root, ds


def test_pn_rows_layout(tiny):
    root, ds = tiny
    feats, labels = ld.loadDataPN(0, "tiny", 3, root=str(root), rng=False)
    assert len(feats) == 12 and labels == ds["minCostList"]
    a = np.asarray(feats[0])
    assert a.shape == (7 * 3, 9)
    assert (a[:, 0] == np.repeat(np.arange(7), 3)).all()
    assert (a[3:, 5:] == 0).all()                                   # global bounds only on category 0 rows
    neutral = (a[:, 1:5] == [0, 1, 1, 1]).all(axis=1)
    used = {int(np.argmax(np.asarray(n[:-6]) == 1)) for n in ds["nodefeatures"][0] if n[0] != 1}
    assert set(np.unique(a[~neutral, 0]).astype(int) + 1) <= used
