"""oracle/ml2pn_oracle.py: the objective of ``ML2PN.calc`` restated."""
from oracle import ml2pn_oracle as mo


def test_mean_runs_over_all_real_picks():
    acts = [[[0.0, 0.5, 1.0, 1.0, 0, 0, 0, 0]], [[0.6, 0.25, 1.0, 1.0, 0, 0, 0, 0]]]
    s = mo.scores(acts, 2, [[0.0, 2.0, 0.0, 2.0]])
    assert s[0] == 0.5 * (0.3 + 1 - 0.25)        # ESWOA.calc would divide by the one pick with q0 > 0
