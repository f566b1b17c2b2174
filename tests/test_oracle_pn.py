"""The PN oracle (oracle/pn_oracle.py) is pinned against fixtures produced by the
real reference (oracle/make_golden.py)."""
import os

import numpy as np
import pytest
import torch

from oracle import make_golden as mg
from oracle import pn_oracle as po

CASE_NAMES = list(mg.CASES)


def _run_oracle(name, faithful=False):
    kw, B, (s_lo, s_hi), s_in, gain, dist = mg.CASES[name]
    cfg = mg.case_config(name)
    x = mg.build_inputs(cfg, B, s_in, dist)
    sd_lo, sd_hi = po.make_state_dict(cfg, s_lo, gain), po.make_state_dict(cfg, s_hi, gain)
    res = po.greedy_low_high(sd_lo, sd_hi, cfg, x, faithful_loops=faithful)
    res["reward_high"] = po.reward(list(res["actions"]), None, cfg.s_category, "High", cfg.embedding_size)
    res["viol_high"] = po.reward(list(res["actions"]), None, cfg.s_category, "Low", cfg.embedding_size)
    return cfg, res


@pytest.mark.parametrize("name", CASE_NAMES)
def test_oracle_matches_reference_fixture(name, golden_dir):
    g = np.load(os.path.join(golden_dir, f"pn_{name}.npz"))
    cfg, res = _run_oracle(name)
    # selections: exact
    assert np.array_equal(res["idx_low"].numpy(), g["idx_low"])
    assert np.array_equal(res["idx_high"].numpy(), g["idx_high"])
    # -inf pattern (visited mask) bit-exact, finite logits to fp32 round-off of the same library
    for key_o, key_g in (("latent", "logits_low"), ("logits_high", "logits_high")):
        a, b = res[key_o].numpy(), g[key_g]
        assert np.array_equal(np.isneginf(a), np.isneginf(b))
        fin = np.isfinite(b)
        np.testing.assert_allclose(a[fin], b[fin], rtol=0, atol=2e-6)
    np.testing.assert_allclose(res["action_probs"].numpy(), g["action_probs_high"], rtol=1e-5, atol=1e-7)
    assert np.array_equal(res["actions"].numpy(), g["actions_high"])
    # reward / objective evaluator: exact (fp32 sequential products + python round)
    assert np.array_equal(res["reward_high"].numpy(), g["reward_high"])
    assert np.array_equal(res["viol_high"].numpy(), g["viol_high"])
    tag = 1 if cfg.embedding_size else 0
    _, obj = po.composition_objective(res["actions"].numpy(), tag)
    assert np.array_equal(obj, g["objfunc_high"])          # unrounded objFunc of the reference's calc()


def test_faithful_loops_same_result():
    _, a = _run_oracle("small_b16", faithful=False)
    _, b = _run_oracle("small_b16", faithful=True)
    for k in a:
        assert torch.equal(a[k], b[k]), k


def test_structural_facts_the_kernels_rely_on(golden_dir):
    """SURVEY 3.4: probs are exactly 0 outside window k; step-k logits carry -inf at the
    k previously chosen positions; selections stay inside their window."""
    g = np.load(os.path.join(golden_dir, "pn_qws_b4.npz"))
    K, B, L = g["logits_low"].shape
    N = L // K
    for k in range(K):
        assert ((g["idx_low"][k] >= k * N) & (g["idx_low"][k] < (k + 1) * N)).all()
        assert np.isneginf(g["logits_low"][k]).sum(axis=1).tolist() == [k] * B
    p = g["probs_high_step1"]
    assert (p[:, :N] == 0).all() and (p[:, 2 * N:] == 0).all()
    np.testing.assert_allclose(p.sum(axis=1), 1.0, atol=1e-6)


def test_teacher_forcing_returns_free_choice():
    cfg = mg.case_config("small_b16")
    x = mg.build_inputs(cfg, 16, 7, "qws")
    sd = po.make_state_dict(cfg, 105)
    with torch.no_grad():
        _, idx, lg = po.pointer_forward(sd, cfg, x, None, "greedy")
        _, idx2, lg2 = po.pointer_forward(sd, cfg, x, None, "greedy", forced_idxs=idx)
    assert all(torch.equal(a, b) for a, b in zip(idx, idx2))
    assert all(torch.equal(a, b) for a, b in zip(lg, lg2))


@pytest.mark.parametrize("name", CASE_NAMES)
def test_oracle_bitwise_equals_reference_fixture(name, golden_dir):
    """Same ATen ops in the same shapes as the reference -> the same bits as the reference's own fp32 run, which the
    fixture stores."""
    gold = np.load(os.path.join(golden_dir, f"pn_{name}.npz"))
    _, res = _run_oracle(name)
    assert np.array_equal(res["idx_high"].numpy(), gold["idx_high"])
    assert np.array_equal(res["latent"].numpy(), gold["logits_low"])
    assert np.array_equal(res["logits_high"].numpy(), gold["logits_high"])
    assert np.array_equal(res["reward_high"].numpy(), gold["reward_high"])
