"""GPU tests of the callers either side of the hot path: sampled decode, REINFORCE replay gradients,
PNLow/PNHigh trainers, ML2PN scoring."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import pn_oracle as po

pytestmark = pytest.mark.gpu


def _model(K, N, level="Low", seed=1, H=256):
    from gnnpn_sc_b200 import modelPN as M
    cfg = po.PNConfig(hidden_size=H, seq_len=K * N, s_number=N, s_category=K)
    m = M.CombinatorialRL(0, H, K * N, 0, 10, 1, M.reward, "Dot", N, K, level=level)
    sd = po.make_state_dict(cfg, seed)
    m.load_state_dict(sd)
    return cfg, sd, m.cuda()


def test_sampled_decode_follows_the_window_distribution():
    from gnnpn_sc_b200.synth import pn_instances
    K, N = 4, 5
    cfg, sd, m = _model(K, N)
    x = pn_instances(1, K, N, seed=3).repeat(20000, 1, 1).cuda()         # same instance 20k times
    m.eval()
    m.actor.generator = torch.Generator(device="cuda").manual_seed(5)      # fixed draws
    with torch.no_grad():
        probs, idx, _ = m.actor(x, None, sample="sample")
    idx = torch.stack(idx)
    assert bool(((idx >= torch.arange(K, device="cuda").view(K, 1) * N) & (idx < torch.arange(1, K + 1, device="cuda").view(K, 1) * N)).all())
    # step 0 is identical across the copies: empirical pick frequencies ~ its softmax
    p0 = probs.window[0, :N].cpu().numpy()
    freq = np.bincount(idx[0].cpu().numpy(), minlength=N)[:N] / idx.shape[1]
    assert np.abs(freq - p0).max() < 0.015, (freq, p0)
    assert len(set(idx[0].tolist())) > 1                                   # actually stochastic


@pytest.mark.parametrize("impl,K,N,B,high", [("own", 6, 4, 16, False), ("own", 6, 4, 16, True), ("own", 47, 5, 40, True),
                                              ("own", 5, 10, 130, False), ("torch", 6, 4, 16, False)])
def test_replay_gradient_equals_oracle_autograd(impl, K, N, B, high):
    """d/dtheta of sum_k log p_k(action_k) through replay_action_probs == autograd through the oracle's graph.
    impl = "own": forward-with-saves + BPTT on the library's kernels (gnnpn_pn_train_*); "torch": the torch replay kept
    for the non-default variants.  `high`: with PNLow's latent added to the logits (trainPNHigh.py:83-84)."""
    from gnnpn_sc_b200.synth import pn_instances
    from conftest import record_parity
    cfg, sd, m = _model(K, N, seed=5)
    x = pn_instances(B, K, N, seed=2)
    g = torch.Generator().manual_seed(9)
    latent = [torch.randn(B, K * N, generator=g) for _ in range(K)] if high else None
    sd_g = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    probs, idx, _ = po.pointer_forward(sd_g, cfg, x, latent, "greedy")
    w = torch.rand(B, generator=g) - 0.3                                   # per-instance advantage
    logp = (w * sum(torch.log(p[torch.arange(B), a]) for p, a in zip(probs, idx))).sum()
    logp.backward()
    m.train()
    m.actor.replay_impl = impl
    idx_c = torch.stack(idx).cuda()
    lat_win = None
    if high:
        dense = torch.stack(latent)                                        # [K, B, L] -> compact window form [B, L]
        lat_win = dense.view(K, B, K, N).diagonal(dim1=0, dim2=2).permute(0, 2, 1).reshape(B, K * N).contiguous().cuda()
    ap = m.actor.replay_action_probs(x.cuda(), idx_c, lat_win)
    (w.cuda() * sum(torch.log(p) for p in ap)).sum().backward()
    worst = 0.0
    for name, p in m.named_parameters():
        g_ref = sd_g[name].grad
        d = (p.grad.cpu() - g_ref).abs().max() / g_ref.abs().max().clamp(min=1e-3)
        worst = max(worst, float(d))
    print(f"replay gradient [{impl}, K={K}, N={N}, B={B}, high={high}] max relative deviation vs oracle autograd: {worst:.2e}")
    record_parity(f"reinforce_gradient_{impl}_K{K}_N{N}_B{B}_{'high' if high else 'low'}", max_rel_dev=worst, tolerance=1e-4)
    assert worst < 1e-4


@pytest.mark.parametrize("B,K,N", [(128, 47, 5), (37, 6, 4), (16, 3, 2), (130, 5, 10)])
def test_bptt_cluster_scan_equals_per_step_kernels(B, K, N):
    """The persistent cluster BPTT (pn_bptt.cu, option bptt = 1) against the per-step kernels it replaces (bptt = 0) on the
    same saves: gate gradients of every (step, instance, gate row) agree to fp32 re-association (the dh GEMM sums its k
    chunks in a different fixed order), ragged batches included; the scan is deterministic."""
    from gnnpn_sc_b200 import ops
    from gnnpn_sc_b200.synth import pn_instances
    cfg, sd, m = _model(K, N, seed=6)
    x = pn_instances(B, K, N, seed=3).cuda()
    g = torch.Generator(device="cuda").manual_seed(1)
    idx = (torch.arange(K, device="cuda").view(K, 1) * N + torch.randint(0, N, (K, B), device="cuda", generator=g)).to(torch.int32)
    enc_w, dec_w = m.actor._packed_weights()
    sv = ops.pn_train_forward(x, enc_w, dec_w, idx, K, N)
    gp = torch.rand(K, B, device="cuda", generator=g) - 0.4
    whe, whd = m.actor.encoder.weight_hh_l0.detach(), m.actor.decoder.weight_hh_l0.detach()
    try:
        ops.set_option("bptt", 0)
        ref_e, ref_d = [t.clone() for t in ops.pn_train_backward(sv, gp, whe, whd, K, N)]
        ops.set_option("bptt", 1)
        got_e, got_d = [t.clone() for t in ops.pn_train_backward(sv, gp, whe, whd, K, N)]
        again_e, again_d = ops.pn_train_backward(sv, gp, whe, whd, K, N)
    finally:
        ops.set_option("bptt", 1)
    assert torch.equal(got_e, again_e) and torch.equal(got_d, again_d)
    for got, ref in ((got_e, ref_e), (got_d, ref_d)):
        scale = float(ref.abs().max())
        assert scale > 0
        assert float((got - ref).abs().max()) <= 2e-6 * scale, float((got - ref).abs().max()) / scale


def test_training_batch_outside_the_column_split_scan_falls_back_to_the_replay():
    """A training batch the column-split scan does not take (> 30 groups of 128) decodes on the CTA-pair scan and replays
    teacher-forced on the strict-fp32 kernels; its gradient equals the sum over two half batches, which DO take the fused
    decode-with-saves path -- to the difference between the tensor-core and the FFMA forward arithmetic."""
    from gnnpn_sc_b200.synth import pn_instances
    K, N, B = 6, 4, 3968
    cfg, sd, m = _model(K, N, seed=8)
    x = pn_instances(B, K, N, seed=12).cuda()
    m.train()
    m.actor.generator = torch.Generator(device="cuda").manual_seed(3)
    R, ap, _, idx, _ = m(x, None, sample="greedy", training="RL")
    assert m.actor._train_saves is None                                    # the fused path refused this batch
    sum(torch.log(p) for p in ap).sum().backward()
    g_full = {n_: p.grad.clone() for n_, p in m.named_parameters()}
    m.zero_grad()
    for lo, hi in ((0, B // 2), (B // 2, B)):
        _, ap_h, _, idx_h, _ = m(x[lo:hi].contiguous(), None, sample="greedy", training="RL")
        assert torch.equal(torch.stack(idx_h), torch.stack(idx)[:, lo:hi])   # same picks on both scans (bit-identical decodes)
        sum(torch.log(p) for p in ap_h).sum().backward()
    worst = max(float((p.grad - g_full[n_]).abs().max() / g_full[n_].abs().max().clamp(min=1e-3)) for n_, p in m.named_parameters())
    assert worst < 1e-4, worst


def test_reinforce_gradient_other_hidden_size():
    """hidden_size = 128: the sampled decode runs on the any-hidden-size kernels, the gradient on the torch replay; it
    equals autograd through the oracle's graph on the same picks."""
    from gnnpn_sc_b200.synth import pn_instances
    K, N, B = 6, 4, 12
    cfg, sd, m = _model(K, N, seed=4, H=128)
    x = pn_instances(B, K, N, seed=8)
    m.train()
    m.actor.generator = torch.Generator(device="cuda").manual_seed(17)      # fixed draws: the test must not depend on what ran before
    R, ap, _, idx, _ = m(x.cuda(), None, sample="sample", training="RL")
    idx_cpu = [t.cpu() for t in idx]
    sd_g = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    probs, _, _ = po.pointer_forward(sd_g, cfg, x, None, "greedy", forced_idxs=idx_cpu)
    sum(torch.log(p[torch.arange(B), a]) for p, a in zip(probs, idx_cpu)).sum().backward()
    sum(torch.log(p) for p in ap).sum().backward()
    worst = max(float((p.grad.cpu() - sd_g[name].grad).abs().max() / sd_g[name].grad.abs().max().clamp(min=1e-3))
                for name, p in m.named_parameters())
    assert worst < 1e-4, worst


def _toy_pn_data(n, K, N, seed=0):
    from gnnpn_sc_b200.synth import pn_instances
    x = pn_instances(n, K, N, seed=seed)
    cat = torch.arange(K).repeat_interleave(N).float().view(1, -1, 1).expand(n, -1, 1)
    feats = torch.cat([cat, x], dim=2).tolist()                            # loadDataPN rows: [cat, 8 values]
    return feats, [0.5] * n


def test_pnlow_then_pnhigh_trainers_and_ml2pn(tmp_path):
    from gnnpn_sc_b200 import trainPN
    K, N = 6, 4
    data = _toy_pn_data(64, K, N)
    root = str(tmp_path)
    low = trainPN.PNLow("toy", 0, 1, K, 1, N, 256, 0, 10, 1, 0.9, 2.0, 1e-4, -1, root=root)
    tr = low.start(data=data, n_epochs=2)
    assert len(tr.train_tour) == 2 and len(tr.val_tour) == 2
    ck = torch.load(os.path.join(root, "solutions", "PNLow", "toy", "epoch1.model"))
    assert set(ck) == {"epoch", "model", "optimizer"}
    with open(os.path.join(root, "solutions", "PNLow", "toy", "allActions1.txt")) as f:
        acts = json.load(f)
    assert len(acts) == K + 2 and len(acts[0]) == 16 and len(acts[0][0]) == 8      # K+2 slots (trainPNLow.py:122)
    before = {k: v.clone() for k, v in ck["model"].items()}
    high = trainPN.PNHigh("toy", 0, 1, K, 1, N, 256, 0, 10, 1, 0.9, 2.0, 5e-5, -1, -1, root=root)
    th = high.start(data=data, n_epochs=1, low_state=ck["model"])
    assert os.path.exists(os.path.join(root, "solutions", "PNHigh", "toy", "epoch0_low.model"))
    with open(os.path.join(root, "solutions", "PNHigh", "toy", "allActions0.txt")) as f:
        acts_h = json.load(f)
    assert len(acts_h) == K
    # PNLow's weights are not stepped by PNHigh training (only model.actor is in the optimiser, trainPNHigh.py:62)
    after = th.low_model.state_dict()
    assert all(torch.equal(before[k].cpu(), after[k].cpu()) for k in before)
    # ML2PN scoring of the saved picks == ML2PN.calc restated (oracle/ml2pn_oracle.py), float64 EXACT; a pick with
    # q0 == 0 is injected: ML2PN.calc averages over all real picks (np.average), unlike modelPN.calc
    from gnnpn_sc_b200 import ML2PN
    from oracle import ml2pn_oracle as mo
    x = torch.tensor(data[0])[48:, :, 1:]                                  # validation quarter
    cons = x[:, 0, 4:8].double().numpy()
    acts_h[1][0][0] = 0.0
    got = ML2PN.composition_scores(acts_h, K, cons)
    want = mo.scores(acts_h, K, cons.tolist())
    assert np.array_equal(got, want)
    with open(os.path.join(root, "solutions", "PNLow", "toy", "allR1.txt")) as f:
        allR = json.load(f)                                                # trainPNLow.py:123-141
    assert set(allR) == {"quality", "averageQ"} and len(allR["quality"]) == 16
    assert allR["averageQ"] == sum(allR["quality"]) / 16


def test_reinforce_step_reduces_loss_surrogate(tmp_path):
    """A few REINFORCE updates on one batch move the sampled reward mean down (sanity of sign and plumbing)."""
    from gnnpn_sc_b200 import trainPN
    K, N = 5, 4
    torch.manual_seed(0)
    data = _toy_pn_data(256, K, N, seed=4)
    low = trainPN.PNLow("toy", 0, 1, K, 1, N, 256, 0, 10, 1, 0.9, 2.0, 3e-3, -1, root=str(tmp_path))
    tr = low.start(data=data, n_epochs=16)
    first, last = np.mean(tr.train_tour[:6]), np.mean(tr.train_tour[-6:])
    print(f"mean sampled reward (violations): first epochs {first:.3f} -> last epochs {last:.3f}")
    assert last <= first + 0.05
