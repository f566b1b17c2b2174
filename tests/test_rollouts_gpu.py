"""Best-of-R sampled decoding: R rollouts of every instance from one set of encodings (gnnpn_pn_decode_rollouts_f32), the
best rollout by the exact reward (gnnpn_pn_best_rollout_f32), and the pipeline stages built on them.

Every rollout must be the single decode the library already does, bit for bit, on every decoder kind, and the best
rollout must be the minimum of gnnpn_pn_reward_f32 over the rollouts with ties to the lowest rollout."""

import numpy as np
import pytest
import torch

from oracle import pn_oracle as po


@pytest.fixture(autouse=True)
def _reset_options():
    yield
    if torch.cuda.is_available():
        from gnnpn_sc_b200 import ops
        ops.set_option("scan", -1)
        ops.set_option("scan_groups", 0)
        ops.set_option("persistent", 3)


def _net(K, N, level="High", seed=2, C=10):
    from gnnpn_sc_b200 import modelPN as M
    cfg = po.PNConfig(seq_len=K * N, s_number=N, s_category=K)
    m = M.CombinatorialRL(0, 256, K * N, 0, C, 1, M.reward, "Dot", N, K, level=level)
    m.load_state_dict(po.make_state_dict(cfg, seed))
    return m.cuda().eval()


# (name, n, K, N, R, scan, scan_groups): the decoder kind each case runs
KINDS = [
    ("fused_nr5", 300, 6, 5, 3, 0, 0),          # blocked encodings, lstm_seq_kernel<true, 5>
    ("fused_nr8", 300, 5, 7, 3, 0, 0),          # <true, 8>
    ("fused_nr10", 200, 4, 10, 2, 0, 0),        # <true, 10>
    ("rowmajor_n11", 200, 3, 11, 3, 0, 0),      # row-major CTA-pair decoder <true, 0>
    ("rowmajor_n32", 150, 3, 32, 2, 0, 0),
    ("colsplit_g1", 200, 5, 5, 3, 1, 1),        # lstm_colsplit_kernel<true, 1>
    ("colsplit_g2", 300, 5, 5, 3, 1, 2),        # <true, 2>
    ("auto_cross", 1000, 4, 5, 4, -1, 0),       # column-split encoder for n, n * R past the column-split limit
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,n,K,N,R,scan,groups", KINDS, ids=[k[0] for k in KINDS])
def test_rollouts_equal_single_decodes(name, n, K, N, R, scan, groups):
    """Rollout r == gnnpn_pn_decode_greedy_f32 on the same encodings and c_state with rollout r's uniforms (rollout 0:
    none): idx, win_logits, win_probs bit-identical; c_state untouched; one encodings buffer of n instances."""
    from gnnpn_sc_b200 import ops
    from gnnpn_sc_b200.synth import pn_instances
    ops.set_option("scan", scan)
    ops.set_option("scan_groups", groups)
    m = _net(K, N)
    actor = m.actor
    actor.generator = torch.Generator(device="cuda").manual_seed(7)
    x = pn_instances(n, K, N, seed=n + K).cuda()
    L = K * N
    lat = torch.randn(n, L, device="cuda", generator=torch.Generator(device="cuda").manual_seed(3))
    enc = actor.encode(x)
    c0 = enc.c.clone()
    idx, wl, wp = actor.decode_rollouts(x, None, R, encoded=enc)
    assert idx.shape == (R, K, n) and wl.shape == (R, n, L)
    assert enc.enc_out.numel() == ops.enc_out_floats(n, L, 256, enc.layout)      # not replicated R times
    assert torch.equal(enc.c, c0)
    # uniforms the rollouts drew from: the same generator state again
    uni = torch.rand(R - 1, K, n, device="cuda", generator=torch.Generator(device="cuda").manual_seed(7))
    _, dec_w = actor._weights()
    kw = dict(use_tanh=True, C=10.0, workspace=enc.ws, enc_layout=enc.layout, hidden=256)
    for r in range(R):
        _, i1, l1, p1 = ops.pn_decode_greedy(x, enc.enc_out, c0.clone(), dec_w, K, N,
                                             sample_uniform=uni[r - 1] if r else None, **kw)
        assert torch.equal(idx[r], i1), (name, r)
        assert torch.equal(wl[r], l1) and torch.equal(wp[r], p1), (name, r)
    # with a latent (PNHigh) on the same kernels
    idx_l, wl_l, _ = ops.pn_decode_rollouts(x, enc.enc_out, c0, dec_w, K, N, R, sample_uniform=uni, latent_win=lat,
                                            use_tanh=True, C=10.0, enc_layout=enc.layout)[1:]
    for r in range(R):
        _, i1, l1, _ = ops.pn_decode_greedy(x, enc.enc_out, c0.clone(), dec_w, K, N, latent_win=lat,
                                            sample_uniform=uni[r - 1] if r else None, **kw)
        assert torch.equal(idx_l[r], i1) and torch.equal(wl_l[r], l1), (name, "latent", r)


@pytest.mark.gpu
@pytest.mark.parametrize("level", ["Low", "High"])
def test_best_rollout_is_the_minimum_reward_lowest_rollout_on_ties(level):
    from gnnpn_sc_b200 import ops
    from gnnpn_sc_b200.synth import pn_instances
    n, K, N, R = 333, 9, 5, 7
    x = pn_instances(n, K, N, seed=5).cuda()
    g = torch.Generator(device="cuda").manual_seed(11)
    idx = (torch.randint(0, N, (R, K, n), device="cuda", generator=g)
           + N * torch.arange(K, device="cuda").view(1, K, 1)).to(torch.int32)
    idx[3] = idx[1]                                           # exact ties between rollouts
    idx[5] = idx[0]
    best_idx, best, rollout, rews = ops.pn_best_rollout(x, idx, level=level, want_rollout_rewards=True)
    per = []
    for r in range(R):
        viol, _, high = ops.pn_reward(x, idx[r])
        per.append(viol.float() if level == "Low" else high)
    per = torch.stack(per)
    assert torch.equal(rews, per)
    want_best, _ = per.min(0)
    assert torch.equal(best, want_best)
    first = (per == want_best[None]).int().argmax(0)           # lowest rollout holding the minimum
    assert torch.equal(rollout.long(), first)
    rows = torch.arange(n, device="cuda")
    assert torch.equal(best_idx, idx[rollout.long(), :, rows].t())
    assert (rollout != 3).all() and (rollout != 5).all()       # a tie never goes to the later copy


@pytest.mark.gpu
@pytest.mark.parametrize("level", ["Low", "High"])
def test_best_of_never_worse_than_greedy_and_one_rollout_is_greedy(level):
    from gnnpn_sc_b200.synth import pn_instances
    n, K, N = 200, 8, 5
    x = pn_instances(n, K, N, seed=9).cuda()
    low, m = _net(K, N, "Low", seed=1), _net(K, N, level, seed=2)
    with torch.no_grad():
        _, _, _, _, latent = low(x, None, sample="greedy", training="SL")
        lat = latent if level == "High" else None             # PNHigh with PNLow's latent
        R_g, _, act_g, idx_g, _ = m(x, None, lat, sample="greedy", training="RL")
    m.actor.generator = torch.Generator(device="cuda").manual_seed(1)
    R1, act1, idx1, roll1 = m.best_of(x, None, lat, rollouts=1)
    assert torch.equal(R1, R_g) and all(torch.equal(a, b) for a, b in zip(idx1, idx_g))
    assert all(torch.equal(a, b) for a, b in zip(act1, act_g)) and (roll1 == 0).all()
    Rb, actb, idxb, rollb = m.best_of(x, None, lat, rollouts=8)
    assert (Rb <= R_g).all()
    # the returned picks are the chosen rollout's, `last` holds that rollout's window outputs, and R is their reward
    R_re = m.reward(actb, None, K, USE_CUDA=True, level=level, embedding_size=0)
    assert torch.equal(R_re, Rb)
    assert torch.equal(m.actor.last["idx"].long(), torch.stack(idxb))
    probs = m.actor.last["win_probs"]
    assert probs.shape == (n, K * N)
    assert torch.allclose(probs.view(n, K, N).sum(2), torch.ones(n, K, device="cuda"), atol=1e-5)


@pytest.mark.gpu
def test_draws_follow_the_decoder_probabilities():
    """Step 0 of every rollout sees the same window distribution; over M = 4095 sampled rollouts of one instance the pick
    frequencies f_j match p_j within 5 standard deviations, |f_j - p_j| <= 5 sqrt(p_j (1 - p_j) / M) + 1 / M (seed
    fixed: the outcome is deterministic; a correct sampler fails this bound with probability < 1e-5 per candidate)."""
    from gnnpn_sc_b200.synth import pn_instances
    K, N, R = 2, 8, 4096
    m = _net(K, N, C=2)                                        # C = 2: a spread distribution
    m.actor.generator = torch.Generator(device="cuda").manual_seed(123)
    x = pn_instances(1, K, N, seed=4, neutral_frac=0.0).cuda()
    idx, _, wp = m.actor.decode_rollouts(x, None, R)
    p = wp[0, 0, :N].double()
    assert torch.equal(wp[:, 0, :N], wp[:1, 0, :N].expand(R, N))
    M = R - 1
    f = torch.bincount(idx[1:, 0, 0].long(), minlength=N).double() / M
    bound = 5 * torch.sqrt(p * (1 - p) / M) + 1.0 / M
    assert p.max() < 0.9, p                                    # the check is not vacuous
    assert ((f - p).abs() <= bound).all(), (f.tolist(), p.tolist())


def _pipe_nets(K, N):
    return _net(K, N, "Low", seed=1), _net(K, N, "High", seed=2)


@pytest.mark.gpu
def test_low_high_rollouts_equal_stage_by_stage():
    from gnnpn_sc_b200.pipeline import low_high
    from gnnpn_sc_b200.synth import pn_instances
    n, K, N, R = 300, 10, 5, 6
    x = pn_instances(n, K, N, seed=2).cuda()
    low, high = _pipe_nets(K, N)
    side = torch.cuda.Stream()
    lat0, R0, idx0 = low_high(low, high, x, side)
    high.actor.generator = torch.Generator(device="cuda").manual_seed(5)
    lat1, R1, idx1 = low_high(low, high, x, side, rollouts=1)
    assert torch.equal(R0, R1) and all(torch.equal(a, b) for a, b in zip(idx0, idx1))      # rollouts=1: today's path
    high.actor.generator = torch.Generator(device="cuda").manual_seed(5)
    _, Rr, idxr = low_high(low, high, x, side, rollouts=R)
    with torch.no_grad():
        _, _, _, _, latent = low(x, None, sample="greedy", training="SL")
    high.actor.generator = torch.Generator(device="cuda").manual_seed(5)
    Rs, _, idxs, _ = high.best_of(x, None, latent, rollouts=R)
    assert torch.equal(Rr, Rs) and all(torch.equal(a, b) for a, b in zip(idxr, idxs))
    assert (Rr <= R0).all()


@pytest.mark.gpu
def test_ml2pn_rollouts_compose_and_seed_eswoa_with_the_best_picks():
    """ML2PN(..., rollouts=R).compose == the stages by hand (candidates -> PNLow greedy -> PNHigh best_of), rollouts=1 ==
    the default pipeline bit for bit, and the ESWOA stage equals the same stage fed the best picks directly."""
    from gnnpn_sc_b200 import synth, loadData, trainML, modelML
    from gnnpn_sc_b200.pipeline import ML2PN, constraint_arrays, woa_arrays
    K, S, N, n, R = 47, 2507, 5, 32, 8
    ds = synth.ml_dataset(n_instances=n, K=K, S=S, seed=11, dist="qws", min_tasks=10)
    samples = trainML.build_samples(loadData.ml_arrays(ds))
    torch.manual_seed(3)
    net = modelML.Net(128, S, 20, 2, 2, isServices=True)
    net.reset_parameters()
    net = net.cuda().eval()
    low, high = _pipe_nets(K, N)
    dev_sample = type(samples[0])(**{k: (v.cuda() if torch.is_tensor(v) else v) for k, v in vars(samples[0]).items()})
    cfg = {"popSize": 20, "MAX_Iter": 10, "reduct": 0}
    rb = trainML.collate_requests(samples, device="cuda")
    cons = [torch.from_numpy(a).cuda() for a in constraint_arrays(ds["nodefeatures"], K)]
    woa = [torch.from_numpy(a).cuda() for a in (*woa_arrays(ds["nodefeatures"], K), np.arange(n, dtype=np.int64))]
    base = ML2PN(net, low, high, dev_sample, ds["serviceFeature"], "cuda", woa=cfg).compose(rb, *cons, woa=woa,
                                                                                         defer_check=True)
    one = ML2PN(net, low, high, dev_sample, ds["serviceFeature"], "cuda", woa=cfg, rollouts=1).compose(
        rb, *cons, woa=woa, defer_check=True)
    for k in ("idx_high", "reward", "objective", "woa_fitness", "woa_services"):
        assert torch.equal(base[k].nan_to_num(nan=-7.0), one[k].nan_to_num(nan=-7.0)), k
    pipe = ML2PN(net, low, high, dev_sample, ds["serviceFeature"], "cuda", woa=cfg, rollouts=R)
    high.actor.generator = torch.Generator(device="cuda").manual_seed(9)
    out = pipe.compose(rb, *cons, woa=woa, defer_check=True)
    rows = out["rows"]
    with torch.no_grad():
        _, _, _, _, latent = low(rows, None, sample="greedy", training="SL")
    high.actor.generator = torch.Generator(device="cuda").manual_seed(9)
    Rs, _, idxs, _ = high.best_of(rows, None, latent, rollouts=R)
    assert torch.equal(out["idx_high"], torch.stack(idxs)) and torch.equal(out["reward"].nan_to_num(nan=-7.0), Rs.nan_to_num(nan=-7.0))
    direct = pipe._woa(rows, torch.stack(idxs), out["picked"].gather(1, torch.stack(idxs).t()), woa, lambda: None)
    for k in ("woa_fitness", "woa_services", "woa_traj", "woa_flags"):
        assert torch.equal(out[k].nan_to_num(nan=-7.0), direct[k].nan_to_num(nan=-7.0)), k


# ----------------------------------------------------------------------------------------------- CPU: refusals
def test_rollout_entry_points_refuse_out_of_scope_arguments():
    from gnnpn_sc_b200 import _lib
    L = _lib.lib()                                  # argument errors come before any CUDA call
    # inputs, enc_out, c_state, latent, alpha, packed, attention, att_params, use_tanh, C, n, L, F, hidden, K, N, dec_h, idx,
    # win_logits, win_probs, sample_uniform, workspace, workspace_bytes, enc_layout
    args = [None, None, None, None, 1.0, None, 0, None, 1, 10.0, 4, 20, 8, 256, 4, 5] + [None] * 6 + [1 << 20, 0]
    assert L.gnnpn_pn_decode_rollouts_f32(*args, 0, None) == -2                   # rollouts < 1
    assert L.gnnpn_pn_decode_rollouts_f32(*args[:13], 128, *args[14:], 2, None) == -2   # hidden != 256
    assert L.gnnpn_pn_decode_rollouts_f32(*args[:12], 9, *args[13:], 2, None) == -2     # more than 8 input columns
    assert L.gnnpn_pn_decode_rollouts_f32(*args, 2, None) == -1                   # NULL pointers, in-scope shape
    assert L.gnnpn_pn_best_rollout_f32(None, None, 4, 20, 8, 4, 0, 1, 0, None, None, None, None, None) == -2
    assert L.gnnpn_pn_best_rollout_f32(None, None, 4, 20, 8, 4, 0, 2, 3, None, None, None, None, None) == -2
    assert L.gnnpn_pn_rollouts_workspace_bytes(100, 256, 0) == 0
    # every rollout has the per-CTA scratch of a batch of n: at least that of n * R rows
    assert L.gnnpn_pn_rollouts_workspace_bytes(130, 256, 16) >= L.gnnpn_pn_workspace_bytes(130 * 16, 256)


@pytest.mark.parametrize("change", ["bahdanau", "glimpse", "embedding", "hidden", "wide", "ffma"])
def test_best_of_refuses_configurations_outside_the_fused_scope(change):
    from gnnpn_sc_b200 import modelPN as M
    K, N = 3, 5
    kw = dict(embedding_size=0, hidden_size=256, n_glimpses=0, attention="Dot", sNumber=N)
    kw.update({"bahdanau": {"attention": "Bahdanau"}, "glimpse": {"n_glimpses": 1}, "embedding": {"embedding_size": 20},
               "hidden": {"hidden_size": 64}, "wide": {"sNumber": 33}, "ffma": {}}[change])
    N = kw["sNumber"]
    m = M.CombinatorialRL(kw["embedding_size"], kw["hidden_size"], K * N, kw["n_glimpses"], 10, 1, M.reward,
                          kw["attention"], N, K, level="High")
    if change == "ffma":
        m.actor.impl = "ffma"
    x = torch.zeros(2, K * N, 9 if change == "embedding" else 8)
    with pytest.raises(NotImplementedError, match="best-of-R"):
        m.best_of(x, None, rollouts=4)
    with pytest.raises(ValueError, match="rollouts"):
        m.actor.decode_rollouts(x, None, 0)
