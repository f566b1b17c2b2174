"""GPU parity of the pointer-network path: CUDA kernels (through the drop-in modules and the C ABI)
against (1) fixtures produced by the real reference and (2) the CPU oracle on the same seeded inputs.

Tolerance (BASELINE.json north_star): selected indices / masks / -inf pattern exact -- any index
mismatch must be explained by a reference top-2 margin below LOGIT_TOL and is counted; fp32 logits and
probabilities within 1e-5 relative (|a-b| <= 1e-5 * max(1, |ref|))."""
import os

import numpy as np
import pytest
import torch

from oracle import make_golden as mg
from oracle import pn_oracle as po

from conftest import record_parity

pytestmark = pytest.mark.gpu
LOGIT_TOL = 1e-5
CUDA_CASES = ["qws_b4", "normal_b2", "small_b16", "sharp_b4", "notanh_b3", "bahdanau_b3", "glimpse_b3", "embed20_b3"]


# "tc": tcgen05 recurrence as dispatched by default -- at these batch sizes the column-split cluster scan
# (tc_colsplit.cu); "tc_pair": the same with option scan=0, i.e. the CTA-pair persistent scan (tc_seq.cu: blocked
# encodings, pointer dots fused into the decoder's cell epilogue) that large batches use; "tc_step": option
# persistent=0, the one-launch-per-step tcgen05 recurrence (tc_kernels.cu); "ffma": the strict-fp32 kernels.
IMPLS = ["tc", "tc_pair", "tc_step", "ffma"]


def _select(impl):
    """Set the scan-kernel options for `impl` (gnnpn_set_option) and return the module-level impl."""
    from gnnpn_sc_b200 import ops
    ops.set_option("scan", 0 if impl == "tc_pair" else -1)
    ops.set_option("persistent", 0 if impl == "tc_step" else 3)
    return "tc" if impl in ("tc_pair", "tc_step") else impl


@pytest.fixture(autouse=True)
def _reset_scan_knob():
    yield
    from gnnpn_sc_b200 import ops
    ops.set_option("scan", -1)
    ops.set_option("scan_groups", 0)
    ops.set_option("persistent", 3)



def _models(name, device="cuda", impl=None):
    from gnnpn_sc_b200 import modelPN as M
    kw, B, (s_lo, s_hi), s_in, gain, dist = mg.CASES[name]
    cfg = mg.case_config(name)
    x = mg.build_inputs(cfg, B, s_in, dist)
    out = []
    for level, seed in (("Low", s_lo), ("High", s_hi)):
        m = M.CombinatorialRL(cfg.embedding_size, cfg.hidden_size, cfg.seq_len, cfg.n_glimpses,
                              cfg.tanh_exploration, int(cfg.use_tanh), M.reward, cfg.attention,
                              cfg.s_number, cfg.s_category, use_cuda=True, level=level)
        m.load_state_dict(po.make_state_dict(cfg, seed, gain), strict=True)
        m.actor.impl = _select(impl)
        out.append(m.to(device).eval())
    return cfg, x, out[0], out[1]


STRESS_FLOOR = {"ffma": 2.0, "tc": 4.0, "tc_pair": 4.0, "tc_step": 4.0, None: 4.0}   # multiples of the reference's own fp32 noise, stress cases only


def _close(a, b, tol=LOGIT_TOL, floor=0.0):
    """|a-b| <= max(tol * max(1,|b|), floor).  `floor` = 4x the reference's own fp32-vs-fp64 deviation, used only
    on stress cases whose weights (LSTM matrices x3) amplify rounding noise beyond 1e-5 for ANY fp32 evaluation
    order -- there the reference's own fp32 run is 1.2e-5..2.3e-5 away from its fp64 run.  The tcgen05 path
    (3xFP16 split with the tensor core's truncating fp32 accumulation, MUFU-based activations) gets 4x, FFMA 2x
    (achieved on a B200: 2.7x and 1.2x, profiles/r02_parity.json)."""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.abs(a - b) <= np.maximum(tol * np.maximum(1.0, np.abs(b)), floor)


def _reference_noise(g, key):
    """max |reference fp32 - reference fp64| on a fixture tensor (0 when the fixture has no fp64 run)."""
    k64 = key + "_f64"
    if k64 not in g.files or not bool(g["picks_equal_in_f64"]):
        return 0.0
    fin = np.isfinite(g[key])
    return float(np.abs(g[key][fin] - g[k64][fin]).max())


def _explain_flips(idx, ref_idx, ref_work_logits, N):
    """Every differing pick must sit on a reference top-2 margin < LOGIT_TOL.  Returns the number of flips."""
    K, B = ref_idx.shape
    flips = 0
    for k, b in zip(*np.nonzero(idx != ref_idx)):
        win = np.sort(ref_work_logits[k, b, k * N:(k + 1) * N])[::-1]
        margin = win[0] - win[1]
        assert margin < LOGIT_TOL * max(1.0, abs(win[0])), f"pick (k={k}, b={b}) differs with margin {margin}"
        flips += 1
    return flips


@pytest.mark.parametrize("impl", IMPLS)
@pytest.mark.parametrize("name", CUDA_CASES)
def test_greedy_low_high_matches_reference_fixture(name, impl, golden_dir):
    g = np.load(os.path.join(golden_dir, f"pn_{name}.npz"))
    cfg, x, low, high = _models(name, impl=impl)
    xc = x.cuda()
    with torch.no_grad():
        _, ap_lo, _, idx_lo, latent = low(xc, None, sample="greedy", training="SL")
        R_hi, ap_hi, act_hi, idx_hi, lg_hi = high(xc, None, latent, sample="greedy", training="RL")
    N = cfg.s_number
    idx_hi_t = idx_hi
    idx_lo = torch.stack(idx_lo).cpu().numpy()
    idx_hi = torch.stack(idx_hi).cpu().numpy()
    flips = _explain_flips(idx_lo, g["idx_low"], g["logits_low"], N)
    assert flips == 0, f"{flips} tolerance-limited picks in PNLow -- downstream comparison undefined for this fixture"
    work_hi = g["logits_high"] + g["logits_low"]
    flips += _explain_flips(idx_hi, g["idx_high"], work_hi, N)
    assert flips == 0
    for mine, key in ((latent, "logits_low"), (lg_hi, "logits_high")):
        ref = g[key]
        dense = torch.stack([mine[k] for k in range(len(mine))]).cpu().numpy()
        assert np.array_equal(np.isneginf(dense), np.isneginf(ref)), "visited-mask (-inf) pattern"
        fin = np.isfinite(ref)
        noise = _reference_noise(g, key)
        err = np.abs(dense[fin] - ref[fin]).max()
        print(f"{name}/{key}[{impl}]: max |dlogit| {err:.2e} (reference's own fp32 noise vs its fp64 run: {noise:.2e})")
        record_parity(f"fixture_{name}_{key}_{impl}", max_abs_dlogit=err, reference_fp32_vs_fp64_noise=noise,
                      max_rel=float((np.abs(dense[fin] - ref[fin]) / np.maximum(1.0, np.abs(ref[fin]))).max()),
                      allowed=("1e-5*max(1,|ref|)" if noise <= LOGIT_TOL / 2 else f"{STRESS_FLOOR[impl]}x reference noise"),
                      pick_flips=flips)
        assert _close(dense[fin], ref[fin], floor=STRESS_FLOOR[impl] * noise if noise > LOGIT_TOL / 2 else 0.0).all(), err
    assert _close(torch.stack(ap_lo).cpu().numpy(), g["action_probs_low"]).all()
    assert _close(torch.stack(ap_hi).cpu().numpy(), g["action_probs_high"]).all()
    assert np.array_equal(torch.stack(act_hi).cpu().numpy(), g["actions_high"])
    assert np.array_equal(R_hi.cpu().numpy(), g["reward_high"])          # bit-exact objective evaluator
    from gnnpn_sc_b200 import ops
    _, obj, _ = ops.pn_reward(xc, torch.stack(idx_hi_t).to(torch.int32), tag=0 if cfg.embedding_size == 0 else 1)
    assert np.array_equal(obj.cpu().numpy(), g["objfunc_high"])          # unrounded objFunc, exact
    r_low = high.reward(act_hi, None, cfg.s_category, USE_CUDA=True, level="Low", embedding_size=cfg.embedding_size)
    assert np.array_equal(r_low.cpu().numpy(), g["viol_high"])


def test_dense_probs_structure(golden_dir):
    g = np.load(os.path.join(golden_dir, "pn_qws_b4.npz"))
    cfg, x, low, high = _models("qws_b4")
    with torch.no_grad():
        _, _, _, _, latent = low(x.cuda(), None, sample="greedy", training="SL")
        probs, *_ = high(x.cuda(), None, latent, sample="greedy", training="SL")
    p1 = probs[1].cpu().numpy()
    assert np.array_equal(p1 == 0, g["probs_high_step1"] == 0)
    assert _close(p1, g["probs_high_step1"]).all()
    assert len(probs) == cfg.s_category


def test_accepts_reference_style_dense_latent_list():
    """A caller holding the reference's K-list of dense [B,L] tensors gets the same picks as the lazy form."""
    cfg, x, low, high = _models("small_b16")
    with torch.no_grad():
        _, _, _, _, latent = low(x.cuda(), None, sample="greedy", training="SL")
        dense = [latent[k].clone() for k in range(len(latent))]
        a = high(x.cuda(), None, latent, sample="greedy", training="SL")[3]
        b = high(x.cuda(), None, dense, sample="greedy", training="SL")[3]
    assert all(torch.equal(u, v) for u, v in zip(a, b))


@pytest.mark.parametrize("impl", IMPLS)
@pytest.mark.parametrize("n,K,N,gain", [(300, 47, 5, 1.0), (129, 50, 10, 1.0), (64, 12, 5, 3.0), (1, 3, 2, 1.0)])
def test_teacher_forced_steps_against_oracle(n, K, N, gain, impl):
    """Per-step comparison with the oracle's picks fed back, so one tolerance-limited pick cannot cascade."""
    from gnnpn_sc_b200 import modelPN as M
    from gnnpn_sc_b200.synth import pn_instances
    cfg = po.PNConfig(seq_len=K * N, s_number=N, s_category=K)
    sd = po.make_state_dict(cfg, 77, gain)
    x = pn_instances(n, K, N, seed=5)
    with torch.no_grad():
        _, idx_ref, lg_ref = po.pointer_forward(sd, cfg, x, None, "greedy")
    m = M.CombinatorialRL(0, 256, K * N, 0, 10, 1, M.reward, "Dot", N, K, level="Low")
    m.load_state_dict(sd)
    m = m.cuda().eval()
    m.actor.impl = _select(impl)
    with torch.no_grad():
        probs, idx, lg = m.actor(x.cuda(), None, sample="greedy", forced_idxs=[t.cuda() for t in idx_ref])
    idx = torch.stack(idx).cpu().numpy()
    ref = torch.stack(idx_ref).numpy()
    ref_lg = torch.stack(lg_ref).numpy()
    flips = _explain_flips(idx, ref, ref_lg, N)
    dense = torch.stack([lg[k] for k in range(K)]).cpu().numpy()
    assert np.array_equal(np.isneginf(dense), np.isneginf(ref_lg))
    fin = np.isfinite(ref_lg)
    err = np.abs(dense[fin] - ref_lg[fin])
    # the oracle's own distance from exact arithmetic: same network in float64, same (forced) picks
    sd64 = {k: v.double() for k, v in sd.items()}
    with torch.no_grad():
        _, _, lg64 = po.pointer_forward(sd64, cfg, x.double(), None, "greedy", forced_idxs=idx_ref)
    noise = float(np.abs(torch.stack(lg64).numpy()[fin] - ref_lg[fin]).max())
    print(f"teacher-forced[{impl}] n={n} K={K} N={N} gain={gain}: {flips} tolerance-limited picks of {K * n}, "
          f"max |dlogit| {err.max():.2e}, oracle fp32-vs-fp64 noise {noise:.2e}")
    assert _close(dense[fin], ref_lg[fin], floor=STRESS_FLOOR[impl] * noise if noise > LOGIT_TOL / 2 else 0.0).all(), err.max()


@pytest.mark.parametrize("impl", IMPLS)
def test_free_running_full_size_properties(impl):
    """QWS shape at a batch the oracle cannot finish quickly: structural properties + reward vs oracle."""
    from gnnpn_sc_b200 import modelPN as M
    from gnnpn_sc_b200.synth import pn_instances
    n, K, N = 4096, 47, 5
    cfg = po.PNConfig(seq_len=K * N, s_number=N, s_category=K)
    x = pn_instances(n, K, N, seed=9).cuda()
    low = M.CombinatorialRL(0, 256, K * N, 0, 10, 1, M.reward, "Dot", N, K, level="Low")
    high = M.CombinatorialRL(0, 256, K * N, 0, 10, 1, M.reward, "Dot", N, K, level="High")
    low.load_state_dict(po.make_state_dict(cfg, 1))
    high.load_state_dict(po.make_state_dict(cfg, 2))
    low, high = low.cuda().eval(), high.cuda().eval()
    low.actor.impl = high.actor.impl = _select(impl)

    def run(xs):
        with torch.no_grad():
            _, _, _, _, lat = low(xs, None, sample="greedy", training="SL")
            R, ap, act, idx, _ = high(xs, None, lat, sample="greedy", training="RL")
        return torch.stack(idx), R, torch.stack(act)

    idx, R, act = run(x)
    idx2, R2, _ = run(x)
    assert torch.equal(idx, idx2) and torch.equal(R, R2)                      # deterministic
    lo = torch.arange(K, device="cuda").view(K, 1) * N
    assert bool(((idx >= lo) & (idx < lo + N)).all())                        # picks stay in their window
    parts = [run(x[s:s + 1000]) for s in range(0, n, 1000)]                  # instance sharding == unsharded
    assert torch.equal(torch.cat([p[0] for p in parts], dim=1), idx)
    assert torch.equal(torch.cat([p[1] for p in parts]), R)
    sub = slice(0, 256)                                                      # reward evaluator vs oracle, exact
    R_ref = po.reward(list(act[:, sub].cpu()), None, K, "High", 0)
    assert torch.equal(R[sub].cpu(), R_ref)


def test_host_buffer_c_abi_matches_module_path():
    import ctypes
    from gnnpn_sc_b200 import modelPN as M, _lib
    from gnnpn_sc_b200.synth import pn_instances
    n, K, N = 200, 47, 5
    cfg = po.PNConfig(seq_len=K * N, s_number=N, s_category=K)
    x = pn_instances(n, K, N, seed=3)
    low = M.CombinatorialRL(0, 256, K * N, 0, 10, 1, M.reward, "Dot", N, K, level="Low")
    high = M.CombinatorialRL(0, 256, K * N, 0, 10, 1, M.reward, "Dot", N, K, level="High")
    low.load_state_dict(po.make_state_dict(cfg, 1))
    high.load_state_dict(po.make_state_dict(cfg, 2))
    low, high = low.cuda().eval(), high.cuda().eval()
    with torch.no_grad():
        _, _, _, il, lat = low(x.cuda(), None, sample="greedy", training="SL")
        R, _, _, ih, _ = high(x.cuda(), None, lat, sample="greedy", training="RL")
    pk_lo = torch.cat(low.actor._packed_weights()).cpu().contiguous()
    pk_hi = torch.cat(high.actor._packed_weights()).cpu().contiguous()
    idx_lo = np.zeros((K, n), np.int32)
    idx_hi = np.zeros((K, n), np.int32)
    rew = np.zeros(n, np.float32)
    xin = x.contiguous().numpy()
    rc = _lib.lib().gnnpn_pn_greedy_low_high_host(
        xin.ctypes.data, n, K * N, 8, 256, K, N, pk_lo.data_ptr(), pk_hi.data_ptr(), 1, 10.0, 1.0,
        idx_lo.ctypes.data, idx_hi.ctypes.data, rew.ctypes.data)
    assert rc == 0
    assert np.array_equal(idx_lo, torch.stack(il).cpu().numpy())
    assert np.array_equal(idx_hi, torch.stack(ih).cpu().numpy())
    assert np.array_equal(rew, R.cpu().numpy())


def test_argument_errors_are_reported_not_thrown():
    from gnnpn_sc_b200 import _lib, modelPN as M
    L = _lib.lib()
    assert L.gnnpn_lstm_encode_f32(None, 1, 1, 8, 256, None, None, None, None, 0, 0, None) == -1    # GNNPN_ENULL
    t = torch.zeros(16, device="cuda")
    assert L.gnnpn_lstm_encode_f32(t.data_ptr(), 1, 1, 8, 128, t.data_ptr(), t.data_ptr(), t.data_ptr(), None, 0, 0, None) == -2
    with pytest.raises(RuntimeError):
        m = M.CombinatorialRL(0, 256, 6, 0, 10, 1, M.reward, "Dot", 2, 3).cuda()
        m(torch.zeros(2, 6, 8), None, sample="greedy", training="SL")                       # CPU tensor -> loud error


def test_host_batch_pipeline_matches_direct_calls():
    """gnnpn_sc_b200.pipeline.GreedyLowHigh (double-buffered uploads) == calling the modules batch by batch."""
    from gnnpn_sc_b200.pipeline import GreedyLowHigh
    from gnnpn_sc_b200.synth import pn_instances
    cfg, _, low, high = _models("qws_b4")
    K, N = cfg.s_category, cfg.s_number
    batches = [pn_instances(n, K, N, seed=90 + i) for i, n in enumerate((130, 64, 200))]     # ragged sizes
    outs = list(GreedyLowHigh(low, high, "cuda").run(batches))
    assert len(outs) == len(batches)
    for x, (idx_host, r_host) in zip(batches, outs):
        with torch.no_grad():
            _, _, _, _, latent = low(x.cuda(), None, sample="greedy", training="SL")
            R, _, _, idx, _ = high(x.cuda(), None, latent, sample="greedy", training="RL")
        assert not idx_host.is_cuda and idx_host.dtype == torch.int32
        assert torch.equal(idx_host.long(), torch.stack(idx).cpu())
        assert torch.equal(r_host, R.cpu())


@pytest.mark.parametrize("impl", ["ffma", "tc_step"])
def test_general_kernels_equal_fused_path_bitwise(impl):
    """Dot / no glimpse / N <= 32 through the general (one-CTA-per-instance) kernels == the fused path, bit for bit
    (same LSTM kernel on both sides: with impl="tc" the fused path runs the persistent scan, whose cell epilogue rounds
    differently from the per-step tcgen05 kernel the general path uses; "tc_step" runs that per-step kernel on both)."""
    from gnnpn_sc_b200.synth import pn_instances
    cfg, _, low, high = _models("qws_b4", impl=impl)
    x = pn_instances(200, cfg.s_category, cfg.s_number, seed=31).cuda()
    outs = []
    for general in (False, True):
        low.actor.force_general = high.actor.force_general = general
        with torch.no_grad():
            _, _, _, idx_lo, latent = low(x, None, sample="greedy", training="SL")
            R, ap, _, idx_hi, lg = high(x, None, latent, sample="greedy", training="RL")
        outs.append((torch.stack(idx_lo), torch.stack(idx_hi), latent.window.clone(), lg.window.clone(),
                     high.actor.last["win_probs"].clone(), R))
    for a, b in zip(*outs):
        assert torch.equal(a, b)


@pytest.mark.parametrize("kw,n", [
    (dict(s_category=5, s_number=40), 37),                                        # window wider than a warp
    (dict(s_category=6, s_number=4, attention="Bahdanau", n_glimpses=1), 33),     # additive attention + glimpse
    (dict(s_category=4, s_number=6, n_glimpses=2), 20),                           # two Dot glimpses
    (dict(s_category=7, s_number=3, embedding_size=20, attention="Bahdanau"), 19),
    (dict(s_category=3, s_number=1000), 6),                                       # scale-up window width (BASELINE config 4)
    (dict(s_category=12, s_number=1000), 20),                                     # 12,000 encoder steps, 12 decode steps of 1000 candidates
])
def test_general_variants_teacher_forced_against_oracle(kw, n):
    from gnnpn_sc_b200 import modelPN as M
    K, N = kw["s_category"], kw["s_number"]
    cfg = po.PNConfig(seq_len=K * N, **kw)
    sd = po.make_state_dict(cfg, 123)
    x = mg.build_inputs(cfg, n, 17, "qws")
    with torch.no_grad():
        pr_ref, idx_ref, lg_ref = po.pointer_forward(sd, cfg, x, None, "greedy")
    m = M.CombinatorialRL(cfg.embedding_size, 256, K * N, cfg.n_glimpses, 10, 1, M.reward, cfg.attention, N, K, level="Low")
    m.load_state_dict(sd, strict=True)
    m = m.cuda().eval()
    for impl in IMPLS:
        m.actor.impl = _select(impl)
        with torch.no_grad():
            probs, idx, lg = m.actor(x.cuda(), None, sample="greedy", forced_idxs=[t.cuda() for t in idx_ref])
        ref_lg = torch.stack(lg_ref).numpy()
        flips = _explain_flips(torch.stack(idx).cpu().numpy(), torch.stack(idx_ref).numpy(), ref_lg, N)
        dense = torch.stack([lg[k] for k in range(K)]).cpu().numpy()
        assert np.array_equal(np.isneginf(dense), np.isneginf(ref_lg))
        fin = np.isfinite(ref_lg)
        err = np.abs(dense[fin] - ref_lg[fin]).max()
        print(f"general {kw} [{impl}]: {flips} tolerance-limited picks, max |dlogit| {err:.2e}")
        assert _close(dense[fin], ref_lg[fin]).all(), err
        pd = torch.stack([probs[k] for k in range(K)]).cpu().numpy()
        assert _close(pd, torch.stack(pr_ref).numpy()).all()


def test_bahdanau_attention_module_against_oracle():
    """Attention.forward(query, ref) for name='Bahdanau' (modelPN.py:93-123): W_ref(ref) and C*tanh(V.tanh(..))."""
    from gnnpn_sc_b200 import modelPN as M
    cfg = po.PNConfig(seq_len=12, s_number=3, s_category=4, attention="Bahdanau")
    sd = po.make_state_dict(cfg, 5)
    att = M.Attention(256, use_tanh=True, C=10, name="Bahdanau")
    att.load_state_dict({k[len("actor.pointer."):]: v for k, v in sd.items() if k.startswith("actor.pointer.")})
    att = att.cuda()
    g = torch.Generator().manual_seed(3)
    q, ref = torch.randn(5, 256, generator=g) * 0.5, torch.randn(5, 12, 256, generator=g) * 0.5
    refp_o, lg_o = po.attention(sd, "pointer", cfg, q, ref, True, 10.0)
    refp, lg = att(q.cuda(), ref.cuda())
    assert refp.shape == refp_o.shape
    assert _close(refp.cpu().numpy(), refp_o.numpy()).all()
    assert _close(lg.cpu().numpy(), lg_o.numpy()).all()


@pytest.mark.parametrize("n,K,N", [(1, 3, 2), (130, 12, 32), (300, 47, 5), (2100, 20, 5), (260, 9, 7), (140, 6, 10), (200, 5, 12)])
def test_column_split_scan_equals_cta_pair_scan_bitwise(n, K, N):
    """The small-batch cluster scan (tc_colsplit.cu) issues the same MMA sequence and the same cell / pointer
    arithmetic as the CTA-pair scan (tc_seq.cu): encodings, decoder states, logits, probabilities and picks are
    bit-identical, so sharding a batch (which changes the kernel the dispatcher picks) cannot change results.
    n = 2100 spans 17 groups: two waves of one-group clusters on a B200 (15 co-resident 8-CTA clusters), or 9 two-group
    clusters with a phantom 18th group."""
    from gnnpn_sc_b200 import modelPN as M
    from gnnpn_sc_b200.synth import pn_instances
    from gnnpn_sc_b200.weights import reference_shaped_state_dict
    x = pn_instances(n, K, N, seed=7).cuda()
    m = M.CombinatorialRL(0, 256, K * N, 0, 10, 1, M.reward, "Dot", N, K, level="High")
    m.load_state_dict(reference_shaped_state_dict(256, 8, 78))
    m = m.cuda().eval()
    lat = [torch.randn(n, K * N, device="cuda") for _ in range(K)]
    outs = {}
    # options (scan, scan_groups): column-split with one / two / three instance groups per cluster (encoder), CTA-pair scan
    from gnnpn_sc_b200 import ops
    for key, (mode, g) in {"cs1": (1, 1), "cs2": (1, 2), "cs3": (1, 3), "pair": (0, 0)}.items():
        ops.set_option("scan", mode)
        ops.set_option("scan_groups", g)
        with torch.no_grad():
            _, idx, _ = m.actor(x, lat, sample="greedy")
        torch.cuda.synchronize()
        last = m.actor.last
        outs[key] = [torch.stack(idx).clone()] + [last[k].clone() for k in ("enc_out", "dec_h", "win_logits", "win_probs")]
        # the pair scan keeps blocked encodings / fused pointer dots for windows of up to 10 candidates
        assert last["enc_layout"] == (ops.ENC_BLOCKED128 if key == "pair" and N <= 10 else ops.ENC_ROWMAJOR)
    for key in ("cs1", "cs2", "cs3"):
        for a, b in zip(outs[key], outs["pair"]):
            assert torch.equal(a, b), key


def _sampled_decode(actor, x, lat, K, N, seed=5):
    """A sample="sample" decode whose uniforms come from a fresh generator, so every kernel draws with the same ones.
    Checks that every pick is the inverse CDF of the kernel's own window probabilities at the uniform PointerNet.forward
    drew (sequential float32 cumulative sum; the last candidate with p > 0 when no candidate qualifies).  Returns
    (picks [K, n], win_logits, win_probs, how many picks differ from the first maximal probability)."""
    actor.generator = torch.Generator(device="cuda").manual_seed(seed)
    with torch.no_grad():
        _, idx, _ = actor(x, lat, sample="sample")
    u = torch.rand(K, x.shape[0], device="cuda", generator=torch.Generator(device="cuda").manual_seed(seed))
    idx = torch.stack(idx).cpu().numpy()
    wl, wp = actor.last["win_logits"].clone(), actor.last["win_probs"].clone()
    p = wp.view(-1, K, N).permute(1, 0, 2).cpu().numpy()                       # [K, n, N]
    hit = u.cpu().numpy()[..., None] < np.cumsum(p, axis=2, dtype=np.float32)
    last_pos = np.where(p > 0, np.arange(N), 0).max(axis=2)
    base = np.arange(K)[:, None] * N
    assert np.array_equal(idx, np.where(hit.any(axis=2), hit.argmax(axis=2), last_pos) + base)
    return idx, wl, wp, int((idx != p.argmax(axis=2) + base).sum())


def _high_net(n, K, N, H=256, seed=3):
    from gnnpn_sc_b200 import modelPN as M
    from gnnpn_sc_b200.synth import pn_instances
    from gnnpn_sc_b200.weights import reference_shaped_state_dict
    x = pn_instances(n, K, N, seed=seed).cuda()
    m = M.CombinatorialRL(0, H, K * N, 0, 10, 1, M.reward, "Dot", N, K, level="High")
    m.load_state_dict(reference_shaped_state_dict(H, 8, 78) if H == 256 else
                      po.make_state_dict(po.PNConfig(hidden_size=H, seq_len=K * N, s_number=N, s_category=K), 11))
    lat = [torch.randn(n, K * N, device="cuda", generator=torch.Generator(device="cuda").manual_seed(seed))] * K
    return m.cuda().eval(), x, lat


@pytest.mark.parametrize("N", [5, 10, 12, 32])
def test_sampled_decode_column_split_equals_cta_pair_bitwise(N):
    """Sampled decodes with a latent draw the same picks and write the same window logits / probabilities on the CTA-pair
    scan (N <= 10: one thread finishes an instance; N > 10: lane segments) and on the column-split scan (one warp per
    instance, one and two groups per cluster), and every draw is the inverse CDF of the window probabilities."""
    from gnnpn_sc_b200 import ops
    K, n = 6, 260
    m, x, lat = _high_net(n, K, N)
    outs = {}
    for key, (mode, g) in {"pair": (0, 0), "cs1": (1, 1), "cs2": (1, 2)}.items():
        ops.set_option("scan", mode)
        ops.set_option("scan_groups", g)
        *outs[key], differ = _sampled_decode(m.actor, x, lat, K, N)
        assert differ > 0, key
        assert m.actor.last["enc_layout"] == (ops.ENC_BLOCKED128 if key == "pair" and N <= 10 else ops.ENC_ROWMAJOR)
    for key in ("cs1", "cs2"):
        assert np.array_equal(outs[key][0], outs["pair"][0]), key
        assert torch.equal(outs[key][1], outs["pair"][1]) and torch.equal(outs[key][2], outs["pair"][2]), key


@pytest.mark.parametrize("impl", ["ffma", "tc_step"])
@pytest.mark.parametrize("N", [5, 12])
def test_sampled_decode_general_kernels_equal_per_step_path_bitwise(impl, N):
    """Sampled decodes on the per-step path (one warp per instance) and through the general kernels (one CTA per
    instance) draw the same picks and write the same window logits / probabilities; every draw is the inverse CDF."""
    K, n = 6, 200
    m, x, lat = _high_net(n, K, N)
    m.actor.impl = _select(impl)
    outs = []
    for general in (False, True):
        m.actor.force_general = general
        *out, differ = _sampled_decode(m.actor, x, lat, K, N)
        assert differ > 0
        outs.append(out)
    assert np.array_equal(outs[0][0], outs[1][0])
    assert torch.equal(outs[0][1], outs[1][1]) and torch.equal(outs[0][2], outs[1][2])


def test_sampled_decode_any_hidden_size_draws_the_inverse_cdf():
    """The any-hidden-size pointer kernel draws the inverse CDF of its own window probabilities."""
    K, N, n = 6, 7, 130
    m, x, lat = _high_net(n, K, N, H=128)
    assert _sampled_decode(m.actor, x, lat, K, N)[3] > 0


@pytest.mark.parametrize("n,K,N,with_latent", [(300, 47, 5, False), (130, 12, 10, True), (5, 3, 32, True)])
def test_attention_windows_entry_equals_the_decode(n, K, N, with_latent):
    """gnnpn_pn_attention_windows_f32 (the decode loop's attention alone, for given decoder states) reproduces the window
    logits / probabilities / picks of the decode those states came from, bit for bit (canonical dot order)."""
    from gnnpn_sc_b200 import modelPN as M, ops
    from gnnpn_sc_b200.synth import pn_instances
    from gnnpn_sc_b200.weights import reference_shaped_state_dict
    x = pn_instances(n, K, N, seed=11).cuda()
    m = M.CombinatorialRL(0, 256, K * N, 0, 10, 1, M.reward, "Dot", N, K, level="High")
    m.load_state_dict(reference_shaped_state_dict(256, 8, 5))
    m = m.cuda().eval()
    lat = [torch.randn(n, K * N, device="cuda") for _ in range(K)] if with_latent else None
    with torch.no_grad():
        _, idx, _ = m.actor(x, lat, sample="greedy")
    last = m.actor.last
    got_idx, wl, wp = ops.pn_attention_windows(last["enc_out"], last["dec_h"], N, latent_win=last["latent_win"],
                                               alpha=float(m.actor.alpha))
    assert torch.equal(wl, last["win_logits"]) and torch.equal(wp, last["win_probs"])
    assert torch.equal(got_idx, last["idx"])


# ----------------------------------------------------------------------------- any hidden size
@pytest.mark.parametrize("H,n,K,N,emb", [(64, 37, 6, 4, 0), (128, 130, 12, 5, 0), (200, 9, 5, 7, 0), (512, 16, 4, 3, 0),
                                         (96, 20, 6, 4, 20)])
def test_any_hidden_size_matches_oracle(H, n, K, N, emb):
    """hidden_size is a free ini parameter (trainPNLow.py:204): sizes other than the shipped 256 run on the strict-fp32
    any-hidden-size kernels (gnnpn_*_anyh_f32).  PNLow -> PNHigh greedy against the oracle: picks exact (a flip must sit on
    a reference margin below the tolerance), window logits / probabilities / encodings / decoder states within 1e-5, the
    -inf pattern of the dense logits exact, reward exact; then a teacher-forced sampled decode."""
    from gnnpn_sc_b200 import modelPN as M
    L = K * N
    cfg = po.PNConfig(hidden_size=H, seq_len=L, s_number=N, s_category=K, embedding_size=emb)
    g = torch.Generator().manual_seed(H + n)
    x = torch.rand(n, L, 8, generator=g)
    if emb:
        x = torch.cat([torch.arange(L).div(N, rounding_mode="floor").float().view(1, L, 1).expand(n, L, 1), x], 2)
    sds = [po.make_state_dict(cfg, 11), po.make_state_dict(cfg, 12)]
    nets = []
    for level, sd in zip(("Low", "High"), sds):
        m = M.CombinatorialRL(emb, H, L, 0, 10, 1, M.reward, "Dot", N, K, level=level)
        m.load_state_dict(sd, strict=True)
        nets.append(m.cuda().eval())
    xc = x.cuda()
    with torch.no_grad():
        _, _, _, idx_lo, lat = nets[0](xc, None, sample="greedy", training="SL")
        R, _, _, idx_hi, lg_hi = nets[1](xc, None, lat, sample="greedy", training="RL")
        p_lo, i_lo, l_lo, int_lo = po.pointer_forward(sds[0], cfg, x, None, "greedy", return_internals=True)
        p_hi, i_hi, l_hi, int_hi = po.pointer_forward(sds[1], cfg, x, l_lo, "greedy", return_internals=True)
    assert torch.equal(torch.stack(idx_lo).cpu(), torch.stack(i_lo)), "PNLow picks"
    assert torch.equal(torch.stack(idx_hi).cpu(), torch.stack(i_hi)), "PNHigh picks"
    worst = {}
    for tag, net, ref_l, ref_p, internals in (("low", nets[0], l_lo, p_lo, int_lo), ("high", nets[1], l_hi, p_hi, int_hi)):
        last = net.actor.last
        dense = torch.stack(ref_l)                                     # [K, n, L]
        win = dense.view(K, n, K, N).diagonal(dim1=0, dim2=2).permute(0, 2, 1).reshape(n, L)
        winp = torch.stack(ref_p).view(K, n, K, N).diagonal(dim1=0, dim2=2).permute(0, 2, 1).reshape(n, L)
        rel = lambda a, b: float(((a - b).abs() / b.abs().clamp(min=1)).max())
        worst[f"logits_{tag}"] = rel(last["win_logits"].cpu(), win)
        worst[f"probs_{tag}"] = rel(last["win_probs"].cpu(), winp)
        worst[f"enc_out_{tag}"] = rel(last["enc_out"].cpu(), internals["enc_out"])
        worst[f"dec_h_{tag}"] = rel(last["dec_h"].cpu(), torch.stack(internals["queries"], 1))
    got_dense = torch.stack([lg_hi[k] for k in range(K)]).cpu()
    ref_dense = torch.stack(l_hi)
    assert torch.equal(torch.isinf(got_dense), torch.isinf(ref_dense)), "-inf pattern of the dense logits"
    fin = torch.isfinite(ref_dense)
    worst["dense_logits_high"] = float(((got_dense[fin] - ref_dense[fin]).abs() / ref_dense[fin].abs().clamp(min=1)).max())
    record_parity(f"any_hidden_size_H{H}_n{n}_K{K}_N{N}_emb{emb}", tolerance=LOGIT_TOL, **worst)
    for k, v in worst.items():
        assert v <= LOGIT_TOL, (k, v)
    rows = torch.arange(n)
    R_ref = po.reward([x[rows, a, :] for a in i_hi], None, K, "High", emb)
    assert torch.equal(R.cpu(), R_ref)
    # sampled decode, teacher-forced on an arbitrary in-window sequence: probabilities of every step against the oracle
    forced = [(k * N + torch.randint(0, N, (n,), generator=g)) for k in range(K)]
    with torch.no_grad():
        probs, _, _ = nets[0].actor(xc, None, sample="sample", forced_idxs=[f.cuda() for f in forced])
        p_ref, _, _ = po.pointer_forward(sds[0], cfg, x, None, "sample", forced_idxs=forced)
    winp = torch.stack(p_ref).view(K, n, K, N).diagonal(dim1=0, dim2=2).permute(0, 2, 1).reshape(n, L)
    assert float((probs.window.cpu() - winp).abs().max()) <= LOGIT_TOL


def test_any_hidden_size_unsupported_variants_raise():
    """Bahdanau / glimpses / windows wider than 32 exist only for hidden_size = 256: a clear error, not garbage."""
    from gnnpn_sc_b200 import modelPN as M
    x = torch.rand(4, 12, 8).cuda()
    for kw in (dict(att="Bahdanau", gl=0), dict(att="Dot", gl=1)):
        m = M.CombinatorialRL(0, 128, 12, kw["gl"], 10, 1, M.reward, kw["att"], 4, 3, level="Low").cuda().eval()
        with pytest.raises(NotImplementedError):
            m(x, None, sample="greedy", training="SL")
