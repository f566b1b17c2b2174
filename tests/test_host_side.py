"""CPU-only checks of the host side: the C-ABI library loads and exports every symbol the header
declares, product-side helpers agree with the oracle's, synthetic data has the reference's layout."""
import os
import re

import numpy as np
import torch

from oracle import pn_oracle as po

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from gnnpn_sc_b200 import _lib
    with open(os.path.join(ROOT, "include", "gnnpn_b200.h")) as f:
        declared = set(re.findall(r"GNNPN_API\s+[\w\s\*]+?\b(gnnpn_\w+)\s*\(", f.read()))
    assert declared, "header parse failed"
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    L = _lib.lib()                      # CDLL + getattr of every symbol; no compute without a GPU
    with open(os.path.join(ROOT, "include", "gnnpn_b200.h")) as f:
        version = int(re.search(r"#define GNNPN_ABI_VERSION (\d+)", f.read()).group(1))
    assert L.gnnpn_abi_version() == version
    assert L.gnnpn_error_string(-2) == b"unsupported shape"
    assert L.gnnpn_pn_packed_lstm_floats(256, 8) == (256 + 32 + 2) * 1024 + 1024 * 320   # FFMA block, bias, start, fp16 hi/lo (halfs)
    # argument errors are detected before any CUDA call, so they are testable on a CPU box
    assert L.gnnpn_lstm_encode_f32(None, 1, 1, 8, 256, None, None, None, None, 0, 0, None) == -1


def test_product_weights_equal_oracle_weights():
    from gnnpn_sc_b200.weights import reference_shaped_state_dict
    cfg = po.PNConfig()
    a, b = reference_shaped_state_dict(256, 8, 5, 3.0), po.make_state_dict(cfg, 5, 3.0)
    assert a.keys() == b.keys()
    assert all(torch.equal(a[k], b[k]) for k in a)


def test_state_dict_keys_match_reference_layout():
    from gnnpn_sc_b200 import modelPN as M
    m = M.CombinatorialRL(0, 256, 235, 0, 10, 1, M.reward, "Dot", 5, 47)
    assert set(m.state_dict()) == set(po.make_state_dict(po.PNConfig(), 0))
    mb = M.CombinatorialRL(20, 256, 18, 1, 10, 1, M.reward, "Bahdanau", 3, 6)
    cfgb = po.PNConfig(seq_len=18, s_number=3, s_category=6, embedding_size=20, attention="Bahdanau")
    ref = po.make_state_dict(cfgb, 0)
    assert set(mb.state_dict()) == set(ref)
    assert all(mb.state_dict()[k].shape == ref[k].shape for k in ref)


def test_no_cpu_fallback():
    import pytest
    from gnnpn_sc_b200 import modelPN as M
    m = M.CombinatorialRL(0, 256, 6, 0, 10, 1, M.reward, "Dot", 2, 3)
    with pytest.raises(RuntimeError):
        m(torch.zeros(2, 6, 8), None, sample="greedy", training="SL")


def test_pn_instances_layout():
    from gnnpn_sc_b200.synth import pn_instances
    x = pn_instances(32, 47, 5, seed=1).view(32, 47, 5, 8).numpy()
    assert (x[:, 1:, :, 4:] == 0).all()                       # global bounds only on category-0 rows
    assert (x[:, 0, :, 5] == 1).all() and (x[:, 0, :, 4] > 0).all()
    neutral = (x[..., :4] == np.array([0, 1, 1, 1], np.float32)).all(-1)
    assert neutral.all(-1).sum() == neutral.any(-1).sum()     # neutral categories are neutral on all N rows
    assert 0.05 < neutral.mean() < 0.4
    assert torch.equal(pn_instances(8, 6, 3, seed=4), pn_instances(8, 6, 3, seed=4))


def test_window_compaction_of_dense_latent():
    from gnnpn_sc_b200.modelPN import _window_of
    K, N, B = 5, 3, 4
    dense = [torch.randn(B, K * N) for _ in range(K)]
    w = _window_of(dense, K, N)
    for k in range(K):
        assert torch.equal(w[:, k * N:(k + 1) * N], dense[k][:, k * N:(k + 1) * N])


def test_constraint_and_service_arrays_follow_loaddatapn():
    """pipeline.constraint_arrays / service_arrays (inputs of the device candidate selection) against the rows the
    numpy restatement of loadDataPN builds from the same JSON objects."""
    import numpy as np
    from gnnpn_sc_b200 import synth, loadData
    from gnnpn_sc_b200.pipeline import constraint_arrays, service_arrays
    K, S, N = 7, 90, 3
    ds = synth.ml_dataset(n_instances=5, K=K, S=S, seed=1, min_tasks=3)
    local, used, glob = constraint_arrays(ds["nodefeatures"], K)
    qos, ptr = service_arrays(ds["serviceFeature"])
    assert qos.shape == (S, 4) and ptr[0] == 0 and ptr[-1] == S and len(ptr) == K + 1
    sf = ds["serviceFeature"]
    ser2cat = np.concatenate([[int(k) - 1] * len(sf[k]) for k in sf.keys()])
    ser2pos = np.concatenate([np.arange(len(sf[k])) for k in sf.keys()])
    for b, nf in enumerate(ds["nodefeatures"]):
        rows = np.asarray(loadData.pn_rows_from_ranking(nf, list(range(S)), sf, ser2cat, ser2pos, N, rng=False))
        rows = rows.reshape(K, N, 9)
        assert np.allclose(rows[0, :, 5:], glob[b])                          # category 0 carries the global bounds
        assert (rows[1:, :, 5:] == 0).all()
        neutral = (rows[:, 0, 1:5] == [0, 1, 1, 1]).all(axis=1)
        assert (~neutral <= used[b].astype(bool)).all()                       # a non-neutral category is a used one
        for c in range(K):
            if not neutral[c]:
                lo2, hi2, lo3, hi3 = local[b, c]
                assert (lo2 <= rows[c, :, 3]).all() and (rows[c, :, 3] <= hi2).all()
                assert (lo3 <= rows[c, :, 4]).all() and (rows[c, :, 4] <= hi3).all()


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the one leg that runs on host cores) prints one JSON line with the driver's keys."""
    import json, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=300, cwd=root)
    assert out.returncode == 0, out.stderr[-400:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    installed = os.path.exists(os.path.join(root, "baseline", "_ref", "src", "models", "modelPN.py"))
    assert line["impl"] == "reference" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == ("reference" if installed else "port")
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["config"]["workload"] == "qws_greedy_pnlow_pnhigh_decode"


def test_anyh_fold_reproduces_the_lstm_preactivations():
    """Host-side folding for the any-hidden-size kernels (ops.anyh_fold): [h | x_raw] . w_cat^T + bias equals
    W_ih . (W_emb x_raw + b_emb) + b_ih + W_hh h + b_hh, and bias0 carries the decoder's start token (modelPN.py:155-163,
    190-191, 205).  Pure torch: runs on the CPU."""
    import torch
    from gnnpn_sc_b200 import ops
    g = torch.Generator().manual_seed(0)
    H, F, n = 48, 8, 5
    w_ih, w_hh = torch.randn(4 * H, H, generator=g), torch.randn(4 * H, H, generator=g)
    b_ih, b_hh = torch.randn(4 * H, generator=g), torch.randn(4 * H, generator=g)
    w_emb, b_emb, start = torch.randn(H, F, generator=g), torch.randn(H, generator=g), torch.randn(H, generator=g)
    w_cat, bias, bias0 = ops.anyh_fold(w_ih, w_hh, b_ih, b_hh, w_emb, b_emb, start)
    assert w_cat.shape == (4 * H, H + F) and bias.shape == (4 * H,) and bias0.shape == (4 * H,)
    h, x = torch.randn(n, H, generator=g).double(), torch.rand(n, F, generator=g).double()
    emb = x @ w_emb.double().T + b_emb.double()
    want = emb @ w_ih.double().T + b_ih.double() + h @ w_hh.double().T + b_hh.double()
    got = torch.cat([h, x], 1) @ w_cat.double().T + bias.double()
    assert float((got - want).abs().max()) < 1e-4 * float(want.abs().max())
    want0 = start.double() @ w_ih.double().T + b_ih.double() + h @ w_hh.double().T + b_hh.double()
    got0 = torch.cat([h, torch.zeros_like(x)], 1) @ w_cat.double().T + bias0.double()
    assert float((got0 - want0).abs().max()) < 1e-4 * float(want0.abs().max())
    assert ops.anyh_fold(w_ih, w_hh, b_ih, b_hh, w_emb, b_emb)[2] is None          # an encoder has no start token


def test_long_row_threshold_policy():
    """The aggregation's automatic long-row threshold, read through the library's workspace query: no split below 2^22
    edges, 256 where a lane group is narrower than a warp (F <= 64), 2048 above.  Argument errors are refused before any
    CUDA call."""
    from gnnpn_sc_b200 import _lib
    L = _lib.lib()
    ws = L.gnnpn_spmm_csr_workspace_bytes
    for F in (32, 64, 128, 256):
        assert ws(2**22 - 1, F, -1) == 0
        assert ws(2**22, F, -1) == ws(2**22, F, 256 if F <= 64 else 2048) > 0
        assert ws(2**22, F, 0) == ws(100, F, 0) == 0
    assert ws(2**22, 64, 256) != ws(2**22, 64, 2048)
    assert ws(2**22, 64, 31) == 0
    p = 1 << 12                                            # any 256-byte aligned address: nothing is dereferenced
    need = ws(2**22, 64, 256)
    call = lambda T, wsb: L.gnnpn_spmm_csr_f32(p, p, p, p, 64, p, 64, 1000, 2**22, 64, 0.0, 0, None, None, None, 0, T, p,
                                               wsb, None)
    before = _lib.launch_count()
    for T in (1, 31):
        assert call(T, need) == -2                         # GNNPN_ESHAPE
    assert call(256, need - 1) == -4                       # GNNPN_EWORKSPACE
    assert call(-1, need - 1) == -4                        # the automatic choice splits here too
    assert _lib.launch_count() == before
