"""The CTA-pair scan (tc_seq.cu) keeps its recurrent operand h in two buffers: step t reads buffer t&1 and writes h'(t)
into the other.  These cases pin that down against the column-split scan (tc_colsplit.cu, one buffer, the same MMA
sequence), bit for bit: encoder lengths and decode lengths of both parities (the last step reads buffer 0 or 1), a pair
whose second CTA is all padding, every decoder row capacity (5 / 8 / 10, and row-major encodings past 10), and a long
encoder."""
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _reset_scan_options():
    yield
    from gnnpn_sc_b200 import ops
    ops.set_option("scan", -1)
    ops.set_option("scan_groups", 0)


# (n, K, N): encoder length L = K * N, K decode steps
CASES = [
    (300, 47, 5),     # L = 235, K odd; 4 CTAs, the last one all padding
    (300, 48, 5),     # L = 240, K even
    (140, 26, 8),     # L = 208, K even, row capacity 8
    (150, 15, 10),    # L = 150, K odd, row capacity 10
    (100, 21, 12),    # row-major encodings, separate pointer phase; L = 252, K odd; the second CTA all padding
    (130, 201, 5),    # long encoder: L = 1005, K = 201
]


@pytest.mark.parametrize("n,K,N", CASES)
def test_pair_scan_h_buffers_equal_column_split_bitwise(n, K, N):
    from gnnpn_sc_b200 import modelPN as M
    from gnnpn_sc_b200 import ops
    from gnnpn_sc_b200.synth import pn_instances
    from gnnpn_sc_b200.weights import reference_shaped_state_dict
    x = pn_instances(n, K, N, seed=11).cuda()
    m = M.CombinatorialRL(0, 256, K * N, 0, 10, 1, M.reward, "Dot", N, K, level="High")
    m.load_state_dict(reference_shaped_state_dict(256, 8, 78))
    m = m.cuda().eval()
    g = torch.Generator(device="cuda").manual_seed(n + K)
    lat = [torch.randn(n, K * N, device="cuda", generator=g) for _ in range(K)]
    outs = {}
    for key, (mode, groups) in {"pair": (0, 0), "cs1": (1, 1)}.items():
        ops.set_option("scan", mode)
        ops.set_option("scan_groups", groups)
        with torch.no_grad():
            _, idx, _ = m.actor(x, lat, sample="greedy")
        torch.cuda.synchronize()
        last = m.actor.last
        outs[key] = [torch.stack(idx).clone()] + [last[k].clone() for k in ("enc_out", "dec_h", "win_logits", "win_probs")]
        assert last["enc_layout"] == (ops.ENC_BLOCKED128 if key == "pair" and N <= 10 else ops.ENC_ROWMAJOR)
    names = ("picks", "enc_out", "dec_h", "win_logits", "win_probs")
    for name, a, b in zip(names, outs["cs1"], outs["pair"]):
        assert torch.equal(a, b), name
