"""GPU parity of the ML-stage kernels (CSR build, gcn_norm, CSR segment-reduce aggregation, node
transform) against the restated PyG-1.7.0 oracle (oracle/ml_oracle.py -- parity unpinned by reference
tests, see its header).  Integer outputs bit-exact; aggregation bit-exact (same sequential order,
mul_rn/add_rn); dense transforms within 1e-5 relative."""
import numpy as np
import pytest
import torch

from oracle import ml_oracle as mo

from conftest import record_parity

pytestmark = pytest.mark.gpu


def _graph(n, e, seed, hub=True, loops=True, dup=True):
    g = torch.Generator().manual_seed(seed)
    src = torch.randint(0, n, (e,), generator=g)
    dst = torch.randint(0, n, (e,), generator=g)
    if hub and e > 8:
        dst[: e // 4] = 3 % n                     # a hub destination
    if dup and e > 4:
        src[-2], dst[-2] = src[0], dst[0]         # duplicate edge
    if loops and e > 6:
        dst[5] = src[5]                           # existing self loop (keeps its weight under gcn_norm)
    if n > 4:
        keep = dst != (n - 2)                     # an empty row
        src, dst = src[keep], dst[keep]
    w = torch.rand(src.numel(), generator=g) + 0.1
    return torch.stack([src, dst]), w


def _ref_csr(ei, w, n):
    order = np.argsort(ei[1].numpy(), kind="stable")
    rowptr = np.zeros(n + 1, np.int64)
    np.add.at(rowptr, ei[1].numpy() + 1, 1)
    return np.cumsum(rowptr), ei[0].numpy()[order].astype(np.int32), None if w is None else w.numpy()[order]


@pytest.mark.parametrize("n,e", [(1, 0), (7, 0), (50, 400), (2507, 60000), (300, 5)])
def test_csr_plain_bit_exact(n, e):
    from gnnpn_sc_b200 import ops
    ei, w = _graph(n, e, seed=n + e) if e else (torch.zeros(2, 0, dtype=torch.long), torch.zeros(0))
    rp, col, val = ops.csr_build(ei.cuda(), w.cuda(), n, ops.CSR_PLAIN)
    r_rp, r_col, r_val = _ref_csr(ei, w, n)
    assert np.array_equal(rp.cpu().numpy(), r_rp)
    assert np.array_equal(col.cpu().numpy(), r_col)
    assert np.array_equal(val.cpu().numpy(), r_val)


@pytest.mark.parametrize("n,e,weighted", [(50, 400, True), (2507, 60000, True), (64, 300, False), (9, 0, True)])
def test_csr_gcn_norm(n, e, weighted):
    from gnnpn_sc_b200 import ops
    ei, w = _graph(n, e, seed=3 * n + e) if e else (torch.zeros(2, 0, dtype=torch.long), torch.zeros(0))
    if not weighted:
        w = None
    ei2, norm = mo.gcn_norm(ei, w, n)
    r_rp, r_col, r_val = _ref_csr(ei2, norm, n)
    rp, col, val = ops.csr_build(ei.cuda(), None if w is None else w.cuda(), n, ops.CSR_GCN_NORM)
    assert np.array_equal(rp.cpu().numpy(), r_rp)
    assert np.array_equal(col.cpu().numpy(), r_col)
    v = val.cpu().numpy()
    ulp = np.abs(v - r_val) / np.spacing(np.abs(r_val).astype(np.float32))
    assert ulp.max(initial=0) <= 1.0, f"gcn_norm differs by {ulp.max()} ulp"
    print(f"gcn_norm n={n} e={e}: max {ulp.max(initial=0):.1f} ulp, exact={np.array_equal(v, r_val)}")


@pytest.mark.parametrize("F", [24, 28, 32, 64, 128, 256, 512])
@pytest.mark.parametrize("weighted", [True, False])
def test_aggregation_bit_exact(F, weighted):
    from gnnpn_sc_b200 import ops
    n, e = 700, 9000
    ei, w = _graph(n, e, seed=F)
    x = torch.randn(n, F)
    ref = mo.aggregate_sum(x, ei, w if weighted else None)
    rp, col, val = ops.csr_build(ei.cuda(), w.cuda() if weighted else None, n, ops.CSR_PLAIN)
    y = ops.spmm_csr(rp, col, val, x.cuda())
    assert torch.equal(y.cpu(), ref), f"max err {(y.cpu() - ref).abs().max()}"


def test_gin_self_term_and_segment_mean():
    from gnnpn_sc_b200 import ops
    n, e, F = 90, 400, 28
    ei, _ = _graph(n, e, seed=1)
    x = torch.randn(n, F)
    eps = torch.tensor(0.25)
    ref = mo.aggregate_sum(x, ei) + (1 + eps) * x
    rp, col, _ = ops.csr_build(ei.cuda(), None, n, ops.CSR_PLAIN)
    y = ops.spmm_csr(rp, col, None, x.cuda(), self_scale=float(1 + eps))
    assert torch.equal(y.cpu(), ref)
    # scatter(reduce='mean') as a CSR over (row -> segment) memberships
    seg = torch.sort(torch.randint(0, 7, (n,))).values
    seg[seg == 4] = 5                                     # an empty segment
    ref_m = mo.segment_mean(x, seg, 7)
    memb = torch.stack([torch.arange(n), seg]).cuda()
    rp, col, _ = ops.csr_build(memb, None, 7, ops.CSR_PLAIN)
    ym = ops.spmm_csr(rp, col, None, x.cuda(), n_rows=7, mean=True)
    assert torch.equal(ym.cpu(), ref_m)


def test_gcn_layer_epilogue():
    from gnnpn_sc_b200 import ops
    n, e, Fin, Fout = 300, 4000, 24, 256
    ei, w = _graph(n, e, seed=11)
    x = torch.randn(n, Fin)
    conv = mo.GCNConvO(Fin, Fout)
    conv.bias.data.normal_()
    bn = torch.nn.BatchNorm1d(Fout).eval()
    bn.running_mean.normal_(); bn.running_var.uniform_(0.5, 2); bn.weight.data.normal_(); bn.bias.data.normal_()
    with torch.no_grad():
        ref = torch.relu(bn(conv(x, ei, w)))
        scale = bn.weight / torch.sqrt(bn.running_var + bn.eps)
        shift = bn.bias - bn.running_mean * scale
    rp, col, val = ops.csr_build(ei.cuda(), w.cuda(), n, ops.CSR_GCN_NORM)
    xw = ops.gemm_bias_act(x.cuda(), conv.weight.data.t().contiguous().cuda())
    y = ops.spmm_csr(rp, col, val, xw, bias=conv.bias.data.cuda(), scale=scale.cuda(), shift=shift.cuda(), act="relu")
    err = (y.cpu() - ref).abs() / ref.abs().clamp(min=1)
    assert err.max() <= 1e-5, err.max()


@pytest.mark.parametrize("impl", ["tc", "ffma"])
@pytest.mark.parametrize("M,N,K", [(1, 128, 128), (97, 256, 28), (5014, 256, 24), (1000, 128, 256), (130, 2507, 128),
                                   (5014, 256, 256), (200000, 256, 256), (257, 48, 4), (300, 16, 60),
                                   (70000, 128, 136), (40000, 240, 252),
                                   (1024, 272, 30080), (300, 48, 9004), (640, 272, 2100)])     # long K, few row tiles: split-K
def test_node_transform_gemm(M, N, K, impl):
    """tcgen05 (persistent 3xFP16-split kernel for K, N <= 256; 3xTF32 mainloop otherwise) and FFMA node transforms
    against an fp64 evaluation on the CPU, ELEMENT-WISE: |y - ref| <= 1e-5 * max(1, |ref|) for every entry."""
    from gnnpn_sc_b200 import ops
    g = torch.Generator().manual_seed(M + N + K)
    a, w, b = torch.randn(M, K, generator=g), torch.randn(N, K, generator=g) / K ** 0.5, torch.randn(N, generator=g)
    scale, shift = torch.rand(N, generator=g) + 0.5, torch.randn(N, generator=g)
    ref = torch.relu(torch.nn.functional.linear(a.double(), w.double(), b.double()) * scale.double() + shift.double())
    y = ops.gemm_bias_act(a.cuda(), w.cuda(), bias=b.cuda(), scale=scale.cuda(), shift=shift.cuda(), act="relu", impl=impl)
    err = ((y.cpu().double() - ref).abs() / ref.abs().clamp(min=1)).max().item()
    # strict-fp32 FFMA accumulates the K terms sequentially in fp32: beyond K ~ 1,700 its own rounding (~ sqrt(K) * 2^-24 per
    # unit of summed magnitude, any fp32 GEMM has it) passes 1e-5, so that path is held to 4 * sqrt(K) * 2^-24 there.  The
    # tensor-core path (split-K chains of 8 k blocks, fp32 adds in split order) is held to 1e-5 at every K.
    tol = 1e-5 if impl == "tc" else max(1e-5, 4.0 * K ** 0.5 * 2.0 ** -24)
    print(f"gemm[{impl}] M={M} N={N} K={K}: max element-wise |err| / max(1,|ref|) {err:.2e} (bound {tol:.1e})")
    record_parity(f"gemm_{impl}_M{M}_N{N}_K{K}", max_elementwise_rel=err, tolerance=tol)
    assert err <= tol, err


def test_gemm_padded_rows_equal_dense_rows():
    """``pad_ld=True`` (rows padded to 8 floats so the tensor-core epilogue stores whole sectors: the ML stage's
    [B, 2507] readout) returns a strided view with exactly the values of the dense result."""
    from gnnpn_sc_b200 import ops
    g = torch.Generator().manual_seed(3)
    for M, N, K in ((5000, 2507, 128), (700, 331, 300)):
        a, w, b = torch.randn(M, K, generator=g).cuda(), (torch.randn(N, K, generator=g) / K ** 0.5).cuda(), torch.randn(N, generator=g).cuda()
        dense = ops.gemm_bias_act(a, w, bias=b, act="sigmoid", impl="tc")
        padded = ops.gemm_bias_act(a, w, bias=b, act="sigmoid", impl="tc", pad_ld=True)
        assert padded.shape == dense.shape and padded.stride(0) % 8 == 0 and padded.stride(0) >= N
        assert torch.equal(padded, dense)
        ref = torch.sigmoid(torch.nn.functional.linear(a.double(), w.double(), b.double()))
        assert float((dense.double() - ref).abs().max()) <= 1e-5


@pytest.mark.parametrize("mag", [1.0e4, 1.0e6])
def test_node_transform_out_of_range_inputs_fall_back(mag):
    """|a| * 2^4 >= 65504 overflows the fp16 split: the converters raise the workspace flag and the guarded strict-fp32
    pass recomputes C on the device -- finite, correct results (fp64 reference, 1e-5 element-wise), rc == 0."""
    from gnnpn_sc_b200 import ops
    g = torch.Generator().manual_seed(11)
    M, N, K = 3000, 256, 256
    a = torch.randn(M, K, generator=g)
    a[::17, ::5] *= mag                                      # un-normalised features (e.g. a response time in ms)
    w, b = torch.randn(N, K, generator=g) / K ** 0.5, torch.randn(N, generator=g)
    ref = torch.nn.functional.linear(a.double(), w.double(), b.double())
    y = ops.gemm_bias_act(a.cuda(), w.cuda(), bias=b.cuda(), impl="tc").cpu().double()
    assert torch.isfinite(y).all()
    # entries where 1e4..1e6-sized terms cancel are held to the magnitude of what was summed (sum_k |a_k w_k| + |b|),
    # the bound any fp32 evaluation order obeys -- not to the cancelled result
    mag_rows = (a.double().abs() @ w.double().abs().T + b.double().abs()).clamp(min=1)
    err = ((y - ref).abs() / mag_rows).max().item()
    record_parity(f"gemm_tc_out_of_range_mag{mag:g}", max_err_over_summed_magnitude=err, tolerance=1e-5)
    assert err <= 1e-5, err
    a[5, 7] = float("inf")                                   # non-finite input: same route, torch's own result
    y = ops.gemm_bias_act(a.cuda(), w.cuda(), bias=b.cuda(), impl="tc").cpu()
    ref32 = torch.nn.functional.linear(a, w, b)
    assert torch.equal(torch.isfinite(y), torch.isfinite(ref32))


@pytest.mark.parametrize("mag", [1e-3, 1.0, 300.0])
def test_node_transform_input_range(mag):
    """The fp16-split node transform keeps fp32-level accuracy over the input magnitudes the ML stage produces
    (raw QoS features ~1e-3..1, post-aggregation sums up to a few hundred); checked against fp64."""
    from gnnpn_sc_b200 import ops
    g = torch.Generator().manual_seed(5)
    M, N, K = 4096, 256, 256
    a = torch.randn(M, K, generator=g) * mag
    a[:, ::7] *= 1e-3                                        # mixed magnitudes inside a row
    w = torch.randn(N, K, generator=g) / K ** 0.5
    ref = (a.double() @ w.double().T)
    y = ops.gemm_bias_act(a.cuda(), w.cuda(), impl="tc").cpu().double()
    err = (y - ref).abs().max() / ref.abs().max()
    ref32 = (torch.nn.functional.linear(a, w).double() - ref).abs().max() / ref.abs().max()
    print(f"gemm range mag={mag}: max err / max|ref| {err:.2e} (torch fp32 CPU: {ref32:.2e})")
    assert err <= 2e-6, err


def test_node_transform_strided_output():
    """C with a leading dimension that is not a multiple of 8 floats takes the narrower store paths."""
    from gnnpn_sc_b200 import ops
    g = torch.Generator().manual_seed(9)
    M, N, K = 1500, 64, 128
    a, w = torch.randn(M, K, generator=g), torch.randn(N, K, generator=g) / K ** 0.5
    ref = torch.nn.functional.linear(a, w)
    for ld in (N + 4, N + 1):
        buf = torch.full((M, ld), 7.0, device="cuda")
        out = buf[:, :N]
        ops.gemm_bias_act(a.cuda(), w.cuda(), out=out, impl="tc")
        assert (out.cpu() - ref).abs().max() <= 1e-5 * ref.abs().max()
        assert torch.all(buf[:, N:] == 7.0)


def test_node_transform_shape_with_misaligned_a_runs_ffma():
    """A node-transform shape whose A is not 16-byte aligned (a contiguous view at a one-float storage offset) runs the
    strict-fp32 FFMA kernel inside the workspace that gnnpn_gemm_workspace_bytes sized: the same bits as impl="ffma"."""
    from gnnpn_sc_b200 import ops
    g = torch.Generator().manual_seed(13)
    M, N, K = 5014, 256, 24
    a = torch.randn(M * K + 1, generator=g).cuda()[1:].view(M, K)
    w, b = torch.randn(N, K, generator=g).cuda() / K ** 0.5, torch.randn(N, generator=g).cuda()
    scale, shift = torch.rand(N, generator=g).cuda() + 0.5, torch.randn(N, generator=g).cuda()
    assert a.is_contiguous() and a.data_ptr() % 16 != 0
    y = ops.gemm_bias_act(a, w, bias=b, scale=scale, shift=shift, act="relu", impl="tc")
    ref = ops.gemm_bias_act(a.clone(), w, bias=b, scale=scale, shift=shift, act="relu", impl="ffma")
    assert torch.equal(y, ref)


# ---------------------------------------------------------------------------------------------------------------------
# hand-derived known-answer tests (tests/ml_kats.py) through the CUDA kernels
# ---------------------------------------------------------------------------------------------------------------------
def test_kat_gcn_norm_csr_and_layer_on_device():
    import ml_kats as kat
    from gnnpn_sc_b200 import ops
    ei = torch.tensor([[s for s, _, _ in kat.GCN_EDGES], [d for _, d, _ in kat.GCN_EDGES]]).cuda()
    w = torch.tensor([x for _, _, x in kat.GCN_EDGES]).cuda()
    rp, col, val = ops.csr_build(ei, w, kat.GCN_N, ops.CSR_GCN_NORM)
    assert rp.tolist() == kat.GCN_CSR_ROWPTR and col.tolist() == kat.GCN_CSR_COL
    want = []
    for r in range(kat.GCN_N):
        for c in kat.GCN_CSR_COL[kat.GCN_CSR_ROWPTR[r]:kat.GCN_CSR_ROWPTR[r + 1]]:
            want.append(float(kat.GCN_NORM[(c, r)]))
    got = val.tolist()
    assert all(abs(g - v) <= 2e-7 * max(1.0, abs(v)) for g, v in zip(got, want)), (got, want)
    assert got[-1] == 0.0                                                  # zero degree: inf -> 0
    x = torch.zeros(kat.GCN_N, 4)
    x[:, :2] = torch.tensor(kat.GCN_X)                                     # feature dim padded to a multiple of 4
    bias = torch.tensor(kat.GCN_BIAS + [0.0, 0.0])
    y = ops.spmm_csr(rp, col, val, x.cuda(), bias=bias.cuda()).cpu()
    for i in range(kat.GCN_N):
        for c in range(2):
            v = float(kat.GCN_OUT[i][c])
            assert abs(y[i, c].item() - v) <= 3e-7 * max(1.0, abs(v)), (i, c, y[i, c].item(), v)
    record_parity("kat_gcn_norm_layer", max_rel=max(abs(y[i, c].item() - float(kat.GCN_OUT[i][c])) / max(1.0, abs(float(kat.GCN_OUT[i][c])))
                                                    for i in range(kat.GCN_N) for c in range(2)), tolerance=3e-7)


def test_kat_gin_and_segment_mean_on_device():
    import ml_kats as kat
    from gnnpn_sc_b200 import ops
    ei = torch.tensor([[s for s, _ in kat.GIN_EDGES], [d for _, d in kat.GIN_EDGES]]).cuda()
    rp, col, _ = ops.csr_build(ei, None, 3, ops.CSR_PLAIN)
    x = torch.zeros(3, 4)
    x[:, 0] = torch.tensor(kat.GIN_X)
    pre = ops.spmm_csr(rp, col, None, x.cuda(), self_scale=1.0 + kat.GIN_EPS).cpu()[:, 0]
    assert pre.tolist() == [float(v) for v in kat.GIN_PRE]                 # exact
    seg = torch.tensor(kat.MEAN_SEG).cuda()
    idx = torch.stack([torch.arange(len(kat.MEAN_SEG), device="cuda"), seg])
    rp, col, _ = ops.csr_build(idx, None, kat.MEAN_SEGMENTS, ops.CSR_PLAIN)
    xm = torch.zeros(len(kat.MEAN_X), 4)
    xm[:, 0] = torch.tensor(kat.MEAN_X)
    out = ops.spmm_csr(rp, col, None, xm.cuda(), n_rows=kat.MEAN_SEGMENTS, mean=True).cpu()[:, 0]
    assert out.tolist() == kat.MEAN_OUT                                    # empty segments -> 0, not NaN


def test_hub_row_with_adaptive_chunk_length():
    """A hub row of more than 256 * 4096 edges gets longer chunks (at most ~4096 chunk sums per row, so the in-order combine
    is not a serial tail): same result as the strictly sequential sum to re-association, deterministic, other rows exact."""
    from gnnpn_sc_b200 import ops
    g = torch.Generator().manual_seed(9)
    n, F, T = 500, 8, 256
    deg = torch.randint(0, 20, (n,), generator=g)
    deg[3], deg[400] = 1_300_000, 70_000                                   # 1.3M edges -> chunks of 320 edges; 70k -> 256
    dst = torch.repeat_interleave(torch.arange(n), deg)
    src = torch.randint(0, n, (dst.numel(),), generator=g)
    w = torch.rand(dst.numel(), generator=g) + 0.05
    x = torch.randn(n, F, generator=g)
    rp, col, val = ops.csr_build(torch.stack([src, dst]).cuda(), w.cuda(), n, ops.CSR_PLAIN)
    y = ops.spmm_csr(rp, col, val, x.cuda(), long_row_threshold=T).cpu()
    assert torch.equal(y, ops.spmm_csr(rp, col, val, x.cuda(), long_row_threshold=T).cpu())
    terms = w.double().view(-1, 1) * x.double()[src]
    ref64 = torch.zeros(n, F, dtype=torch.float64).index_add_(0, dst, terms)
    mag = torch.zeros(n, F, dtype=torch.float64).index_add_(0, dst, terms.abs()).clamp(min=1)
    err = ((y.double() - ref64).abs() / mag).max().item()
    record_parity("spmm_hub_row_adaptive_chunks", max_err_over_summed_magnitude=err, tolerance=1e-5, max_in_degree=1_300_000)
    assert err <= 1e-5, err
    short = deg <= T
    y0 = ops.spmm_csr(rp, col, val, x.cuda(), long_row_threshold=0).cpu()  # unsplit: strictly sequential
    assert torch.equal(y[short], y0[short])


def test_long_row_split_hub_destinations():
    """Skewed in-degrees (hub rows): rows at or below the threshold are bit-identical to the index_add_ order oracle, split
    rows agree to 1e-5 (re-association of chunk sums only), the result is deterministic, and the fused epilogue (mean,
    bias, ReLU) is applied once per row."""
    from gnnpn_sc_b200 import ops
    g = torch.Generator().manual_seed(5)
    n, F, T = 3000, 64, 256                                               # rows > 256 edges split into chunks of 256
    deg = torch.randint(0, 40, (n,), generator=g)
    deg[7], deg[1500], deg[2999] = 120000, 5000, 257                       # hubs; 257 = just above the threshold
    deg[11] = 256                                                          # exactly at the threshold: not split
    dst = torch.repeat_interleave(torch.arange(n), deg)
    src = torch.randint(0, n, (dst.numel(),), generator=g)
    w = torch.rand(dst.numel(), generator=g) + 0.05
    x = torch.randn(n, F, generator=g)
    ei = torch.stack([src, dst])
    ref = mo.aggregate_sum(x, ei, w)                                       # sequential fp32 in edge order per row
    ref64 = torch.zeros(n, F, dtype=torch.float64).index_add_(0, dst, w.double().view(-1, 1) * x.double()[src])
    rp, col, val = ops.csr_build(ei.cuda(), w.cuda(), n, ops.CSR_PLAIN)
    y = ops.spmm_csr(rp, col, val, x.cuda(), long_row_threshold=T).cpu()
    y2 = ops.spmm_csr(rp, col, val, x.cuda(), long_row_threshold=T).cpu()
    assert torch.equal(y, y2)                                              # deterministic
    short = deg <= T
    assert torch.equal(y[short], ref[short])                              # bit-identical where no split happened
    scale = (w.double().view(-1, 1) * x.double()[src]).abs()
    mag = torch.zeros(n, F, dtype=torch.float64).index_add_(0, dst, scale).clamp(min=1)
    err = ((y.double() - ref64).abs() / mag).max().item()
    err_seq = ((ref.double() - ref64).abs() / mag).max().item()
    record_parity("spmm_long_row_split", max_err_over_summed_magnitude=err, sequential_fp32_err=err_seq, tolerance=1e-5,
                  max_in_degree=120000, threshold=T)
    assert err <= 1e-5, err
    bias = torch.randn(F, generator=g)
    ym = ops.spmm_csr(rp, col, val, x.cuda(), mean=True, bias=bias.cuda(), act="relu", long_row_threshold=T).cpu()
    want = torch.relu(ref64 / deg.clamp(min=1).double().view(-1, 1) + bias.double())
    assert ((ym.double() - want).abs() / want.abs().clamp(min=1)).max() <= 1e-5
    y0 = ops.spmm_csr(rp, col, val, x.cuda(), long_row_threshold=0).cpu()  # unsplit path: whole matrix bit-identical
    assert torch.equal(y0, ref)


def test_automatic_long_row_threshold():
    """With long_row_threshold=None the library picks the threshold: a graph of exactly 2^22 edges is split at 256 edges
    for F = 64 (lane groups narrower than a warp) and at 2048 for F = 128, one edge fewer is not split at all.  The graph
    has rows of 257..2,000 edges and rows above 2,048, so the three explicit choices give three different results."""
    from gnnpn_sc_b200 import _lib, ops
    g = torch.Generator().manual_seed(17)
    n, E = 1 << 16, 1 << 22
    deg = torch.zeros(n, dtype=torch.int64)
    mid = torch.randperm(n, generator=g)[:304]
    deg[mid[:300]] = torch.randint(257, 2001, (300,), generator=g)
    deg[mid[300:]] = torch.randint(3000, 10001, (4,), generator=g)
    rest = (deg == 0).nonzero().flatten()
    deg[rest] = (E - int(deg.sum())) // rest.numel()
    deg[rest[:E - int(deg.sum())]] += 1
    assert int(deg.sum()) == E and int(deg[rest].max()) <= 256
    col = torch.randint(0, n, (E,), generator=g, dtype=torch.int32).cuda()
    val = (torch.rand(E, generator=g) + 0.05).cuda()

    def csr(d):
        rp = torch.zeros(n + 1, dtype=torch.int64)
        rp[1:] = d.cumsum(0)
        return rp.cuda(), col[:int(d.sum())], val[:int(d.sum())]

    def default_call(rp, c, v, x):                                         # -> (y, kernels launched)
        before = _lib.launch_count()
        y = ops.spmm_csr(rp, c, v, x)
        torch.cuda.synchronize()
        return y, _lib.launch_count() - before

    rp, c, v = csr(deg)
    for F, T in ((64, 256), (128, 2048)):
        x = torch.randn(n, F, generator=g).cuda()
        y, k = default_call(rp, c, v, x)
        assert k == 4                                                      # find, short rows, chunks, combine
        assert torch.equal(y, ops.spmm_csr(rp, c, v, x, long_row_threshold=T))
        for other in (256, 0):
            if other != T:
                assert not torch.equal(y, ops.spmm_csr(rp, c, v, x, long_row_threshold=other))
    deg1 = deg.clone()
    deg1[rest[0]] -= 1
    rp1, c1, v1 = csr(deg1)
    for F in (64, 128):
        x = torch.randn(n, F, generator=g).cuda()
        y, k = default_call(rp1, c1, v1, x)
        assert k == 1
        assert torch.equal(y, ops.spmm_csr(rp1, c1, v1, x, long_row_threshold=0))
