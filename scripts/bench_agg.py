"""Aggregation micro-benchmark (BASELINE.json configs[4], SURVEY 8d config 5): CSR segment-reduce GB/s over edge count and
feature width against the measured HBM peak.

    python scripts/bench_agg.py [--quick] [--out gpurun_out/agg_sweep.jsonl] [--one-launch]

ALGORITHMIC bytes = E*(4 + 4w + 4F) + N*4F + (N+1)*8   (col, val, one gathered row per edge; output written once; int64
rowptr read once).  Graph families:
  uniform        in-degree d for every row (16, or 64 when N*F would not fit), uniform sources
  src_zipf       uniform in-degree, Zipf-like skewed SOURCES (hot gathered rows)
  indeg_zipf     hub DESTINATION rows: every row has 8 edges and the other half of the edges is spread Zipf(1.0) over the
                 rows (the largest has >= 10^5 edges), rows in random order -- the shape of the service co-usage graph
                 (src/loadData.py:55-65); run with the long-row split path (ops.spmm_csr default) and, for comparison,
                 without it (long_row_threshold = 0)
  indeg_zipf_pure  the same without the floor: half of the edges sit in ~10^3 hub rows, most other rows have 1-3 edges
                 (per-row overhead, not hubs, bounds the short-row kernel there)
  qws_cousage    the synthetic QWS co-usage graph itself (S = 2,507 services, ~92k directed edges, gcn_norm weights), B
                 copies side by side as Net.forward batches them
Points whose gathered feature matrix is small against the 126 MB L2 are partly L2-served (the figure may exceed the HBM
peak): `gather_matrix_MB` is reported, and `--one-launch` runs every point exactly once so that the same command under
`ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum` gives the DRAM bytes per point (scripts/agg_label_l2.py merges
them: l2_served = measured DRAM bytes < 0.8 x algorithmic)."""
import argparse, json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from gnnpn_sc_b200 import ops


def peak():
    p = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "MEASURED_PEAKS.json")
    return json.load(open(p))["hbm_gbs"] if os.path.exists(p) else 6650.0


def make_csr(N, d, skew, weighted, dev):
    """uniform in-degree d; skew > 0: Zipf-like skewed sources"""
    E = N * d
    g = torch.Generator(device=dev).manual_seed(7)
    rowptr = torch.arange(0, E + 1, d, device=dev, dtype=torch.int64)
    if skew > 0:
        col = torch.empty(E, device=dev, dtype=torch.int32)
        chunk = 1 << 26
        for s in range(0, E, chunk):
            m = min(chunk, E - s)
            u = torch.rand(m, device=dev, generator=g)
            col[s:s + m] = (N * u.pow(1.0 + skew)).to(torch.int32).clamp_(max=N - 1)
    else:
        col = torch.randint(0, N, (E,), device=dev, dtype=torch.int32, generator=g)
    val = torch.rand(E, device=dev, generator=g) if weighted else None
    return rowptr, col, val, E


def make_csr_indegree_zipf(N, E_target, weighted, dev, alpha=1.0, floor=8):
    """Hub destination rows: every row has `floor` edges and the remaining edges are distributed Zipf(alpha) over the
    rows (floor = 0: pure Zipf, most rows have 1-3 edges); rows in random order, uniform sources."""
    g = torch.Generator(device=dev).manual_seed(11)
    w = 1.0 / torch.arange(1, N + 1, device=dev, dtype=torch.float64).pow(alpha)
    deg = floor + torch.floor(w / w.sum() * (E_target - floor * N)).to(torch.int64)
    deg = deg[torch.randperm(N, device=dev, generator=g)]
    rowptr = torch.zeros(N + 1, device=dev, dtype=torch.int64)
    rowptr[1:] = deg.cumsum(0)
    E = int(rowptr[-1].item())
    col = torch.randint(0, N, (E,), device=dev, dtype=torch.int32, generator=g)
    val = torch.rand(E, device=dev, generator=g) if weighted else None
    return rowptr, col, val, E, int(deg.max().item())


def make_qws_cousage(B, dev):
    from gnnpn_sc_b200 import synth, loadData
    ds = synth.ml_dataset(n_instances=1024, K=47, S=2507, seed=0)
    ei, w = loadData.cousage_graph(ds["labels"])
    ei = torch.tensor(ei, dtype=torch.long).view(2, -1)
    w = torch.tensor(w, dtype=torch.float)
    S = 2507
    eib = torch.cat([ei + b * S for b in range(B)], 1).to(dev)
    wb = w.repeat(B).to(dev)
    rowptr, col, val = ops.csr_build(eib, wb, B * S, ops.CSR_GCN_NORM)
    deg = rowptr[1:] - rowptr[:-1]
    return rowptr, col, val, int(col.numel()), int(deg.max().item()), B * S


def time_point(rowptr, col, val, x, y, iters, flush, one_launch, **kw):
    if one_launch:
        ops.spmm_csr(rowptr, col, val, x, out=y, **kw)
        torch.cuda.synchronize()
        return float("nan")
    for _ in range(3):
        ops.spmm_csr(rowptr, col, val, x, out=y, **kw)
    ts = []
    for _ in range(iters):
        if flush is not None:
            flush.add_(1.0)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); ops.spmm_csr(rowptr, col, val, x, out=y, **kw); b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return sorted(ts)[len(ts) // 2]


def record(family, E, N, F, weighted, ms, **extra):
    w = 1 if weighted else 0
    alg = E * (4 + 4 * w + 4 * F) + N * 4 * F + (N + 1) * 8
    compulsory = E * (4 + 4 * w) + 2 * N * 4 * F + (N + 1) * 8
    pk = peak()
    r = {"family": family, "E": E, "N": N, "F": F, "weighted": bool(weighted), "ms": ms, "algorithmic_bytes": alg,
         "alg_GBps": alg / ms / 1e6, "frac_of_hbm_peak": alg / ms / 1e6 / pk, "compulsory_GBps": compulsory / ms / 1e6,
         "gather_matrix_MB": N * F * 4 / 1e6, "peak_GBps": pk}
    r.update(extra)
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true")
    ap.add_argument("--one-launch", action="store_true", help="one launch per point, no timing (for an ncu DRAM-bytes pass)")
    ap.add_argument("--out", default="gpurun_out/agg_sweep.jsonl")
    args = ap.parse_args()
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    dev = torch.device("cuda")
    flush = torch.zeros(64 << 20, device=dev)
    Es = [1 << 20, 1 << 24] if args.quick else [1 << 20, 1 << 22, 1 << 24, 1 << 26, 1 << 28, 1 << 30]
    Fs = [64, 256] if args.quick else [32, 64, 128, 256]
    with open(args.out, "w") as f:
        def emit(r):
            f.write(json.dumps(r) + "\n"); f.flush()
            print(json.dumps(r), flush=True)
        for E_target in Es:
            for F in Fs:
                for family, weighted in (("uniform", True), ("uniform", False), ("src_zipf", True), ("indeg_zipf", True),
                                         ("indeg_zipf_pure", True)):
                    if (family != "uniform" or not weighted) and E_target not in (1 << 24, 1 << 28):
                        continue
                    try:
                        d = 16
                        N = E_target // d
                        if 2 * N * F * 4 > 120e9:
                            d = 64
                            N = E_target // d
                        iters = 3 if E_target >= (1 << 28) else 7
                        if family == "indeg_zipf_pure" and E_target != (1 << 24):
                            continue
                        if family.startswith("indeg_zipf"):
                            rowptr, col, val, E, dmax = make_csr_indegree_zipf(N, E_target, weighted, dev,
                                                                               floor=8 if family == "indeg_zipf" else 0)
                            x = torch.empty(N, F, device=dev).uniform_(-1, 1)
                            y = torch.empty(N, F, device=dev)
                            ms = time_point(rowptr, col, val, x, y, iters, flush, args.one_launch)
                            ms0 = time_point(rowptr, col, val, x, y, iters, flush, args.one_launch, long_row_threshold=0)
                            emit(record(family, E, N, F, weighted, ms, max_in_degree=dmax, long_row_threshold="auto",
                                        ms_without_split=ms0))
                        else:
                            rowptr, col, val, E = make_csr(N, d, 1.0 if family == "src_zipf" else 0.0, weighted, dev)
                            x = torch.empty(N, F, device=dev).uniform_(-1, 1)
                            y = torch.empty(N, F, device=dev)
                            ms = time_point(rowptr, col, val, x, y, iters, flush, args.one_launch)
                            emit(record(family, E, N, F, weighted, ms, deg=d))
                        del rowptr, col, val, x, y
                    except torch.OutOfMemoryError:
                        emit({"family": family, "E": E_target, "F": F, "weighted": weighted, "error": "oom"})
                    torch.cuda.empty_cache()
        for B in (8, 256):
            rowptr, col, val, E, dmax, N = make_qws_cousage(B, dev)
            for F, T in ((256, 2048),):   # the split path at F = 256's automatic threshold, also for B = 8 (< 2^22 edges)
                x = torch.empty(N, F, device=dev).uniform_(-1, 1)
                y = torch.empty(N, F, device=dev)
                ms = time_point(rowptr, col, val, x, y, 7, flush, args.one_launch, long_row_threshold=T)
                ms0 = time_point(rowptr, col, val, x, y, 7, flush, args.one_launch, long_row_threshold=0)
                emit(record("qws_cousage", E, N, F, True, ms, max_in_degree=dmax, copies=B, long_row_threshold=T,
                            ms_without_split=ms0))


if __name__ == "__main__":
    main()
