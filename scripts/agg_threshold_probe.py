"""Long-row threshold probe: in-degree-Zipf graph (bench_agg.make_csr_indegree_zipf, E ~ 2^28), whole-call time of
ops.spmm_csr over split thresholds T (chunks of max(256, T / 8) edges) and feature widths, next to the uniform graph of the same size."""
import json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from scripts.bench_agg import make_csr, make_csr_indegree_zipf, time_point, peak

dev = torch.device("cuda")
flush = torch.zeros(64 << 20, device=dev)
E_t = 1 << int(os.environ.get("LOG2E", "28"))
N = E_t // 16
pk = peak()
for F in (32, 64, 128, 256):
    x = torch.empty(N, F, device=dev).uniform_(-1, 1)
    y = torch.empty(N, F, device=dev)
    rowptr, col, val, E = make_csr(N, 16, 0.0, True, dev)
    alg = E * (8 + 4 * F) + N * 4 * F + (N + 1) * 8
    ms = time_point(rowptr, col, val, x, y, 3, flush, False, long_row_threshold=0)
    ms_dyn = time_point(rowptr, col, val, x, y, 3, flush, False, long_row_threshold=2048)   # same kernel + the (empty) split passes
    print(json.dumps({"family": "uniform", "F": F, "E": E, "ms_static_kernel": ms, "frac": alg / ms / 1e6 / pk,
                      "ms_split_path": ms_dyn, "frac_split_path": alg / ms_dyn / 1e6 / pk}), flush=True)
    del rowptr, col, val
    rowptr, col, val, E = make_csr(N, 8, 0.0, True, dev)              # the Zipf family's floor: 8 edges per row
    alg = E * (8 + 4 * F) + N * 4 * F + (N + 1) * 8
    ms = time_point(rowptr, col, val, x, y, 3, flush, False, long_row_threshold=0)
    print(json.dumps({"family": "uniform_d8", "F": F, "E": E, "ms": ms, "frac": alg / ms / 1e6 / pk}), flush=True)
    del rowptr, col, val
    for fam, floor in (("indeg_zipf", 8), ("indeg_zipf_pure", 0)):
        rowptr, col, val, E, dmax = make_csr_indegree_zipf(N, E_t, True, dev, floor=floor)
        alg = E * (8 + 4 * F) + N * 4 * F + (N + 1) * 8
        for T, dyn in ((128, 0), (256, 0), (2048, 0)):
            ms = time_point(rowptr, col, val, x, y, 3, flush, False, long_row_threshold=T)
            print(json.dumps({"family": fam, "F": F, "E": E, "T": T, "dyn": dyn, "ms": ms,
                              "frac": alg / ms / 1e6 / pk, "dmax": dmax}), flush=True)
        del rowptr, col, val
    rowptr = col = val = None
    del rowptr, col, val, x, y
    torch.cuda.empty_cache()
