"""ML+2PN+WOA from host request graphs through ``pipeline.ML2PN.run`` (the ESWOA stage on the device), at the QWS and
Normal shapes of environment.ini's [QWS-WOA] / [Normal-WOA] sections.  One JSON line per shape:

* ``e2e``: instances/s of ``ML2PN.run`` over pinned host batches (request graphs, constraint tensors and the ESWOA
  arrays uploaded, services + objective + WOA results read back), whole batches of n instances, steady state;
* ``stage_ms``: CUDA events at the stage boundaries inside ``compose`` (ML + 2PN up to the objective, WOA prepare,
  WOA search), back-to-back steps;
* ``file_path``: the existing route on a bounded sample of the same picks -- ``allActions`` files ->
  ``WOA(..., engine="device").start()`` -- wall clock, the before-number;
* the GPU's name and power limit, read in the same run.

256 distinct synthetic request graphs (gnnpn_sc_b200.synth) are tiled to n instances; every instance is computed.
Writes only to a temporary directory (the file-path sample) and stdout.

    python scripts/bench_ml2pn_woa.py --n 18944 --steps 3 --file-sample 256
"""
from __future__ import annotations

import argparse
import configparser
import contextlib
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = {"qws": dict(section="QWS-WOA", S=2507, gcn=2, dist="qws"),
          "normal": dict(section="Normal-WOA", S=2500, gcn=4, dist="normal")}


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return {"gpu": q[0], "power_limit": q[1]}
    except (OSError, IndexError, subprocess.SubprocessError):
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": "unknown"}


def run_shape(shape: str, n: int, steps: int, file_sample: int):
    from gnnpn_sc_b200 import synth, loadData, trainML, modelML, modelPN as M, WOA as W
    from gnnpn_sc_b200.pipeline import ML2PN, constraint_arrays, woa_arrays
    from gnnpn_sc_b200.weights import reference_shaped_state_dict
    cfg = SHAPES[shape]
    ini = configparser.ConfigParser()
    ini.read(os.path.join(ROOT, "environment.ini"))
    sec = ini[cfg["section"]]
    K, N, S = int(sec["serCategory"]), int(sec["serviceNumber"]), cfg["S"]
    P, iters, reduct = int(sec["popSize"]), int(sec["MAX_Iter"]), float(sec["reduct"])
    dev = torch.device("cuda")
    ds = synth.ml_dataset(n_instances=256, K=K, S=S, seed=3, dist=cfg["dist"])
    samples = trainML.build_samples(loadData.ml_arrays(ds))
    reps = (n + len(samples) - 1) // len(samples)
    samples_n, nodef = (samples * reps)[:n], (ds["nodefeatures"] * reps)[:n]
    torch.manual_seed(0)
    net = modelML.Net(128, S, 20, 2, cfg["gcn"], isServices=True).to(dev)
    net.reset_parameters()
    pn = []
    for level, seed in (("Low", 1), ("High", 2)):
        m = M.CombinatorialRL(0, 256, K * N, 0, 10, 1, M.reward, "Dot", N, K, level=level)
        m.load_state_dict(reference_shaped_state_dict(256, 8, seed))
        pn.append(m.to(dev).eval())
    svc = type(samples[0])(**{k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in vars(samples[0]).items()})
    pipe = ML2PN(net.eval(), pn[0], pn[1], svc, ds["serviceFeature"], dev,
                 woa={"popSize": P, "MAX_Iter": iters, "reduct": reduct})
    ids = np.arange(n, dtype=np.int64)
    host = (trainML.collate_requests(samples_n, pin=True),
            *[torch.from_numpy(a).pin_memory() for a in constraint_arrays(nodef, K)],
            [torch.from_numpy(a).pin_memory() for a in (*woa_arrays(nodef, K), ids)])

    # per-stage times: compose on device-resident inputs, steps back to back
    rb = trainML.collate_requests(samples_n, device=dev)
    cons = [t.to(dev) for t in host[1:4]]
    woa = [t.to(dev) for t in host[4]]
    pipe.compose(rb, *cons, woa=woa)                                          # warm-up
    runs = []
    for _ in range(steps + 1):
        evs = []
        out = pipe.compose(rb, *cons, stage_events=evs, woa=woa, defer_check=True)
        runs.append(evs)
    torch.cuda.synchronize()
    b = [sum(evs[i].elapsed_time(evs[i + 1]) for evs in runs[1:]) / steps for i in range(6)]
    stage = {"ml_2pn": b[0] + b[1] + b[2] + b[3], "woa_prepare": b[4], "woa_search": b[5]}
    fit = out["woa_fitness"].cpu().numpy()

    # end to end from host batches
    list(pipe.run([host]))                                                     # warm the copy stream and pinned buffers
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for res in pipe.run([host] * steps):
        pass
    torch.cuda.synchronize()
    e2e_s = (time.perf_counter() - t0) / steps
    assert np.array_equal(res[2].numpy(), fit)

    # before: the same picks through allActions files and the file-level driver, on the first file_sample instances
    m = min(file_sample, n)
    idx = out["idx_high"][:, :m].cpu().numpy()
    rows = out["rows"][:m].cpu().numpy()
    with tempfile.TemporaryDirectory() as root:
        fds = dict(ds)
        fds["nodefeatures"] = [nodef[0]] * (3 * m) + nodef[:m]                # the test split is the last quarter
        fds["minCostList"] = [1.0] * (4 * m)
        fds["labels"] = [[0] * S] * (4 * m)
        fds["edge_indices"] = [ds["edge_indices"][0]] * (4 * m)
        synth.write_dataset(root, "ds", fds)
        actions = [[[float(v) for v in rows[i, idx[k, i], :4]] + [0, 0, 0, 0] for i in range(m)] for k in range(K)]
        os.makedirs(os.path.join(root, "solutions", "PNHigh", "ds"))
        with open(os.path.join(root, "solutions", "PNHigh", "ds", "allActions0.txt"), "w") as f:
            json.dump(actions, f)
        t0 = time.perf_counter()
        with contextlib.redirect_stdout(sys.stderr):                       # start() prints its progress line
            res_file = W.WOA("ds", K, 0, 1, 0, 0, N, reduct, 0, iters, P, root=root, engine="device").start()
        file_s = time.perf_counter() - t0
    # the file driver seeds instance k with 3m + k, the pipeline with k: the mean fitness values are comparable, not equal
    return {"workload": f"ml2pn_woa_{shape}", "K": K, "N": N, "S": S, "popSize": P, "MAX_Iter": iters, "reduct": reduct,
            "instances": n, "e2e": {"value": n / e2e_s, "unit": "instances/s", "ms_per_batch": e2e_s * 1e3},
            "stage_ms": stage, "woa_mean_fitness": float(fit.mean()),
            "file_path": {"instances": m, "s": file_s, "value": m / file_s, "unit": "instances/s",
                          "mean_fitness": float(np.mean([1.0 / q for q in res_file["quality"]]))},
            **gpu_info(), "note": "e2e: ML2PN.run on pinned host batches, whole batches; stage_ms: CUDA events inside "
                                  "compose; file_path: allActions -> WOA(engine='device').start(), wall clock"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=18944)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--file-sample", type=int, default=256)
    ap.add_argument("--shapes", default="qws,normal")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_ml2pn_woa.py measures the GPU: no CUDA device visible"
    for shape in args.shapes.split(","):
        print(json.dumps(run_shape(shape, args.n, args.steps, args.file_sample)), flush=True)


if __name__ == "__main__":
    main()
