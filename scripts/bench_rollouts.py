"""Best-of-R sampled decoding through ML+2PN: what an extra PNHigh rollout costs and what best-of-R gains over greedy, at
the QWS and Normal shapes of environment.ini's [QWS-WOA] / [Normal-WOA] sections.  One JSON line per (shape, n, R):

* ``e2e``: ms per batch and instances/s of ``pipeline.ML2PN(..., rollouts=R).run`` over pinned host batches (request
  graphs and constraint tensors uploaded, services + objective read back), whole batches of n, steady state;
* ``decoder_ms`` / ``decoder_ms_per_rollout``: one ``gnnpn_pn_decode_rollouts_f32`` launch of PNHigh (CUDA events,
  encodings computed once before the timed launches), and that over R;
* ``high_stage_ms``: PNHigh's part of the decode, shared encodings (one encoder + one rollout launch + the best-rollout
  kernel) against ``naive`` row replication (the rows repeated R times through the encoder and a sampled decode, then
  the same best-rollout kernel), CUDA events; the naive arm runs for R <= 4 at n = 18,944 (its encodings are R x 4.6 GB);
* ``score``: mean ML+2PN score of the chosen compositions (``gnnpn_ml2pn_score_f64`` as ``ML2PN.check`` computes it:
  objective + 1 per violated global constraint, lower is better), best-of-R and greedy, on the same batch;
* the GPU's name and power limit, read in the same run.

256 distinct synthetic request graphs (gnnpn_sc_b200.synth) are tiled to n instances.  Writes only to stdout.

    python scripts/bench_rollouts.py --n 1920,18944 --rollouts 1,4,16,64 --steps 3
"""
from __future__ import annotations

import argparse
import configparser
import json
import os
import subprocess
import sys
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


def events_ms(fn, reps):
    """Mean CUDA-event time of fn() over reps calls after one warm-up call."""
    fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def mean_score(rows, idx, K):
    """Mean ``ML2PN.calc`` score of the picks ``idx`` [K, n] (``ML2PN.composition_scores``, as ``ML2PN.check``)."""
    from gnnpn_sc_b200.ML2PN import composition_scores
    r = rows.cpu().numpy()
    i = idx.cpu().numpy()
    acts = [r[np.arange(r.shape[0]), i[k]] for k in range(K)]                 # K x [n, 8]
    return float(composition_scores(acts, K, r[:, 0, 4:8].astype(np.float64)).mean())


def run_shape(shape, ns, Rs, steps, gi):
    from gnnpn_sc_b200 import synth, loadData, trainML, modelML, modelPN as M, ops
    from gnnpn_sc_b200.pipeline import ML2PN, constraint_arrays
    from gnnpn_sc_b200.weights import reference_shaped_state_dict
    cfg = SHAPES[shape]
    ini = configparser.ConfigParser()
    ini.read(os.path.join(ROOT, "environment.ini"))
    sec = ini[cfg["section"]]
    K, N, S = int(sec["serCategory"]), int(sec["serviceNumber"]), cfg["S"]
    dev = torch.device("cuda")
    ds = synth.ml_dataset(n_instances=256, K=K, S=S, seed=3, dist=cfg["dist"])
    samples = trainML.build_samples(loadData.ml_arrays(ds))
    torch.manual_seed(0)
    net = modelML.Net(128, S, 20, 2, cfg["gcn"], isServices=True).to(dev)
    net.reset_parameters()
    pn = []
    for level, seed in (("Low", 1), ("High", 2)):
        m = M.CombinatorialRL(0, 256, K * N, 0, 10, 1, M.reward, "Dot", N, K, level=level)
        m.load_state_dict(reference_shaped_state_dict(256, 8, seed))
        pn.append(m.to(dev).eval())
    low, high = pn
    svc = type(samples[0])(**{k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in vars(samples[0]).items()})
    for n in ns:
        reps = (n + len(samples) - 1) // len(samples)
        samples_n, nodef = (samples * reps)[:n], (ds["nodefeatures"] * reps)[:n]
        host = (trainML.collate_requests(samples_n, pin=True),
                *[torch.from_numpy(a).pin_memory() for a in constraint_arrays(nodef, K)])
        rb = trainML.collate_requests(samples_n, device=dev)
        cons = [t.to(dev) for t in host[1:4]]
        greedy_score = None
        for R in Rs:
            pipe = ML2PN(net.eval(), low, high, svc, ds["serviceFeature"], dev, rollouts=R)
            high.actor.generator = torch.Generator(device=dev).manual_seed(0)
            out = pipe.compose(rb, *cons)
            rows = out["rows"]
            score = mean_score(rows, out["idx_high"], K)
            if R == 1:
                greedy_score = score
            list(pipe.run([host]))                                             # warm the copy stream and pinned buffers
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in pipe.run([host] * steps):
                pass
            torch.cuda.synchronize()
            e2e_s = (time.perf_counter() - t0) / steps

            with torch.no_grad():
                _, _, _, _, latent = low(rows, None, sample="greedy", training="SL")
            actor = high.actor
            actor.own_enc_buffer(rows)
            enc = actor.encode(rows)
            dec_ms = events_ms(lambda: actor.decode_rollouts(rows, latent, R, encoded=enc), steps)
            del enc
            shared_ms = events_ms(lambda: high.best_of(rows, None, latent, rollouts=R), steps)
            naive_ms = None
            if R > 1 and (n < 10000 or R <= 4):
                x_rep = rows.repeat(R, 1, 1)
                lat_rep = M.WindowLogits(K, latent.window.repeat(R, 1), None)
                saved = actor.enc_buffer
                actor.enc_buffer = None                                        # the replicated batch gets its own buffer

                def naive():
                    with torch.no_grad():
                        _, _, _, idx_rep, _ = high(x_rep, None, lat_rep, sample="sample", training="SL")
                    ops.pn_best_rollout(rows, torch.stack(idx_rep).to(torch.int32).view(K, R, n).transpose(0, 1))
                naive_ms = events_ms(naive, steps)
                actor.enc_buffer = saved
                del x_rep, lat_rep
                torch.cuda.empty_cache()
            print(json.dumps({
                "workload": f"ml2pn_rollouts_{shape}", "K": K, "N": N, "S": S, "instances": n, "rollouts": R,
                "e2e": {"ms_per_batch": e2e_s * 1e3, "value": n / e2e_s, "unit": "instances/s"},
                "decoder_ms": dec_ms, "decoder_ms_per_rollout": dec_ms / R,
                "high_stage_ms": {"shared": shared_ms, "naive": naive_ms},
                "score": {"best_of_R": score, "greedy": greedy_score}, **gi,
                "note": "e2e: ML2PN.run on pinned host batches; decoder / high_stage: CUDA events; score: mean "
                        "gnnpn_ml2pn_score_f64 over the batch, lower is better"}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", default="1920,18944")
    ap.add_argument("--rollouts", default="1,4,16,64")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--shapes", default="qws,normal")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_rollouts.py measures the GPU: no CUDA device visible"
    Rs = [int(r) for r in args.rollouts.split(",")]
    assert Rs[0] == 1, "the first R must be 1: the greedy score every other point is compared with"
    gi = gpu_info()
    for shape in args.shapes.split(","):
        run_shape(shape, [int(v) for v in args.n.split(",")], Rs, args.steps, gi)


if __name__ == "__main__":
    main()
