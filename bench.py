#!/usr/bin/env python
"""bench.py -- composition instances/sec of the greedy ML+2PN decode (PNLow -> latent -> PNHigh,
trainPNHigh.py:131-144) on synthetic QWS-shaped instances, per the driver contract.

    python bench.py --gpus 1 --steps 5 --warmup 3                       # our CUDA path
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...                                 # reference CPU algorithm (oracle port)
    python bench.py --dump-outputs DIR ...                               # also write the last step's outputs as .npy

One "step" = one pass of the hot path over one batch of n instances per GPU:
encoder LSTM (L steps) + fused greedy decode (K steps) for PNLow, the same for PNHigh with PNLow's
window logits as latent, then the objective evaluator.  `value` = instances/s with inputs resident in
HBM; `e2e` = the same through the public module API (CombinatorialRL.forward) starting from pinned
HOST inputs and ending with the picks + rewards back on the host, copies inside the timed region.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

K_TASKS, N_CAND, HID, FEAT = 47, 5, 256, 8          # environment.ini [QWS-PNLow]/[QWS-PNHigh]
L_SEQ = K_TASKS * N_CAND
WORKLOAD = "qws_greedy_pnlow_pnhigh_decode"
FLOPS_PER_INSTANCE_STEP = 2 * HID * 4 * HID + 2 * FEAT * 4 * HID   # h.W_hh^T + folded x projection
ISSUED_OVER_ALGORITHMIC = 3 * (HID + 16) / (HID + FEAT)            # a_lo.w_hi + a_hi.w_hi + a_hi.w_lo, x padded to 16


def ncu_traffic(n: int, key: str = "encoder_dram_bytes"):
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel from the committed `ncu --set full`
    capture (profiles/*_seq_traffic.json), per launch; only reported when it was captured at this n."""
    p = os.path.join(ROOT, "profiles", "r02_seq_traffic.json")
    try:
        with open(p) as f:
            d = json.load(f)
        return d[key] if int(d["instances"]) == int(n) else None
    except (OSError, KeyError, ValueError):
        return None


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"hbm_gbs": d["hbm_gbs"], "bf16_burst": d["bf16_tflops"],
                "bf16_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "src": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_burst": 1590.0, "bf16_sustained": 1400.0, "src": "fallback"}


def decode_roofline(n, dec_launch_ms, pk, layout):
    """HBM roofline of the fused pointer decode (one launch = K steps: LSTM cell + window dots + softmax + pick).
    ALGORITHMIC bytes per instance (DESIGN 3.2): every encoding row read once (L*H*4), the window logits and
    probabilities written once (2*L*4), PNLow's latent window read by PNHigh (L*4, averaged over the two networks: L*2),
    picks (K*4), the picked raw rows (K*F*4) and the cell state in / out (2*H*4).  The decoder hidden states are not
    written by the fused decoder (nobody reads them in this loop)."""
    per_inst = L_SEQ * HID * 4 + 2 * L_SEQ * 4 + L_SEQ * 2 + K_TASKS * 4 + K_TASKS * FEAT * 4 + 2 * HID * 4
    if layout == 0:
        per_inst += K_TASKS * HID * 4                       # row-major path also writes dec_h
    gbs = n * per_inst / (dec_launch_ms * 1e-3) / 1e9
    return {"kernel": "lstm_seq_kernel<true,2,5> (persistent tcgen05 decoder: K steps in one launch, pointer dot products "
                      "fused into the cell epilogue over blocked encodings, thread-per-instance softmax / pick)"
                      if layout else "lstm_seq_kernel<true,2,0> (persistent decoder + separate pointer phase)",
            "bound": "hbm", "achieved": gbs, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": gbs / pk["hbm_gbs"],
            "avg_launch_ms": dec_launch_ms, "algorithmic_bytes_per_launch": n * per_inst,
            "traffic": ncu_traffic(n, "decoder_dram_bytes") if layout else None,
            "peak_source": pk["src"] + ": MEASURED_PEAKS.json hbm_gbs (copy bandwidth)"}


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:                                           # reap it: the benchmark leaves no process behind
                self.proc.wait(timeout=10)
            except subprocess.TimeoutExpired:
                self.proc.kill()
                self.proc.wait()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i] == "Active"})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ----------------------------------------------------------------------------- reference arm / cpu baseline
REF_MODEL = os.path.join(ROOT, "baseline", "_ref", "src", "models", "modelPN.py")


def _load_reference_module():
    """The UNMODIFIED reference ``src/models/modelPN.py`` (placed under baseline/_ref by
    baseline/install_reference.py), loaded by path under a private name, or None when it is not installed."""
    if not os.path.exists(REF_MODEL):
        return None
    import importlib.util
    spec = importlib.util.spec_from_file_location("_reference_modelPN", REF_MODEL)
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    return ref


def cpu_reference_rate(batches: int, batch: int = 128):
    """The reference's own CPU path on this box's host cores: greedy PNLow -> PNHigh + its ``reward()``
    (trainPNHigh.py:131-144) at the reference's batch size.  Runs the real ``CombinatorialRL`` classes from
    baseline/_ref when installed (kind "reference"), else the oracle port of the same loop (kind "port").
    Returns (instances/s, seconds per batch list, kind)."""
    import contextlib
    import io
    import torch
    from oracle import pn_oracle as po
    from gnnpn_sc_b200.synth import pn_instances
    torch.set_num_threads(os.cpu_count() or 1)
    cfg = po.PNConfig(seq_len=L_SEQ, s_number=N_CAND, s_category=K_TASKS)
    sd_lo, sd_hi = po.make_state_dict(cfg, 1), po.make_state_dict(cfg, 2)
    x = pn_instances(batch, K_TASKS, N_CAND, seed=1234)
    ref = _load_reference_module()
    if ref is not None:
        nets = []
        for level, sd in (("Low", sd_lo), ("High", sd_hi)):
            have_cuda = torch.cuda.is_available()
            if not have_cuda:                                # modelPN.py:151 calls .cuda() unconditionally
                saved, torch.Tensor.cuda = torch.Tensor.cuda, (lambda self, *a, **k: self)
            try:
                m = ref.CombinatorialRL(0, HID, L_SEQ, 0, 10, 1, ref.reward, "Dot", N_CAND, K_TASKS, use_cuda=False,
                                        level=level)
            finally:
                if not have_cuda:
                    torch.Tensor.cuda = saved
            m.actor.alpha = m.actor.alpha.cpu()              # CPU run of the reference (SURVEY 8c)
            m.load_state_dict(sd)
            nets.append(m.eval())

        def one_batch():
            with torch.no_grad(), contextlib.redirect_stdout(io.StringIO()):      # reward() prints every batch
                _, _, _, _, latent = nets[0](x, None, sample="greedy", training="SL")
                R, _, _, _, _ = nets[1](x, None, latent, sample="greedy", training="RL")
            return R
        kind = "reference"
    else:
        def one_batch():
            res = po.greedy_low_high(sd_lo, sd_hi, cfg, x, faithful_loops=True)
            return po.reward(list(res["actions"]), None, K_TASKS, "High", 0)
        kind = "port"
    times = []
    for i in range(batches + 1):                       # first batch is warm-up
        t0 = time.perf_counter()
        one_batch()
        if i:
            times.append(time.perf_counter() - t0)
    return batch / min(times), times, kind


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    batch = 128
    t0 = time.perf_counter()
    rate, times, kind = cpu_reference_rate(args.steps, batch)
    ms = 1e3 * statistics.mean(times)
    value = batch / statistics.mean(times)
    line = {
        "impl": "reference", "metric": "composition instances/sec (ML+2PN greedy)", "value": value,
        "unit": "instances/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": {"workload": WORKLOAD, "instances_per_step": batch, "K": K_TASKS,
                                        "N": N_CAND, "L": L_SEQ, "hidden": HID},
        "cpu_baseline": {"value": value, "unit": "instances/s", "cores": os.cpu_count(), "kind": kind,
                         "sample": f"{args.steps} batches of {batch} instances (reference batch size, "
                                   "trainPNHigh.py:248), " + (
                                       "the reference's own CombinatorialRL.forward x2 + reward() from baseline/_ref"
                                       if kind == "reference" else "oracle port of modelPN.py incl. its per-row loops")
                                   + ", torch CPU fp32, all host threads"},
        "e2e": {"value": value, "unit": "instances/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": time.perf_counter() - t0,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------- full ML+2PN pipeline (BASELINE config 3)
PIPE_SHAPES = {"normal": dict(K=50, N=10, S=2500, gcn=4, dist="normal"),      # environment.ini [Normal-*]
               "qws": dict(K=47, N=5, S=2507, gcn=2, dist="qws")}              # environment.ini [QWS-*]


def pipeline_block(dev, shape: str, n: int, steps: int, warmup: int):
    """`main.py <ds> ML+2PN` as one device-resident pipeline on n request instances: Net scores (modelML.py:131-176) ->
    per-category top-N feasible candidates (loadData.py:99-150) -> PNLow greedy -> PNHigh greedy (trainPNHigh.py:131-144)
    -> objective (ML2PN.py:6-12).  `value`: inputs resident in HBM, the ML stage INSIDE the timed region; `e2e`: request
    graphs + constraint tensors uploaded from pinned host memory and the chosen services + objective read back, every step.
    256 distinct synthetic request graphs (gnnpn_sc_b200.synth) are tiled to n instances; every instance is computed."""
    import torch
    from gnnpn_sc_b200 import synth, loadData, trainML, modelML, ops, modelPN as M
    from gnnpn_sc_b200.pipeline import ML2PN, constraint_arrays
    from gnnpn_sc_b200.weights import reference_shaped_state_dict
    cfg = PIPE_SHAPES[shape]
    K, N, S = cfg["K"], cfg["N"], cfg["S"]
    ds = synth.ml_dataset(n_instances=256, K=K, S=S, seed=3, dist=cfg["dist"])
    samples = trainML.build_samples(loadData.ml_arrays(ds))
    reps = (n + len(samples) - 1) // len(samples)
    samples_n, nodef = (samples * reps)[:n], (ds["nodefeatures"] * reps)[:n]
    torch.manual_seed(0)
    net = modelML.Net(128, S, 20, 2, cfg["gcn"], isServices=True).to(dev)
    net.reset_parameters()
    net.eval()
    pn = []
    for level, seed in (("Low", 1), ("High", 2)):
        m = M.CombinatorialRL(0, HID, K * N, 0, 10, 1, M.reward, "Dot", N, K, level=level)
        m.load_state_dict(reference_shaped_state_dict(HID, FEAT, seed))
        pn.append(m.to(dev).eval())
    svc = type(samples[0])(**{k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in vars(samples[0]).items()})
    pipe = ML2PN(net, pn[0], pn[1], svc, ds["serviceFeature"], dev)
    host = trainML.collate_requests(samples_n, pin=True)
    cons_host = [torch.from_numpy(a).pin_memory() for a in constraint_arrays(nodef, K)]
    h2d = sum(t.numel() * t.element_size() for t in (host.x, host.edge_index, host.batch, *cons_host))

    def upload():
        b = type(host)(x=host.x.to(dev, non_blocking=True), edge_index=host.edge_index.to(dev, non_blocking=True),
                       batch=host.batch.to(dev, non_blocking=True), num_graphs=host.num_graphs)
        return b, [t.to(dev, non_blocking=True) for t in cons_host]

    batch, cons = upload()
    out = {}

    def device_step():
        out.update(pipe.compose(batch, *cons))

    def e2e_steps(k):
        # the public host-batch API: every step uploads its request graphs + constraint tensors from pinned host memory (copy
        # stream, under the previous step's kernels) and reads the chosen services + objective back to the host
        for res in pipe.run((host, *cons_host) for _ in range(k)):
            pass
        return res

    def timed(fn, k):
        torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(k):
            fn()
        t1.record()
        torch.cuda.synchronize()
        return t0.elapsed_time(t1) / k

    for _ in range(warmup):
        device_step()
    ms = timed(device_step, steps)
    # per-stage times from CUDA events recorded INSIDE compose at the stage boundaries, steady state: the steps run back
    # to back (no host sync between them, as in the whole-step timing above); the first one only fills the queue
    names = ("net_scores", "select_candidates", "pnlow_pnhigh", "objective")
    runs = []
    for _ in range(steps + 1):
        evs = []
        out.update(pipe.compose(batch, *cons, stage_events=evs))
        runs.append(evs)
    torch.cuda.synchronize()
    stage = {k: sum(evs[i].elapsed_time(evs[i + 1]) for evs in runs[1:]) / steps for i, k in enumerate(names)}
    e2e_steps(4)                                         # warm the copy stream's allocator pool and the pinned result buffers
    k_e2e = max(6, 2 * steps)                            # the first upload of a run is not overlapped: amortise it
    e2e_ms = timed(lambda: e2e_steps(k_e2e), 1) / k_e2e
    d2h = n * K * 4 + n * 4
    return {"workload": f"ml2pn_pipeline_{shape}", "K": K, "N": N, "L": K * N, "S": S, "gcn_layers": cfg["gcn"],
            "instances": n, "ms_per_step": ms, "value": n / (ms * 1e-3), "unit": "instances/s", "stage_ms": stage,
            "e2e": {"value": n / (e2e_ms * 1e-3), "unit": "instances/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "mean_violations": float(out["violations"].float().mean()), "mean_objective": float(out["objective"].mean()),
            "note": "ML stage inside the timed region; stage_ms from CUDA events at the stage boundaries inside compose"}


DUMP_INSTANCES = 8192          # at most 8192 x 1,040 floats (34 MB) for the qws shape, whatever the batch


def dump_outputs(path: str, n: int, arrays):
    """``--dump-outputs``: write ``{name: (device tensor, instance axis)}`` as ``path/<name>.npy`` in float32 (picks and
    violation counts are small integers, exact in float32).  Batches above DUMP_INSTANCES instances keep a fixed, seeded
    sample of instances, the same in every array; ``instances.npy`` lists them (float64)."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    rows = np.arange(n)
    if n > DUMP_INSTANCES:
        rows = np.sort(np.random.default_rng(0).choice(n, DUMP_INSTANCES, replace=False))
    np.save(os.path.join(path, "instances.npy"), rows.astype(np.float64))
    for name, (t, axis) in arrays.items():
        sel = t.index_select(axis, torch.from_numpy(rows).to(t.device))
        np.save(os.path.join(path, f"{name}.npy"), sel.cpu().numpy().astype(np.float32))


# ----------------------------------------------------------------------------- our arm
def run_ours(args):
    import torch
    import torch.distributed as dist
    from gnnpn_sc_b200 import _lib, modelPN as M, ops
    from gnnpn_sc_b200.synth import pn_instances
    from gnnpn_sc_b200.weights import reference_shaped_state_dict

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    n = args.instances
    x_host = pn_instances(n, K_TASKS, N_CAND, seed=1234 + rank).pin_memory()
    x = x_host.to(dev)
    nets = []
    for level, seed in (("Low", 1), ("High", 2)):
        m = M.CombinatorialRL(0, HID, L_SEQ, 0, 10, 1, M.reward, "Dot", N_CAND, K_TASKS, level=level)
        m.load_state_dict(reference_shaped_state_dict(HID, FEAT, seed))
        nets.append(m.to(dev).eval())
    low, high = nets
    low.actor.impl = high.actor.impl = args.kernel
    enc_w_lo, dec_w_lo = low.actor._packed_weights()
    enc_w_hi, dec_w_hi = high.actor._packed_weights()

    # persistent device buffers for the HBM-resident loop (no allocation inside the timed region)
    ws = ops.pn_workspace(n, HID, dev, args.kernel)
    # encodings layout the dispatcher wants for this batch: blocked (pointer dots fused into the decoder's cell
    # epilogue) when the batch runs on the persistent CTA-pair scan
    layout = ops.pn_enc_layout(n, L_SEQ, FEAT, K_TASKS, N_CAND, ws is not None)
    enc_out = ops.enc_out_empty(n, L_SEQ, HID, layout, dev)
    c = torch.empty(n, HID, device=dev)
    # decoder hidden states (dec_h) are a by-product nobody reads in this loop: the fused decoder keeps them on chip
    bufs = [(torch.empty(n, K_TASKS, HID, device=dev) if layout == ops.ENC_ROWMAJOR else None,
             torch.empty(K_TASKS, n, device=dev, dtype=torch.int32),
             torch.empty(n, L_SEQ, device=dev), torch.empty(n, L_SEQ, device=dev)) for _ in range(2)]
    enc_ev, dec_ev = [], []
    enc_mib = (enc_out.numel() * 4) >> 20
    reward = [None]                                        # pn_reward of the latest step (violations, objFunc, reward)

    def device_step(record: bool):
        lat = None
        for lvl, (ew, dw) in enumerate(((enc_w_lo, dec_w_lo), (enc_w_hi, dec_w_hi))):
            if record:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
            ops.lstm_encode(x, ew, HID, enc_out, c, workspace=ws, layout=layout)
            if record:
                e1.record()
                enc_ev.append((e0, e1))
            _, idx, wl, _ = ops.pn_decode_greedy(x, enc_out, c, dw, K_TASKS, N_CAND, latent_win=lat, out=bufs[lvl],
                                                 workspace=ws, enc_layout=layout)
            if record:
                e2 = torch.cuda.Event(enable_timing=True)
                e2.record()
                dec_ev.append((e1, e2))
            lat = wl
        reward[0] = ops.pn_reward(x, idx)

    from gnnpn_sc_b200.pipeline import GreedyLowHigh
    composer = GreedyLowHigh(low, high, dev)

    def e2e_steps(k):
        # public API from HOST batches: every step uploads its own batch from pinned memory (overlapped with the
        # previous step's kernels by the double-buffered loader) and reads picks + rewards back to the host
        for idx_host, r_host in composer.run(x_host for _ in range(k)):
            pass
        return idx_host, r_host

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(steps):
            fn()
        t1.record()
        barrier()
        ms = torch.tensor([t0.elapsed_time(t1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    for _ in range(args.warmup):
        device_step(False)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = _lib.launch_count()
    ms_total = timed(lambda: device_step(True), args.steps)
    launches = _lib.launch_count() - launches0
    if rank == 0 and args.dump_outputs:
        # bufs[level] = (dec_h, picks [K, n], window logits [n, L], window probabilities [n, L]) of the last step
        dump_outputs(args.dump_outputs, n, {
            "pnlow_picks": (bufs[0][1], 1), "pnlow_window_logits": (bufs[0][2], 0), "pnlow_window_probs": (bufs[0][3], 0),
            "pnhigh_picks": (bufs[1][1], 1), "pnhigh_window_logits": (bufs[1][2], 0), "pnhigh_window_probs": (bufs[1][3], 0),
            "violations": (reward[0][0], 0), "objective": (reward[0][1], 0), "reward": (reward[0][2], 0)})
    enc_launch_ms = sum(a.elapsed_time(b) for a, b in enc_ev) / len(enc_ev)        # avg encoder-scan launch, ms
    dec_launch_ms = sum(a.elapsed_time(b) for a, b in dec_ev) / len(dec_ev)        # avg fused-decode launch, ms
    seq_on = args.kernel == "tc" and (ops.get_option("persistent") & 1)
    enc_ms = enc_launch_ms / L_SEQ                                                 # per recurrence step

    e2e_steps(max(1, min(args.warmup, 2)))
    e2e_ms = timed(lambda: e2e_steps(args.steps), 1)
    clocks = sampler.stop() if rank == 0 else None

    # latency of ONE reference-sized batch (B = 128, trainPNLow.py:221) through the public pipeline call (low_high: the two
    # encoders side by side on two streams, then the decoders): the dispatcher runs the column-split cluster scan there;
    # option scan = 0 forces the CTA-pair scan for comparison
    small = None
    if rank == 0:
        from gnnpn_sc_b200.pipeline import low_high
        nb = 128
        xs = x[:nb].contiguous()
        side_s = torch.cuda.Stream(dev)
        chk = low.actor.check_inputs, high.actor.check_inputs
        low.actor.check_inputs = high.actor.check_inputs = False          # no host sync inside the timed loop

        def small_step():
            with torch.no_grad():
                return low_high(low, high, xs, side_s, own_buffers=False)[1]

        small = {"instances": nb}
        for key, mode in (("ms", -1), ("ms_cta_pair_scan", 0)):
            ops.set_option("scan", mode)
            for _ in range(3):
                small_step()
            torch.cuda.synchronize()
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            for _ in range(10):
                small_step()
            t1.record()
            torch.cuda.synchronize()
            small[key] = t0.elapsed_time(t1) / 10
        ops.set_option("scan", -1)
        low.actor.check_inputs, high.actor.check_inputs = chk
        low.actor.last = high.actor.last = None
        small["instances_per_s"] = nb / (small["ms"] * 1e-3)

    # second half of BASELINE.json's metric: CSR aggregation GB/s against the HBM peak (one point of the sweep in
    # scripts/bench_agg.py: E = 2^26 edges, mean degree 16, F = 64, weighted -- 17.9 GB of algorithmic traffic >> L2)
    agg = None
    if rank == 0 and not args.no_aggregation:
        from scripts.bench_agg import make_csr
        Na, Fa = (1 << 26) // 16, 64
        rowptr, col, val, Ea = make_csr(Na, 16, 0.0, True, dev)
        xa = torch.empty(Na, Fa, device=dev).uniform_(-1, 1)
        ya = torch.empty(Na, Fa, device=dev)
        for _ in range(3):
            ops.spmm_csr(rowptr, col, val, xa, out=ya)
        ts = []
        for _ in range(5):
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record(); ops.spmm_csr(rowptr, col, val, xa, out=ya); t1.record(); torch.cuda.synchronize()
            ts.append(t0.elapsed_time(t1))
        ms_a = sorted(ts)[len(ts) // 2]
        bytes_a = Ea * (8 + 4 * Fa) + Na * 4 * Fa + (Na + 1) * 8
        agg = {"kernel": "spmm_csr_kernel", "E": Ea, "N": Na, "F": Fa, "ms": ms_a, "algorithmic_bytes": bytes_a,
               "GBps": bytes_a / ms_a / 1e6, "frac_of_hbm_peak": bytes_a / ms_a / 1e6 / peaks()["hbm_gbs"]}
        del rowptr, col, val, xa, ya

    # the attention of the decode loop ALONE (no LSTM step in the launches): the stand-alone pointer kernel over all K steps on
    # row-major encodings and the decoder states of a real decode -- the HBM roofline point of north_star's "attention"
    attention = None
    if rank == 0 and world == 1 and not args.no_attention and layout == ops.ENC_BLOCKED128:
        ops.lstm_encode(x, enc_w_hi, HID, enc_out, c, workspace=ws, layout=layout)
        dec_h_a = torch.empty(n, K_TASKS, HID, device=dev)
        ops.pn_decode_greedy(x, enc_out, c, dec_w_hi, K_TASKS, N_CAND, out=(dec_h_a,) + tuple(bufs[1][1:]), workspace=ws,
                             enc_layout=layout)
        enc_rm = ops.enc_to_rowmajor(enc_out, n, L_SEQ, HID)
        out_a = (torch.empty(K_TASKS, n, device=dev, dtype=torch.int32), torch.empty(n, L_SEQ, device=dev),
                 torch.empty(n, L_SEQ, device=dev))
        for _ in range(3):
            ops.pn_attention_windows(enc_rm, dec_h_a, N_CAND, out=out_a)
        ts = []
        for _ in range(5):
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record(); ops.pn_attention_windows(enc_rm, dec_h_a, N_CAND, out=out_a); t1.record(); torch.cuda.synchronize()
            ts.append(t0.elapsed_time(t1))
        ms_at = sorted(ts)[len(ts) // 2]
        same = bool(torch.equal(out_a[1], bufs[1][2]) and torch.equal(out_a[0], bufs[1][1]))
        bytes_at = n * (L_SEQ * HID * 4 + K_TASKS * HID * 4 + 2 * L_SEQ * 4 + K_TASKS * 4)
        attention = {"kernel": "pointer_step_dot_kernel x K (stand-alone attention over the windows, row-major encodings)",
                     "ms": ms_at, "algorithmic_bytes": bytes_at, "GBps": bytes_at / ms_at / 1e6,
                     "frac_of_hbm_peak": bytes_at / ms_at / 1e6 / peaks()["hbm_gbs"],
                     "bitwise_equal_to_fused_decoder": same}
        del enc_rm, dec_h_a, out_a

    pipeline = None
    if rank == 0 and world == 1 and not args.no_pipeline:
        del enc_out, bufs                                    # the pipeline allocates its own encodings (2 x 9.7 GB at Normal)
        torch.cuda.empty_cache()
        pipeline = [pipeline_block(dev, shape, n, max(3, args.steps // 2), 2) for shape in ("normal", "qws")]

    lt = torch.tensor([launches], device=dev, dtype=torch.int64)
    if world > 1:
        dist.all_reduce(lt)
    if rank == 0:
        pk = peaks()
        ms_per_step = ms_total / args.steps
        value = world * n / (ms_per_step * 1e-3)
        e2e_value = world * n / (e2e_ms / args.steps * 1e-3)
        achieved = n * FLOPS_PER_INSTANCE_STEP / (enc_ms * 1e-3) / 1e12
        peak = pk["bf16_sustained"] / 2
        issued = achieved * ISSUED_OVER_ALGORITHMIC if args.kernel == "tc" else achieved
        if seq_on:
            kname = ("lstm_seq_kernel<false,2> (persistent tcgen05 encoder scan: all L steps in one launch, "
                     "3xFP16-split MMAs with fp32 accumulate in TMEM + fused LSTM cell)")
        elif args.kernel == "tc":
            kname = "tc_mainloop_kernel<LstmEpilogue> (tcgen05 recurrence GEMM + fused cell, one launch per step)"
        else:
            kname = "lstm_step_ffma_kernel (fp32 FFMA recurrence GEMM + fused cell)"
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            rate, times, kind = cpu_reference_rate(args.cpu_batches)
            cpu = {"value": rate, "unit": "instances/s", "cores": os.cpu_count(), "kind": kind,
                   "sample": f"best of {len(times)} batches of 128 instances (reference batch size), " + (
                       "the reference's own modelPN.CombinatorialRL x2 + reward() (baseline/_ref)" if kind == "reference"
                       else "oracle port of modelPN.py incl. its per-row python loops") + ", torch CPU fp32"}
        line = {
            "metric": "composition instances/sec (ML+2PN greedy)", "value": value, "unit": "instances/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": WORKLOAD, "instances_per_gpu_per_step": n, "K": K_TASKS, "N": N_CAND,
                       "L": L_SEQ, "hidden": HID, "kernel": args.kernel, "parallelism": f"instance-sharded x{world}, no collective",
                       "l2": f"working set {enc_mib} MiB of encodings per step >> 126 MB L2"},
            "roofline": {"kernel": kname, "bound": "tensor",
                         "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                         "traffic": ncu_traffic(n), "avg_launch_ms": enc_launch_ms if seq_on else enc_ms,
                         "steps_per_launch": L_SEQ if seq_on else 1,
                         "algorithmic_flops_per_launch": n * FLOPS_PER_INSTANCE_STEP * (L_SEQ if seq_on else 1),
                         "issued_tflops": issued, "issued_frac_of_bf16_sustained": issued / pk["bf16_sustained"],
                         "peak_source": f"{pk['src']}: fp32-accuracy GEMM -> TF32 dense proxy = 1/2 bf16 sustained "
                                        f"({pk['bf16_sustained']:.0f} TFLOP/s, SURVEY 8d); the 3 fp16 passes the split "
                                        "issues are not counted in `achieved`"},
            "roofline_decode": decode_roofline(n, dec_launch_ms, pk, layout),
            "cpu_baseline": cpu,
            "e2e": {"value": e2e_value, "unit": "instances/s", "h2d_bytes_per_step": x_host.numel() * 4,
                    "d2h_bytes_per_step": K_TASKS * n * 4 + n * 4, "ms_per_step": e2e_ms / args.steps},
            "gpu_launches": int(lt.item()), "clocks": clocks,
            "small_batch": small, "aggregation": agg, "roofline_attention": attention, "pipeline": pipeline,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# ----------------------------------------------------------------------------- scale-up workload (BASELINE config 4)
def run_scaleup(args):
    """100 abstract tasks x 1000 candidates per task (L = 100,000), instance-sharded over the ranks with no collective
    (SURVEY 8e): every rank decodes its own block PNLow -> PNHigh -> objective.  One step = one pass over n instances per
    GPU; the encodings are 102 MB per instance, so a 180 GB GPU holds one network's encodings of ~1,500 instances at a
    time (PNLow's are released before PNHigh's are produced).  Latency-bound: 100,000 dependent LSTM steps per network."""
    import torch
    import torch.distributed as dist
    from gnnpn_sc_b200 import _lib, modelPN as M
    from gnnpn_sc_b200.synth import pn_instances
    from gnnpn_sc_b200.weights import reference_shaped_state_dict
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    K, N = 100, 1000
    L = K * N
    n = args.instances if args.instances != 18944 else 1280          # 10 groups of 128: 131 GB of encodings (one network at a time)
    x_host = pn_instances(n, K, N, seed=77 + rank).pin_memory()
    nets = []
    for level, seed in (("Low", 1), ("High", 2)):
        m = M.CombinatorialRL(0, HID, L, 0, 10, 1, M.reward, "Dot", N, K, level=level)
        m.load_state_dict(reference_shaped_state_dict(HID, FEAT, seed))
        m.actor.check_inputs = False
        nets.append(m.to(dev).eval())
    low, high = nets
    # one encodings buffer, shared: PNLow's encodings are dead once its decode is enqueued (same stream order)
    low.actor.enc_buffer = high.actor.enc_buffer = torch.empty(n * L * HID, device=dev)

    def step(x):
        with torch.no_grad():
            _, _, _, _, latent = low(x, None, sample="greedy", training="SL")
            lat = M.WindowLogits(K, latent.window, None)      # keep only the compact window: PNLow's encodings are freed
            del latent
            low.actor.last = None
            R, _, _, idx, _ = high(x, None, lat, sample="greedy", training="RL")
            high.actor.last = None
        return R, torch.stack(idx).to(torch.int32)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(steps):
            fn()
        t1.record()
        barrier()
        ms = torch.tensor([t0.elapsed_time(t1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    x = x_host.to(dev)
    for _ in range(args.warmup):
        step(x)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = _lib.launch_count()
    ms = timed(lambda: step(x), args.steps) / args.steps
    launches = _lib.launch_count() - launches0

    def e2e():
        R, idx = step(x_host.to(dev, non_blocking=True))
        return R.cpu(), idx.cpu()
    e2e_ms = timed(e2e, max(1, args.steps // 2)) / max(1, args.steps // 2)
    clocks = sampler.stop() if rank == 0 else None
    lt = torch.tensor([launches], device=dev, dtype=torch.int64)
    if world > 1:
        dist.all_reduce(lt)
    if rank == 0:
        value = world * n / (ms * 1e-3)
        print(json.dumps({
            "metric": "composition instances/sec (ML+2PN greedy)", "value": value, "unit": "instances/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "scaleup_100x1000_greedy_pnlow_pnhigh_decode", "instances_per_gpu_per_step": n, "K": K,
                       "N": N, "L": L, "hidden": HID, "parallelism": f"instance-sharded x{world}, no collective",
                       "l2": f"{n * L * HID * 4 >> 30} GiB of encodings per network per step >> 126 MB L2"},
            "per_gpu_instances_per_s": value / world,
            "latency": {"dependent_lstm_steps_per_network": L + K, "us_per_encoder_step": ms * 1e3 / (2 * (L + K)),
                        "note": "column-split cluster scan (8-CTA clusters); step time bounds the whole pass"},
            "e2e": {"value": world * n / (e2e_ms * 1e-3), "unit": "instances/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": x_host.numel() * 4, "d2h_bytes_per_step": K * n * 4 + n * 4},
            "gpu_launches": int(lt.item()), "clocks": clocks}))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--instances", type=int, default=18944,
                    help="composition instances per GPU per step (default: one full wave, 148 SMs x 128)")
    ap.add_argument("--cpu-batches", type=int, default=8)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-aggregation", action="store_true", help="skip the CSR aggregation GB/s point")
    ap.add_argument("--no-attention", action="store_true", help="skip the attention-only (stand-alone pointer kernel) roofline point")
    ap.add_argument("--no-pipeline", action="store_true", help="skip the full ML+2PN pipeline block (BASELINE config 3)")
    ap.add_argument("--kernel", default="tc", choices=["tc", "ffma"],
                    help="recurrence kernel: tcgen05 3xTF32 (default) or strict-fp32 FFMA")
    ap.add_argument("--workload", default="qws", choices=["qws", "scaleup"],
                    help="qws: the headline (BASELINE config 2/3); scaleup: 100 tasks x 1000 candidates (config 4)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (picks, window logits and probabilities "
                         "of PNLow and PNHigh, objective and reward; rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.workload != "qws"):
        ap.error("--dump-outputs writes the outputs of the headline workload (--impl ours --workload qws)")
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "scaleup":
        run_scaleup(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
