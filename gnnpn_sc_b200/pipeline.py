"""Host-side driver of the greedy ML+2PN decode -- the validation loop of ``trainPNHigh.py:131-144``
(PNLow greedy -> latent -> PNHigh greedy -> actions / reward) fed from HOST batches.

The reference runs that loop batch by batch with a blocking ``.cuda()`` per batch and ``.cpu()`` per step
(trainPNHigh.py:135-144).  Here the upload of batch i+1 runs on a side stream while the kernels of batch i
execute, and the small results (picks ``int32 [K, n]``, reward ``fp32 [n]``) come back through pinned buffers.
All arithmetic stays in the CUDA kernels behind ``modelPN.CombinatorialRL`` -- this file is plumbing.
"""
from __future__ import annotations

from typing import Iterable, Iterator, Tuple

import torch


NUM_SMS = 148          # B200


@torch.no_grad()
def _one_batch_behind(host_batches, upload, enqueue, device) -> Iterator[Tuple[torch.Tensor, ...]]:
    """Runs a pipeline over host batches with every batch's results read back one batch late.

    ``upload(item, slot)`` starts the host->device copy of one batch (on a copy stream) and returns a handle for
    ``enqueue(handle)``, which orders the current stream after that copy, enqueues the batch's kernels and returns
    (device results, device range flag | None).  The upload of batch i+1 overlaps the kernels of batch i, and the kernels
    of batch i+1 are enqueued before the host waits for the results of batch i (asynchronous device->host copies into
    double-buffered pinned tensors + an event), so the GPU never idles while the host prepares the next launches.  The
    input range flag travels with the results (no mid-batch sync).  Yields the results as cpu tensors, in order."""
    from .modelPN import PointerNet
    main = torch.cuda.current_stream(device)
    pinned = [None, None]
    pending = None                                        # (pinned results, pinned flag, event, handle) of the previous batch

    def finish(p):
        results, flag, ev, _ = p
        ev.synchronize()
        PointerNet.raise_if_out_of_range(flag)
        return tuple(t.clone() for t in results)          # the pinned buffers are reused two batches later

    it = iter(host_batches)
    item = next(it, None)
    handle = None if item is None else upload(item, 0)
    slot = 0
    while handle is not None:
        item = next(it, None)
        nxt = None if item is None else upload(item, slot ^ 1)   # overlaps this batch's kernels
        results, flag = enqueue(handle)
        if (pinned[slot] is None or len(pinned[slot][0]) != len(results)
                or any(o.shape != r.shape for o, r in zip(pinned[slot][0], results))):
            pinned[slot] = ([torch.empty(r.shape, dtype=r.dtype, pin_memory=True) for r in results],
                            torch.zeros(1, dtype=torch.int32, pin_memory=True))
        out, flag_pin = pinned[slot]
        for o, r in zip(out, results):
            o.copy_(r, non_blocking=True)
        if flag is not None:
            flag_pin.copy_(flag, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(main)
        if pending is not None:
            yield finish(pending)
        pending = (out, flag_pin if flag is not None else None, ev, handle)    # the handle keeps the batch's inputs alive
        handle, slot = nxt, slot ^ 1
    if pending is not None:
        yield finish(pending)


class GreedyLowHigh:
    def __init__(self, low, high, device=None, rollouts: int = 1):
        """``rollouts``: PNHigh decodes best-of-``rollouts`` (``low_high``); 1 is the greedy decode."""
        self.low, self.high = low.eval(), high.eval()
        self.rollouts = rollouts
        self.high.actor.check_inputs = False      # PNHigh decodes the rows PNLow has just range-checked
        self.device = torch.device(device if device is not None else "cuda")
        if self.device.type != "cuda":
            raise RuntimeError("GreedyLowHigh needs a CUDA device: the B200 path has no CPU fallback")
        self._copy = torch.cuda.Stream(self.device)
        self._side = torch.cuda.Stream(self.device)   # PNHigh's encoder runs here, next to PNLow's on the main stream
        self._stage = [None, None]            # device staging buffers (double buffer)
        self._ready = [torch.cuda.Event(), torch.cuda.Event()]
        self._consumed = [None, None]

    def _upload(self, x_host: torch.Tensor, slot: int) -> int:
        buf = self._stage[slot]
        if buf is None or buf.shape != x_host.shape:
            buf = self._stage[slot] = torch.empty(x_host.shape, device=self.device, dtype=torch.float32)
        if not x_host.is_pinned():
            x_host = x_host.pin_memory()
        with torch.cuda.stream(self._copy):
            if self._consumed[slot] is not None:          # the kernels that last read this buffer are done
                self._copy.wait_event(self._consumed[slot])
            buf.copy_(x_host, non_blocking=True)
            self._ready[slot].record(self._copy)
        return slot

    def _enqueue(self, slot: int):
        main = torch.cuda.current_stream(self.device)
        main.wait_event(self._ready[slot])
        latent, R, idx, flag = low_high(self.low, self.high, self._stage[slot], self._side, check="defer",
                                        rollouts=self.rollouts)
        self._consumed[slot] = torch.cuda.Event()
        self._consumed[slot].record(main)                 # after every kernel that reads the staging buffer
        return (torch.stack(idx).to(torch.int32), R), flag

    def run(self, host_batches: Iterable[torch.Tensor]) -> Iterator[Tuple[torch.Tensor, torch.Tensor]]:
        """Yields ``(idx_high int32 [K, n] (cpu), reward fp32 [n] (cpu))`` per host batch ``fp32 [n, L, F]``, in order,
        software-pipelined by one batch; the host batches upload into two reused device staging buffers."""
        return _one_batch_behind(host_batches, self._upload, self._enqueue, self.device)


def low_high(low, high, x, side_stream, own_buffers: bool = True, check: str = "now", rollouts: int = 1):
    """PNLow greedy -> latent -> PNHigh greedy on the rows ``x`` (trainPNHigh.py:131-144).  The two encoders are independent
    (same rows, different weights): PNHigh's is enqueued on ``side_stream`` and runs concurrently with PNLow's whenever the
    batch leaves SMs free (one encoder occupies ceil(n / 128) SMs); the decoders follow on the current stream.
    ``own_buffers``: both actors keep their encodings buffer across calls (``actor.last["enc_out"]`` of a call is then only
    valid until the next call).  The input range flag is read ONCE, after everything is enqueued (no mid-pipeline sync);
    ``check="defer"`` does not read it at all and returns it as a fourth value (device int32 [1] or None) for the caller.
    ``rollouts`` > 1: PNHigh decodes best-of-``rollouts`` (``CombinatorialRL.best_of``: rollout 0 greedy, the others
    sampled, the lowest reward kept) from its one encoder pass; PNLow stays greedy, its latent is what PNHigh consumes.
    Returns (latent, reward, K-list of picks)."""
    from . import ops
    main = torch.cuda.current_stream(x.device)
    if own_buffers:
        for m in (low, high):
            m.actor.own_enc_buffer(x)
    # two streams only while both encoders fit on the machine together (one CTA per 128 rows, 148 SMs).  At a full wave
    # the second encoder's CTAs would interleave with PNLow's decoder and delay it: measured 15.5 ms against 14.5 ms
    # back to back at n = 18,944 (profiles/r02_pn_batch_sweep.jsonl)
    groups = (x.shape[0] + 127) // 128
    concurrent = 2 * groups <= NUM_SMS
    # Column-split encoders (<= 30 groups): a B200 holds 15 of their 8-CTA clusters at a time.  Both networks' encoders run side
    # by side only if together they need at most 15 clusters, so the groups per cluster are chosen for that: 8..14 groups ->
    # two per cluster (<= 7 clusters each, 9.1 us per step instead of two sequential scans at 6.6 us), 15..21 -> three per
    # cluster (<= 7 each, ~12.5 us per step); above that the automatic choice (two per cluster, one encoder after the other).
    g_opt = 0
    if ops.get_option("scan") == -1 and ops.get_option("scan_groups") == 0:
        g_opt = 2 if 8 <= groups <= 14 else (3 if 15 <= groups <= 21 else 0)
    if g_opt:
        ops.set_option("scan_groups", g_opt)              # read by the dispatcher at launch time (host side)
    try:
        if concurrent:
            side_stream.wait_stream(main)                 # x is ready on the main stream; last call's decoders are done
            with torch.cuda.stream(side_stream):
                enc_hi = high.actor.encode(x)
        enc_lo = low.actor.encode(x)
        if not concurrent:
            enc_hi = high.actor.encode(x)
    finally:
        if g_opt:
            ops.set_option("scan_groups", 0)
    deferred = low.actor.defer_range_check
    low.actor.defer_range_check = True
    try:
        _, _, _, _, latent = low(x, None, sample="greedy", training="SL", encoded=enc_lo)
    finally:
        low.actor.defer_range_check = deferred
    if rollouts == 1:
        R, _, _, idx, _ = high(x, None, latent, sample="greedy", training="RL", encoded=enc_hi)
    else:
        R, _, idx, _ = high.best_of(x, None, latent, rollouts=rollouts, encoded=enc_hi)
    flag = low.actor.last["range_flag"]
    if check == "defer":
        return latent, R, idx, flag
    if not deferred:
        low.actor.raise_if_out_of_range(flag)
    return latent, R, idx


# ----------------------------------------------------------------------------- ML -> candidates -> 2PN on the device
def constraint_arrays(nodefeatures, K: int):
    """Per-instance constraint tensors from the raw ``nodefeatures.data`` rows (one-hot(K+1) + 6 floats), as
    ``loadDataPN`` reads them (loadData.py:107-114): local bounds ``[n,K,4]`` = (lo2,hi2,lo3,hi3) of the task node
    of each category, ``used [n,K]``, global bounds ``[n,4]`` of the global-constraint node."""
    import numpy as np
    n = len(nodefeatures)
    local = np.zeros((n, K, 4), dtype=np.float32)
    used = np.zeros((n, K), dtype=np.uint8)
    glob = np.zeros((n, 4), dtype=np.float32)
    for b, inst in enumerate(nodefeatures):
        a = np.asarray(inst, dtype=np.float64)
        kind = np.argmax(a[:, :-6] == 1, axis=1)
        bounds = np.concatenate([a[:, -5:-3], a[:, -2:]], axis=1)
        for t, row in zip(kind, bounds):
            if t == 0:
                glob[b] = row
            else:
                local[b, t - 1] = row
                used[b, t - 1] = 1
    return local, used, glob


def woa_arrays(nodefeatures, K: int):
    """What the ESWOA stage reads from the raw ``nodefeatures.data`` rows, parsed as ``loadDataOther`` parses them
    (gnnpn_sc_b200/WOA.py:541-554), all float64 as the JSON values are:
    ``req_cat int32 [n, K]`` = the category of every task node after the first node, in request-node order (-1 padded),
    ``n_req int32 [n]``, ``local f64 [n, K, 4]`` = (lo_cost, hi_cost, lo_q, hi_q) of the last task node of each category,
    ``glob f64 [n, 4]`` = (lo1, hi1, lo2, hi2) of the last global-constraint node.  A global node after the first node, or
    more tasks than categories (a category requested twice), raise ``ValueError``: ``loadDataOther`` accepts them, but the
    device stage does not take them (``gnnpn_woa_prepare_f64`` flag 8)."""
    import numpy as np
    n = len(nodefeatures)
    req = np.full((n, K), -1, dtype=np.int32)
    n_req = np.zeros(n, dtype=np.int32)
    local = np.zeros((n, K, 4), dtype=np.float64)
    glob = np.zeros((n, 4), dtype=np.float64)
    for b, inst in enumerate(nodefeatures):
        kinds = [node[:-6].index(1) for node in inst]
        for node, kind in zip(inst, kinds):
            vals = node[-5:-3] + node[-2:]
            if node[0] == 1:
                glob[b] = vals
            else:
                local[b, kind - 1] = vals
        tasks = [kind - 1 for kind in kinds[1:]]
        if min(tasks, default=0) < 0 or len(tasks) > K:
            raise ValueError(f"instance {b}: a global node after the first node, or more tasks than categories")
        req[b, :len(tasks)] = tasks
        n_req[b] = len(tasks)
    return req, n_req, local, glob


def service_arrays(serviceFeature, dtype=None):
    """``svc_qos [S,4]`` (last four attributes, loadData.py:40; float32, or ``dtype``) and ``cat_ptr [K+1]`` in
    category-key order."""
    import numpy as np
    keys = sorted(int(k) for k in serviceFeature.keys())
    qos, ptr = [], [0]
    for k in keys:
        rows = np.asarray(serviceFeature[str(k)], dtype=np.float64)[:, -4:]
        qos.append(rows)
        ptr.append(ptr[-1] + len(rows))
    return np.concatenate(qos).astype(dtype or np.float32), np.asarray(ptr, dtype=np.int32)


class ML2PN:
    """The whole inference pipeline of ``main.py <ds> ML+2PN`` on one device, batched over request instances:
    ``Net`` scores (modelML.py:131-176) -> per-category top-N feasible candidates (loadDataPN, loadData.py:99-150,
    ranking order) -> PNLow greedy -> PNHigh greedy (trainPNHigh.py:131-144) -> objective (ML2PN.py:6-12).
    Nothing leaves the GPU between the stages.

    ``woa``: optional ESWOA fine-tuning stage after the objective (the third stage of ``ML2PNWOATest``,
    gnnpn_sc_b200/WOA.py), a dict with ``popSize``, ``MAX_Iter`` and ``reduct`` (0, or 0.55 in the Normal ini
    sections).  PNHigh's picks seed it, as ``WOA.start`` seeds it from ``allActions`` files.

    ``rollouts``: PNHigh decodes best-of-``rollouts`` (``low_high``; 1, the default, is the greedy decode); the best
    rollout's picks are the ones scored and the ones that seed ESWOA."""

    def __init__(self, net, low, high, service_sample, serviceFeature, device=None, woa=None, rollouts: int = 1):
        self.device = torch.device(device if device is not None else "cuda")
        self.net, self.low, self.high = net.eval(), low.eval(), high.eval()
        self.high.actor.check_inputs = False      # same rows as PNLow
        qos, ptr = service_arrays(serviceFeature)
        self.svc_qos = torch.from_numpy(qos).to(self.device)
        self.cat_ptr = torch.from_numpy(ptr).to(self.device)
        self.max_category_size = int((ptr[1:] - ptr[:-1]).max())         # static: no device read per call
        self.K = len(ptr) - 1
        self.N = low.sNumber
        self.rollouts = rollouts
        self.service_enc = net.service_encodings(service_sample)          # static: encoded once
        self._side = torch.cuda.Stream(self.device)
        self._copy = torch.cuda.Stream(self.device)                       # host->device uploads of run()
        self.woa = None
        if woa is not None:
            import numpy as np
            from .WOA import _round5
            self.woa = {"popSize": int(woa["popSize"]), "MAX_Iter": int(woa["MAX_Iter"]),
                        "reduct": float(woa.get("reduct") or 0.0)}
            if not (1 <= self.woa["popSize"] <= 128 and self.K <= 128 and self.woa["MAX_Iter"] >= 0):
                raise ValueError("the device ESWOA stage takes popSize <= 128 and at most 128 categories")
            raw, _ = service_arrays(serviceFeature, dtype=np.float64)
            self.svc_raw = torch.from_numpy(raw).to(self.device)                       # the JSON values
            self.svc_round = torch.from_numpy(_round5(raw)).to(self.device)            # Python round(x, 5)

    def run(self, host_batches):
        """The pipeline from HOST batches: every item is ``(request_batch, local_bounds, used, global_bounds)`` with pinned
        host tensors (``trainML.collate_requests(..., pin=True)``, ``constraint_arrays``), optionally followed by the
        ESWOA stage's ``(req_cat, n_req, local, glob, instance_ids)`` (``woa_arrays``; see ``compose``).  Yields, in order,
        ``(services int32 [n, K] (cpu), objective fp32 [n] (cpu))`` -- plus ``woa_fitness``, ``woa_services`` and
        ``woa_traj`` for items with the ESWOA arrays -- software-pipelined by one batch; every batch is uploaded into fresh
        device tensors.  Instances the ESWOA stage cannot run raise after their batch."""
        from . import ops

        def upload(item, slot):
            rb, lb, us, gb = item[:4]
            with torch.cuda.stream(self._copy):
                dev = type(rb)(x=rb.x.to(self.device, non_blocking=True), edge_index=rb.edge_index.to(self.device, non_blocking=True),
                               batch=rb.batch.to(self.device, non_blocking=True), num_graphs=rb.num_graphs)
                cons = [t.to(self.device, non_blocking=True) for t in (lb, us, gb)]
                woa = [t.to(self.device, non_blocking=True) for t in item[4]] if len(item) > 4 else None
                ev = torch.cuda.Event()
                ev.record(self._copy)
            return dev, cons, woa, ev

        def enqueue(up):
            dev, cons, woa, ev_up = up
            main = torch.cuda.current_stream(self.device)
            main.wait_event(ev_up)
            for t in (dev.x, dev.edge_index, dev.batch, *cons, *(woa or ())):
                t.record_stream(main)                        # allocated on the copy stream, consumed on the main one
            r = self.compose(dev, *cons, defer_check=True, woa=woa)
            res = (r["services"].to(torch.int32), r["objective"])
            if woa is not None:
                res += (r["woa_fitness"], r["woa_services"], r["woa_traj"], r["woa_flags"])
            return res, r["range_flag"]

        def checked(results):
            for res in results:
                if len(res) > 2:
                    ops.raise_if_woa_flagged(res[-1])
                    res = res[:-1]
                yield res

        return checked(_one_batch_behind(host_batches, upload, enqueue, self.device))

    @torch.no_grad()
    def compose(self, request_batch, local_bounds, used, global_bounds, stage_events=None, defer_check: bool = False,
                woa=None):
        """``request_batch``: collated request graphs (x, edge_index, batch) on the device; constraint tensors from
        ``constraint_arrays``.  Returns scores, PN rows, picked service ids per row, PNHigh picks and objective.
        ``stage_events``: optional list that receives five CUDA events recorded on the current stream at the stage
        boundaries (start, scores, candidates, PNLow+PNHigh, objective) -- bench.py's per-stage times -- and two more with
        ``woa`` (ESWOA prepare, search).
        ``woa``: ``(req_cat, n_req, local, glob, instance_ids int64 [n])`` on the device (``woa_arrays`` + the instances'
        numbers, the Philox seed of each, as ``WOA.start`` seeds instance k with k) runs the ESWOA stage after the
        objective (the constructor's ``woa`` configuration) and adds ``woa_fitness f64 [n]``, ``woa_services int32 [n, K]``
        (best composition as service ids by category, -1 where unused), ``woa_traj f64 [n, MAX_Iter]`` and
        ``woa_flags int32 [n]``; instances the stage cannot run raise here, or with ``defer_check`` are left to the
        caller in ``woa_flags`` (``ops.raise_if_woa_flagged``)."""
        from . import ops

        def mark():
            if stage_events is not None:
                ev = torch.cuda.Event(enable_timing=True)
                ev.record()
                stage_events.append(ev)

        mark()
        scores = self.net.score_requests(request_batch, self.service_enc)                     # [B, S]
        mark()
        rows, picked = ops.select_candidates(scores, self.svc_qos, self.cat_ptr, local_bounds, used, global_bounds,
                                             self.N, with_category=False, return_picked=True,
                                             max_category_size=self.max_category_size)          # [B, K*N, 8]
        mark()
        # defer_check: the input range flag is returned (``range_flag``) instead of being read here (one host sync less)
        latent, R, idx, flag = low_high(self.low, self.high, rows, self._side, check="defer", rollouts=self.rollouts)
        if not defer_check:
            self.low.actor.raise_if_out_of_range(flag)
        idx = torch.stack(idx)                                                                # [K, B]
        services = picked.gather(1, idx.t())                                                  # chosen service per task (-1: unused)
        mark()
        viol, obj, _ = ops.pn_reward(rows, idx.to(torch.int32))
        mark()
        out = {"scores": scores, "rows": rows, "picked": picked, "idx_high": idx, "services": services,
               "reward": R, "violations": viol, "objective": obj, "range_flag": flag}
        if woa is not None:
            out.update(self._woa(rows, idx, services, woa, mark))
            if not defer_check:
                ops.raise_if_woa_flagged(out["woa_flags"])
        return out

    def _woa(self, rows, idx, services, woa, mark):
        """ESWOA stage: candidate lists + seed + initial population on the device, then the unchanged search."""
        from . import ops
        if self.woa is None:
            raise ValueError("ML2PN was built without a woa configuration")
        req_cat, n_req, local, glob, inst = woa
        B, K, P = rows.shape[0], self.K, self.woa["popSize"]
        pick = idx.t().long()                                                                  # [B, K]
        seed_rows = rows.gather(1, pick[..., None].expand(B, K, rows.shape[2]))[..., :4].contiguous()
        seeds = (inst.to(torch.int64) & 0x7FFFFFFFFFFFFFFF).contiguous()
        p = ops.woa_prepare(self.svc_raw, self.svc_round, self.cat_ptr, req_cat.to(torch.int32).contiguous(),
                            n_req.to(torch.int32).contiguous(), local.contiguous(), glob.contiguous(), seed_rows,
                            services.to(torch.int32).contiguous(), seeds, P, self.woa["reduct"])
        mark()
        traj = torch.empty(B, self.woa["MAX_Iter"], device=rows.device, dtype=torch.float64)
        ops.woa_search(p["qos"], p["base"], p["size"], p["klen"], glob.contiguous(), p["pops"], p["best_fit"],
                       p["best_ref"], p["best_vec"], seeds, traj)
        mark()
        # best position (local index per list, Python semantics) -> service ids by category
        valid = torch.arange(K, device=rows.device)[None, :] < p["klen"][:, None]
        pos = p["best_vec"].long().remainder(p["size"].long())
        svc = torch.where(valid, p["ids"][p["base"].long() + pos], -1)
        by_cat = torch.full((B, K + 1), -1, device=rows.device, dtype=torch.int32)
        by_cat.scatter_(1, torch.where(valid, p["list_cat"].long(), K), svc)
        return {"woa_fitness": p["best_fit"], "woa_services": by_cat[:, :K].contiguous(), "woa_traj": traj,
                "woa_flags": p["flags"]}
