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


class GreedyLowHigh:
    def __init__(self, low, high, device=None):
        self.low, self.high = low.eval(), high.eval()
        self.high.actor.check_inputs = False      # PNHigh decodes the rows PNLow has just range-checked
        self.device = torch.device(device if device is not None else "cuda")
        if self.device.type != "cuda":
            raise RuntimeError("GreedyLowHigh needs a CUDA device: the B200 path has no CPU fallback")
        self._copy = torch.cuda.Stream(self.device)
        self._side = torch.cuda.Stream(self.device)   # PNHigh's encoder runs here, next to PNLow's on the main stream
        self._stage = [None, None]            # device staging buffers (double buffer)
        self._ready = [torch.cuda.Event(), torch.cuda.Event()]
        self._consumed = [None, None]
        self._out = [None, None]              # pinned result buffers (double buffer)

    def _upload(self, slot: int, x_host: torch.Tensor) -> None:
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

    @torch.no_grad()
    def run(self, host_batches: Iterable[torch.Tensor]) -> Iterator[Tuple[torch.Tensor, torch.Tensor]]:
        """Yields ``(idx_high int32 [K, n] (cpu), reward fp32 [n] (cpu))`` per host batch ``fp32 [n, L, F]``, in order.
        Software-pipelined by one batch: the kernels of batch i+1 are enqueued before the host waits for the results of
        batch i (asynchronous device->host copies into pinned buffers + an event), so the GPU never idles while the host
        prepares the next launches; the input range flag travels with the results (no mid-batch sync)."""
        it = iter(host_batches)
        nxt = next(it, None)
        slot = 0
        if nxt is not None:
            self._upload(slot, nxt)
        main = torch.cuda.current_stream(self.device)
        pending = None                                    # (pinned idx, pinned reward, pinned flag, event) of the previous batch

        def finish(p):
            idx_pin, r_pin, flag_pin, ev = p
            ev.synchronize()
            if flag_pin is not None and int(flag_pin[0]):
                self.low.actor.raise_if_out_of_range(flag_pin)
            return idx_pin.clone(), r_pin.clone()         # the pinned buffers are reused two batches later

        while nxt is not None:
            cur_slot = slot
            nxt = next(it, None)
            if nxt is not None:                           # upload of the next batch overlaps this batch's kernels
                self._upload(cur_slot ^ 1, nxt)
            main.wait_event(self._ready[cur_slot])
            x = self._stage[cur_slot]
            latent, R, idx, flag = low_high(self.low, self.high, x, self._side, check="defer")
            idx32 = torch.stack(idx).to(torch.int32)
            out = self._out[cur_slot]
            if out is None or out[0].shape != idx32.shape:
                out = self._out[cur_slot] = (torch.empty(idx32.shape, dtype=torch.int32).pin_memory(),
                                             torch.empty(R.shape, dtype=torch.float32).pin_memory(),
                                             torch.zeros(1, dtype=torch.int32).pin_memory())
            out[0].copy_(idx32, non_blocking=True)
            out[1].copy_(R, non_blocking=True)
            if flag is not None:
                out[2].copy_(flag, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(main)
            self._consumed[cur_slot] = ev
            if pending is not None:
                yield finish(pending)
            pending = (out[0], out[1], out[2] if flag is not None else None, ev)
            slot = cur_slot ^ 1
        if pending is not None:
            yield finish(pending)


def _own_enc_buffer(actor, n: int, L: int, F: int, device):
    """Gives ``actor`` a persistent encodings buffer for batches of n rows (kept across calls: a 4.6 GB block per network
    at n = 18,944 that would otherwise go through the caching allocator -- per stream, with deferred frees for buffers
    that crossed streams -- on every call).  A caller-set larger buffer is left alone."""
    from . import ops
    if actor.embedding_size != 0 or actor.impl == "ffma" or actor._anyh():
        return
    need = ops.enc_out_floats(n, L, actor.hidden_size, actor.enc_layout(n, F))
    if actor.enc_buffer is None or actor.enc_buffer.numel() < need:
        actor.enc_buffer = None                           # release the old block before asking for the larger one
        actor.enc_buffer = torch.empty(need, device=device, dtype=torch.float32)


def low_high(low, high, x, side_stream, own_buffers: bool = True, check: str = "now"):
    """PNLow greedy -> latent -> PNHigh greedy on the rows ``x`` (trainPNHigh.py:131-144).  The two encoders are independent
    (same rows, different weights): PNHigh's is enqueued on ``side_stream`` and runs concurrently with PNLow's whenever the
    batch leaves SMs free (one encoder occupies ceil(n / 128) SMs); the decoders follow on the current stream.
    ``own_buffers``: both actors keep their encodings buffer across calls (``actor.last["enc_out"]`` of a call is then only
    valid until the next call).  The input range flag is read ONCE, after everything is enqueued (no mid-pipeline sync);
    ``check="defer"`` does not read it at all and returns it as a fourth value (device int32 [1] or None) for the caller.
    Returns (latent, reward, K-list of picks)."""
    from . import ops
    main = torch.cuda.current_stream(x.device)
    if own_buffers:
        for m in (low, high):
            _own_enc_buffer(m.actor, x.shape[0], x.shape[1], x.shape[2], x.device)
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
    R, _, _, idx, _ = high(x, None, latent, sample="greedy", training="RL", encoded=enc_hi)
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


def service_arrays(serviceFeature):
    """``svc_qos [S,4]`` (last four attributes, loadData.py:40) and ``cat_ptr [K+1]`` in category-key order."""
    import numpy as np
    keys = sorted(int(k) for k in serviceFeature.keys())
    qos, ptr = [], [0]
    for k in keys:
        rows = np.asarray(serviceFeature[str(k)], dtype=np.float64)[:, -4:]
        qos.append(rows)
        ptr.append(ptr[-1] + len(rows))
    return np.concatenate(qos).astype(np.float32), np.asarray(ptr, dtype=np.int32)


class ML2PN:
    """The whole inference pipeline of ``main.py <ds> ML+2PN`` on one device, batched over request instances:
    ``Net`` scores (modelML.py:131-176) -> per-category top-N feasible candidates (loadDataPN, loadData.py:99-150,
    ranking order) -> PNLow greedy -> PNHigh greedy (trainPNHigh.py:131-144) -> objective (ML2PN.py:6-12).
    Nothing leaves the GPU between the stages."""

    def __init__(self, net, low, high, service_sample, serviceFeature, device=None):
        self.device = torch.device(device if device is not None else "cuda")
        self.net, self.low, self.high = net.eval(), low.eval(), high.eval()
        self.high.actor.check_inputs = False      # same rows as PNLow
        qos, ptr = service_arrays(serviceFeature)
        self.svc_qos = torch.from_numpy(qos).to(self.device)
        self.cat_ptr = torch.from_numpy(ptr).to(self.device)
        self.max_category_size = int((ptr[1:] - ptr[:-1]).max())         # static: no device read per call
        self.K = len(ptr) - 1
        self.N = low.sNumber
        self.service_enc = net.service_encodings(service_sample)          # static: encoded once
        self._side = torch.cuda.Stream(self.device)
        self._copy = torch.cuda.Stream(self.device)                       # host->device uploads of run()

    @torch.no_grad()
    def run(self, host_batches):
        """The pipeline from HOST batches: every item is ``(request_batch, local_bounds, used, global_bounds)`` with pinned
        host tensors (``trainML.collate_requests(..., pin=True)``, ``constraint_arrays``).  Yields, in order,
        ``(services int32 [n, K] (cpu), objective fp32 [n] (cpu))``.  The upload of batch i+1 runs on a copy stream under the
        kernels of batch i, and the results of batch i are waited for only after batch i+1 has been enqueued."""
        main = torch.cuda.current_stream(self.device)

        def upload(item):
            rb, lb, us, gb = item
            with torch.cuda.stream(self._copy):
                dev = type(rb)(x=rb.x.to(self.device, non_blocking=True), edge_index=rb.edge_index.to(self.device, non_blocking=True),
                               batch=rb.batch.to(self.device, non_blocking=True), num_graphs=rb.num_graphs)
                cons = [t.to(self.device, non_blocking=True) for t in (lb, us, gb)]
                ev = torch.cuda.Event()
                ev.record(self._copy)
            return dev, cons, ev

        def finish(p):
            svc_pin, obj_pin, flag_pin, ev, keep = p
            ev.synchronize()
            if flag_pin is not None and int(flag_pin[0]):
                self.low.actor.raise_if_out_of_range(flag_pin)
            return svc_pin.clone(), obj_pin.clone()

        it = iter(host_batches)
        nxt = next(it, None)
        up = upload(nxt) if nxt is not None else None
        pending, out, slot = None, [None, None], 0
        while up is not None:
            dev, cons, ev_up = up
            nxt = next(it, None)
            up = upload(nxt) if nxt is not None else None    # next upload overlaps this batch's kernels
            main.wait_event(ev_up)
            for t in (dev.x, dev.edge_index, dev.batch, *cons):
                t.record_stream(main)                        # allocated on the copy stream, consumed on the main one
            r = self.compose(dev, *cons, defer_check=True)
            svc, obj, flag = r["services"].to(torch.int32), r["objective"], r["range_flag"]
            if out[slot] is None or out[slot][0].shape != svc.shape:
                out[slot] = (torch.empty(svc.shape, dtype=torch.int32).pin_memory(),
                             torch.empty(obj.shape, dtype=torch.float32).pin_memory(),
                             torch.zeros(1, dtype=torch.int32).pin_memory())
            out[slot][0].copy_(svc, non_blocking=True)
            out[slot][1].copy_(obj, non_blocking=True)
            if flag is not None:
                out[slot][2].copy_(flag, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(main)
            if pending is not None:
                yield finish(pending)
            pending = (out[slot][0], out[slot][1], out[slot][2] if flag is not None else None, ev, (dev, cons))
            slot ^= 1
        if pending is not None:
            yield finish(pending)

    @torch.no_grad()
    def compose(self, request_batch, local_bounds, used, global_bounds, stage_events=None, defer_check: bool = False):
        """``request_batch``: collated request graphs (x, edge_index, batch) on the device; constraint tensors from
        ``constraint_arrays``.  Returns scores, PN rows, picked service ids per row, PNHigh picks and objective.
        ``stage_events``: optional list that receives five CUDA events recorded on the current stream at the stage
        boundaries (start, scores, candidates, PNLow+PNHigh, objective) -- bench.py's per-stage times."""
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
        latent, R, idx, flag = low_high(self.low, self.high, rows, self._side, check="defer")
        if not defer_check:
            self.low.actor.raise_if_out_of_range(flag)
        idx = torch.stack(idx)                                                                # [K, B]
        services = picked.gather(1, idx.t())                                                  # chosen service per task (-1: unused)
        mark()
        viol, obj, _ = ops.pn_reward(rows, idx.to(torch.int32))
        mark()
        return {"scores": scores, "rows": rows, "picked": picked, "idx_high": idx, "services": services,
                "reward": R, "violations": viol, "objective": obj, "range_flag": flag}
