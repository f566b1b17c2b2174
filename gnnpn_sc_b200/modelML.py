"""Drop-in replacement for the reference's ``src/models/modelML.py`` on B200.

``Net`` keeps the reference's constructor, ``reset_parameters()``, ``forward(data)`` and ``state_dict``
keys (modelML.py:55-176; PyG 1.7.0 parameter layout for the convolutions: ``nodeConvs.{i}.nn.{0,1,3}.*``,
``nodeConvs.{i}.eps``, ``serviceConvs.{i}.weight [in,out]`` / ``.bias``) without depending on
torch_geometric / torch_scatter.  ``forward`` runs on the sm_100a kernels of ``libgnnpn_b200.so``:

* ``gnnpn_embed_concat_f32``  NodeEncoder table-0 lookup + concat            (modelML.py:133-137,145-149)
* ``gnnpn_csr_build``         edge_index -> CSR; gcn_norm once per static service graph (cached)
* ``gnnpn_spmm_csr_f32``      GIN sum + (1+eps)x, GCN normalised sum + bias + BN + ReLU, scatter-mean
* ``gnnpn_gemm_f32_bias_act`` every Linear / X.W with bias, eval-BatchNorm and ReLU/sigmoid folded in

Inference (``eval()`` / no grad) is entirely on those kernels.  With gradients enabled (``TrainML.train``) the
aggregations, every dense transform and train-mode BatchNorm + ReLU run on the library's kernels too, forward and
backward, wrapped in ``torch.autograd.Function`` (``_Aggregate``, ``_MatmulNT``, ``_BatchNormAct``).
No CPU fallback: CUDA tensors only.
"""
from __future__ import annotations

import math
from typing import Dict, Optional, Tuple

import torch
import torch.nn as nn
import torch.nn.functional as F
from torch.nn import BatchNorm1d, Embedding, Linear, ModuleList, ReLU, Sequential, Sigmoid

from . import ops


# --------------------------------------------------------------------------- CSR cache + autograd aggregation
class _Csr:
    __slots__ = ("rowptr", "col", "val", "n")

    def __init__(self, rowptr, col, val, n):
        self.rowptr, self.col, self.val, self.n = rowptr, col, val, n


def _csr(edge_index: torch.Tensor, weight: Optional[torch.Tensor], n: int, mode: int) -> _Csr:
    rp, col, val = ops.csr_build(edge_index, weight, n, mode)
    return _Csr(rp, col, val, n)


class _Aggregate(torch.autograd.Function):
    """y = A x with A given as destination-major CSR (+ optional (1+eps) self term handled by the caller).
    backward: grad_x = A^T grad_y through the CSR of the transposed graph (built once per graph)."""

    @staticmethod
    def forward(ctx, x, fwd: _Csr, bwd: _Csr):
        ctx.bwd = bwd
        return ops.spmm_csr(fwd.rowptr, fwd.col, fwd.val, x.contiguous(), n_rows=fwd.n)

    @staticmethod
    def backward(ctx, gy):
        b = ctx.bwd
        return ops.spmm_csr(b.rowptr, b.col, b.val, gy.contiguous(), n_rows=b.n), None, None


def _gemm_nt(a: torch.Tensor, b: torch.Tensor, bias=None) -> torch.Tensor:
    """a [M,K] @ b[N,K]^T (+ bias) through ``ops.gemm_bias_act``, which picks the kernel from the shape.  Training keeps
    K % 4 != 0 or N % 16 != 0 on the strict-fp32 FFMA kernel: a tensor-core kernel there would change the gradients' bits."""
    a, b = a.contiguous(), b.contiguous()
    K, N = a.shape[1], b.shape[0]
    return ops.gemm_bias_act(a, b, bias=bias, impl=None if K % 4 == 0 and N % 16 == 0 else "ffma")


class _MatmulNT(torch.autograd.Function):
    """C = A . B^T (+ bias) with every contraction -- forward, dA = dC . B, dB = dC^T . A -- on the library's GEMM
    kernels (the reference trains through torch.nn.Linear / PyG GCNConv's ``x @ weight``, modelML.py:77-104,164-176)."""

    @staticmethod
    def forward(ctx, a, b, bias):
        ctx.save_for_backward(a, b)
        ctx.has_bias = bias is not None
        return _gemm_nt(a.detach(), b.detach(), None if bias is None else bias.detach())

    @staticmethod
    def backward(ctx, dc):
        a, b = ctx.saved_tensors
        dc = dc.contiguous()
        da = _gemm_nt(dc, b.t()) if ctx.needs_input_grad[0] else None                  # [M,N] . [N,K]
        db = _gemm_nt(dc.t(), a.t()) if ctx.needs_input_grad[1] else None             # [N,M] . [M,K]
        dbias = dc.sum(0) if ctx.has_bias and ctx.needs_input_grad[2] else None
        return da, db, dbias


class _BatchNormAct(torch.autograd.Function):
    """Train-mode BatchNorm1d (+ fused ReLU) on ``gnnpn_bn_train_forward_f32`` / ``gnnpn_bn_train_backward_f32``."""

    @staticmethod
    def forward(ctx, y, gamma, beta, bn, relu):
        y = y.contiguous()
        out, mean, rstd = ops.bn_train_forward(y, gamma.detach(), beta.detach(), bn.eps, bn.momentum if bn.momentum is not None else 0.1,
                                               relu, bn.running_mean if bn.track_running_stats else None,
                                               bn.running_var if bn.track_running_stats else None)
        if bn.track_running_stats and bn.num_batches_tracked is not None:
            bn.num_batches_tracked += 1
        ctx.save_for_backward(y, out, gamma, mean, rstd)
        ctx.relu = relu
        return out

    @staticmethod
    def backward(ctx, dout):
        y, out, gamma, mean, rstd = ctx.saved_tensors
        dx, dg, db = ops.bn_train_backward(y, out, dout.contiguous(), gamma.detach(), mean, rstd, ctx.relu)
        return dx, dg, db, None, None


def _linear(x, lin: "Linear"):
    return _MatmulNT.apply(x, lin.weight, lin.bias)


def _bn_act(y, bn: "BatchNorm1d", relu: bool = True):
    return _BatchNormAct.apply(y, bn.weight, bn.bias, bn, relu)


def _pad4(x: torch.Tensor) -> torch.Tensor:
    k = (-x.shape[1]) % 4
    return x if k == 0 else F.pad(x, (0, k))


# --------------------------------------------------------------------------- modules with the reference's names
class NodeEncoder(nn.Module):
    """modelML.py:9-29: nine Embedding(100, C) tables, summed over the input's columns."""

    def __init__(self, hiddenChannels):
        super().__init__()
        self.embeddings = ModuleList([Embedding(100, hiddenChannels) for _ in range(9)])

    def reset_parameters(self):
        for e in self.embeddings:
            e.reset_parameters()

    def forward(self, x):
        if x.dim() == 1:
            x = x.unsqueeze(1)
        out = 0
        for i in range(x.size(1)):
            out = out + self.embeddings[i](x[:, i].long())
        return out


class EdgeEncoder(NodeEncoder):
    """modelML.py:32-52 (never instantiated by the reference; kept for interface parity)."""


class GINConv(nn.Module):
    """PyG 1.7.0 ``GINConv(nn, train_eps=True)``: nn((1+eps)*x_i + sum_{j->i} x_j)."""

    def __init__(self, nn_module: nn.Module, eps: float = 0.0, train_eps: bool = False):
        super().__init__()
        self.nn = nn_module
        self.initial_eps = eps
        if train_eps:
            self.eps = nn.Parameter(torch.tensor([eps]))
        else:
            self.register_buffer("eps", torch.tensor([eps]))

    def reset_parameters(self):
        for m in self.nn:
            if hasattr(m, "reset_parameters"):
                m.reset_parameters()
        self.eps.data.fill_(self.initial_eps)


class GCNConv(nn.Module):
    """PyG 1.7.0 ``GCNConv``: weight [in,out] (glorot), bias [out] (zeros); D^-1/2 (A+I) D^-1/2 (X W) + b."""

    def __init__(self, in_channels: int, out_channels: int):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.weight = nn.Parameter(torch.empty(in_channels, out_channels))
        self.bias = nn.Parameter(torch.empty(out_channels))
        self.reset_parameters()

    def reset_parameters(self):
        a = math.sqrt(6.0 / (self.in_channels + self.out_channels))
        self.weight.data.uniform_(-a, a)
        self.bias.data.zero_()


def _bn_fold(bn: BatchNorm1d) -> Tuple[torch.Tensor, torch.Tensor]:
    scale = bn.weight / torch.sqrt(bn.running_var + bn.eps)
    return scale.contiguous(), (bn.bias - bn.running_mean * scale).contiguous()


class Net(nn.Module):
    def __init__(self, hiddenChannels, outChannels, embeddingChannels, numLayersGIN, numLayersGCN,
                 isServices=True, dropout=0.0):
        super().__init__()
        self.sigmoid = Sigmoid()
        self.numLayersGIN, self.numLayersGCN = numLayersGIN, numLayersGCN
        self.dropout = dropout
        self.outChannels = outChannels
        self.reqAndServiceChannels = embeddingChannels
        self.qosNumber, self.constraintNumber = 4, 2
        self.isService = isServices
        H, E = hiddenChannels, embeddingChannels
        self.nodeEncoder, self.serviceEncoder = NodeEncoder(E), NodeEncoder(E)
        self.nodeConvs, self.nodeBatchNorms = ModuleList(), ModuleList()
        for layer in range(numLayersGIN):
            cin = E + self.constraintNumber * 3 if layer == 0 else H
            mlp = Sequential(Linear(cin, 2 * H), BatchNorm1d(2 * H), ReLU(), Linear(2 * H, H))
            self.nodeConvs.append(GINConv(mlp, train_eps=True))
            self.nodeBatchNorms.append(BatchNorm1d(H))
        self.nodeLin = Linear(H, H)
        self.serviceConvs, self.serviceBatchNorms = ModuleList(), ModuleList()
        for layer in range(numLayersGCN):
            self.serviceConvs.append(GCNConv(E + self.qosNumber if layer == 0 else 2 * H, 2 * H))
            self.serviceBatchNorms.append(BatchNorm1d(2 * H))
        self.serviceLin = Linear(2 * H, H)
        self.noServicesLins = ModuleList(
            [Linear(E + self.qosNumber if layer == 0 else 2 * H, 2 * H) for layer in range(numLayersGCN)])
        self._csr_cache: Dict[tuple, tuple] = {}

    def reset_parameters(self):
        self.nodeEncoder.reset_parameters()
        self.serviceEncoder.reset_parameters()
        for conv, bn in zip(self.nodeConvs, self.nodeBatchNorms):
            conv.reset_parameters()
            bn.reset_parameters()
        self.nodeLin.reset_parameters()
        for conv, bn in zip(self.serviceConvs, self.serviceBatchNorms):
            conv.reset_parameters()
            bn.reset_parameters()
        self.serviceLin.reset_parameters()

    # ---- graph structure helpers -------------------------------------------------------------
    def _cached(self, slot: str, tensors, build):
        """One-entry cache per ``slot`` keyed on the IDENTITY (+ in-place version) of the source tensors.  The entry
        holds references to them, so a freed-and-reused device address can never produce a stale hit (a pointer /
        shape key could: the caching allocator hands the same address to the next batch's ``edge_index``)."""
        hit = self._csr_cache.get(slot)
        if hit is not None and len(hit[0]) == len(tensors) and all(
                (a is b) and (a is None or a._version == v) for (a, v), b in zip(hit[0], tensors)):
            return hit[1]
        value = build()
        self._csr_cache[slot] = ([(t, None if t is None else t._version) for t in tensors], value)
        return value

    def _service_csr(self, data, n_nodes: int, need_transpose: bool):
        """gcn_norm + CSR of the service graph; rebuilt whenever ``data`` carries different tensors."""
        ei, ew = data.edge_index_service, data.edge_attr_service
        entry = self._cached("service", (ei, ew), lambda: {"n": n_nodes, "fwd": _csr(ei, ew, n_nodes, ops.CSR_GCN_NORM),
                                                           "bwd": None})
        if entry["n"] != n_nodes:
            self._csr_cache.pop("service", None)
            return self._service_csr(data, n_nodes, need_transpose)
        if need_transpose and entry["bwd"] is None:
            fwd = entry["fwd"]
            # transpose of the normalised matrix: edge (src=col -> dst=row) becomes (row -> col), same values
            rows = torch.repeat_interleave(torch.arange(n_nodes, device=ei.device),
                                           fwd.rowptr[1:] - fwd.rowptr[:-1])
            t_index = torch.stack([rows, fwd.col.long()])
            entry["bwd"] = _csr(t_index, fwd.val, n_nodes, ops.CSR_PLAIN)
        return entry["fwd"], entry["bwd"]

    @staticmethod
    def _membership_csr(seg: torch.Tensor, n_seg: int) -> _Csr:
        """scatter(reduce='mean') as a CSR over (row -> segment) memberships, rows in index order."""
        idx = torch.stack([torch.arange(seg.numel(), device=seg.device), seg.long()])
        return _csr(idx, None, n_seg, ops.CSR_PLAIN)

    def _request_structure(self, data, n_req: int):
        """(request-graph CSR, request-membership CSR, B): static per collated batch, so built once per ``data``
        (one ``.item()`` sync and two CSR builds per batch instead of per forward)."""
        def build():
            B = getattr(data, "num_graphs", None)           # known on the host for collated batches: no device sync
            if B is None:
                B = int(data.batch.max().item()) + 1 if n_req else 0
            return _csr(data.edge_index, None, n_req, ops.CSR_PLAIN), self._membership_csr(data.batch, B), B
        return self._cached("request", (data.edge_index, data.batch), build)

    def _service_membership(self, S: int, B: int, n_svc: int, device) -> _Csr:
        """serviceBatch = [0..S-1] x B (modelML.py:167-171) as a membership CSR; depends on (S, B, n_svc) only."""
        key = ("svc_memb", S, B, n_svc, str(device))
        hit = self._csr_cache.get(key)
        if hit is None:
            svc_batch = torch.arange(S, device=device).repeat(B)[:n_svc]
            hit = self._membership_csr(svc_batch, S)
            self._csr_cache[key] = hit
        return hit

    def _eps(self, conv) -> float:
        """GIN eps as a host float, synchronised only when the parameter changed."""
        key = ("eps", id(conv))
        hit = self._csr_cache.get(key)
        if hit is None or hit[0] is not conv.eps or hit[1] != conv.eps._version:
            hit = (conv.eps, conv.eps._version, float(conv.eps.detach().item()))
            self._csr_cache[key] = hit
        return hit[2]

    # ---- forward --------------------------------------------------------------------------------
    def forward(self, data):
        if not data.x.is_cuda:
            raise RuntimeError("Net.forward needs CUDA tensors: the B200 path has no CPU fallback")
        if torch.is_grad_enabled() and self.training:
            return self._forward_train(data)
        with torch.no_grad():
            return self._forward_infer(data)

    def _encode_requests(self, data):
        """Request side (modelML.py:133-143,165-166): GIN layers -> nodeLin -> mean over each request graph -> [B, H]."""
        x_raw = data.x.squeeze().float()
        n_req = x_raw.shape[0]
        x = ops.embed_concat(x_raw, self.nodeEncoder.embeddings[0].weight)                 # [n, 28] (26 + pad)
        req, memb, B = self._request_structure(data, n_req)
        for conv, bn in zip(self.nodeConvs, self.nodeBatchNorms):
            agg = ops.spmm_csr(req.rowptr, req.col, None, x, n_rows=n_req, self_scale=1.0 + self._eps(conv))
            lin0, bn0, _, lin1 = conv.nn
            s0, t0 = self._fold(bn0)
            h = ops.gemm_bias_act(agg, _pad_w(lin0.weight, agg.shape[1]), bias=lin0.bias, scale=s0, shift=t0, act="relu")
            s1, t1 = self._fold(bn)
            x = ops.gemm_bias_act(h, lin1.weight, bias=lin1.bias, scale=s1, shift=t1, act="relu")
        x = ops.gemm_bias_act(x, self.nodeLin.weight, bias=self.nodeLin.bias)
        return ops.spmm_csr(memb.rowptr, memb.col, None, x, n_rows=B, mean=True), B        # [B, H]

    def _encode_service_nodes(self, data):
        """Service side (modelML.py:145-164): GCN layers (or the Linear stand-ins) -> serviceLin -> [n_svc, H]."""
        xs_raw = data.x_service.squeeze().float()
        n_svc = xs_raw.shape[0]
        xs = ops.embed_concat(xs_raw, self.serviceEncoder.embeddings[0].weight)            # [B*S, 24]
        if self.isService:
            svc, _ = self._service_csr(data, n_svc, need_transpose=False)
        for i in range(self.numLayersGCN):
            s, t = self._fold(self.serviceBatchNorms[i])
            if self.isService:
                conv = self.serviceConvs[i]
                xw = ops.gemm_bias_act(xs, _pad_w(conv.weight.t(), xs.shape[1]))
                xs = ops.spmm_csr(svc.rowptr, svc.col, svc.val, xw, n_rows=n_svc, bias=conv.bias, scale=s, shift=t,
                                  act="relu")
            else:
                lin = self.noServicesLins[i]
                xs = ops.gemm_bias_act(xs, _pad_w(lin.weight, xs.shape[1]), bias=lin.bias, scale=s, shift=t, act="relu")
        return ops.gemm_bias_act(xs, self.serviceLin.weight, bias=self.serviceLin.bias), n_svc

    def _forward_infer(self, data):
        x, B = self._encode_requests(data)
        xs, n_svc = self._encode_service_nodes(data)
        S = self.outChannels
        memb_s = self._service_membership(S, B, n_svc, xs.device)                          # modelML.py:167-171
        xs = ops.spmm_csr(memb_s.rowptr, memb_s.col, None, xs, n_rows=S, mean=True)        # [S, H]
        return ops.gemm_bias_act(x, xs, act="sigmoid")                                     # sigmoid(x @ xs^T)

    # ---- batched inference with the (static) service side computed once ------------------------------------
    @torch.no_grad()
    def service_encodings(self, sample):
        """[S, H] service encodings from ONE copy of the service graph (``sample.x_service [S,5]``,
        ``edge_index_service``, ``edge_attr_service``).  The reference embeds the whole service graph in every
        sample and re-encodes B copies per batch (trainML.py:91-114); with an S-offset collation all copies are
        identical, so encoding one copy and reusing it for every request gives the same scores."""
        xs, n_svc = self._encode_service_nodes(sample)
        assert n_svc == self.outChannels
        return xs

    @torch.no_grad()
    def score_requests(self, data, service_enc):
        """sigmoid(x_req . service_enc^T) ``[B, S]`` for a collated batch of request graphs (``data.x``,
        ``data.edge_index``, ``data.batch``) against cached ``service_encodings``."""
        x, _ = self._encode_requests(data)
        return ops.gemm_bias_act(x, service_enc, act="sigmoid", pad_ld=True)       # [B, S] view of rows padded to 8 floats

    def _fold(self, bn: BatchNorm1d):
        if self.training:
            raise RuntimeError("the fused inference path needs eval-mode BatchNorm (call .eval())")
        return _bn_fold(bn)

    def _forward_train(self, data):
        """Autograd path (TrainML.train, trainML.py:34-47) on the library's kernels, forward AND backward: CSR
        aggregations (``_Aggregate``), every dense transform (``_MatmulNT`` -> gnnpn_gemm_f32_bias_act) and train-mode
        BatchNorm + ReLU (``_BatchNormAct`` -> gnnpn_bn_train_*).  Embedding lookups, the segment mean, the sigmoid and
        the loss stay element-wise / indexing torch ops."""
        x_raw = data.x.squeeze().float()
        n_req = x_raw.shape[0]
        x = torch.cat((self.nodeEncoder(x_raw[:, 0].view(-1, 1).long()), x_raw[:, 1:]), -1)
        req = _csr(data.edge_index, None, n_req, ops.CSR_PLAIN)
        req_t = _csr(data.edge_index.flip(0), None, n_req, ops.CSR_PLAIN)
        for conv, bn in zip(self.nodeConvs, self.nodeBatchNorms):
            xp = _pad4(x)
            agg = _Aggregate.apply(xp, req, req_t)[:, : x.shape[1]] + (1 + conv.eps) * x
            lin0, bn0, _, lin1 = conv.nn                                    # Linear, BatchNorm1d, ReLU, Linear
            h = _bn_act(_linear(agg, lin0), bn0, relu=True)
            x = F.dropout(_bn_act(_linear(h, lin1), bn, relu=True), self.dropout, training=True)
        xs_raw = data.x_service.squeeze().float()
        n_svc = xs_raw.shape[0]
        xs = torch.cat((self.serviceEncoder(xs_raw[:, 0].view(-1, 1).long()), xs_raw[:, 1:]), -1)
        if self.isService:
            svc, svc_t = self._service_csr(data, n_svc, need_transpose=True)
        for i in range(self.numLayersGCN):
            if self.isService:
                conv = self.serviceConvs[i]
                xs = _Aggregate.apply(_MatmulNT.apply(xs, conv.weight.t(), None), svc, svc_t) + conv.bias
            else:
                xs = _linear(xs, self.noServicesLins[i])
            xs = F.dropout(_bn_act(xs, self.serviceBatchNorms[i], relu=True), self.dropout, training=True)
        xs = _linear(xs, self.serviceLin)
        x = _linear(x, self.nodeLin)
        B = int(data.batch.max().item()) + 1
        ones = torch.ones(n_req, device=x.device)
        x = torch.zeros(B, x.shape[1], device=x.device).index_add_(0, data.batch, x) / \
            torch.zeros(B, device=x.device).index_add_(0, data.batch, ones).clamp(min=1).view(-1, 1)
        S = self.outChannels
        xs = xs.view(-1, S, xs.shape[1]).mean(0) if n_svc % S == 0 else xs
        return self.sigmoid(_MatmulNT.apply(x, xs, None))


def _pad_w(w: torch.Tensor, k: int) -> torch.Tensor:
    """nn.Linear-layout weight [N,K'] zero-padded along K to the (multiple-of-4) width of its padded input."""
    w = w.detach()
    if w.shape[1] == k:
        return w.contiguous()
    return F.pad(w, (0, k - w.shape[1])).contiguous()
