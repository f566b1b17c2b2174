"""CPU oracle for the pointer-network path  --  TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import this module.  The product path
(``gnnpn_sc_b200``) never imports anything under ``oracle/`` and has no CPU
fallback.

What it is: a functional, state-dict driven restatement in CPU torch (strict
fp32) of the reference's pointer network, following

* ``src/models/modelPN.py:75-123``   Attention (Dot / Bahdanau, C*tanh)
* ``src/models/modelPN.py:165-173``  visited mask
* ``src/models/modelPN.py:175-241``  PointerNet.forward
* ``src/models/modelPN.py:282-306``  CombinatorialRL.forward
* ``src/models/modelPN.py:15-72``    calc / reward

It calls the same torch library operators in the same shapes as the reference
(``torch.lstm``, ``bmm``, ``softmax``, ``max``) so that on one machine it is
bit-identical to the reference; the Python-level per-row loops of the reference
(window mask ``modelPN.py:220-222``) are vectorised unless ``faithful_loops``
is set, which replays them op for op (used for the CPU timing baseline so the
timed work equals what the reference executes).

Pinning: ``oracle/make_golden.py`` runs the *real* reference on the same tensors
and writes its outputs to ``tests/golden/pn_*.npz``; ``tests/test_oracle_pn.py``
checks this restatement against those fixtures, bit for bit.
"""
from __future__ import annotations

import dataclasses
import math
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.nn.functional as F

QOS_AND_CONS = 8   # modelPN.py:10
QOS_NUM = 4        # modelPN.py:11
CONS_NUM = 2       # modelPN.py:12


@dataclasses.dataclass
class PNConfig:
    """Constructor arguments of the reference ``PointerNet`` (modelPN.py:127-139)."""
    hidden_size: int = 256
    seq_len: int = 235
    s_number: int = 5          # candidates per abstract task (window width N)
    s_category: int = 47       # abstract tasks (decode steps K)
    embedding_size: int = 0
    n_glimpses: int = 0
    tanh_exploration: float = 10.0
    use_tanh: bool = True
    attention: str = "Dot"
    alpha: float = 1.0         # modelPN.py:151 (plain tensor ones(1))

    @property
    def in_features(self) -> int:
        return self.embedding_size + QOS_AND_CONS


# --------------------------------------------------------------------------
# deterministic weights (numpy PCG64 -> stable across torch versions)
# --------------------------------------------------------------------------
def make_state_dict(cfg: PNConfig, seed: int, gain: float = 1.0) -> Dict[str, torch.Tensor]:
    """A ``CombinatorialRL.state_dict()``-shaped dict of fp32 tensors.

    Same key set / shapes as the reference modules create (modelPN.py:153-163,
    83-91) and the same U(-1/sqrt(H), 1/sqrt(H)) family of initial values, but
    drawn from numpy so fixtures do not depend on torch's RNG stream.
    ``gain`` multiplies the LSTM matrices ("sharpened" weights, SURVEY 8d cfg 2).
    """
    rng = np.random.default_rng(seed)
    H, Fin = cfg.hidden_size, cfg.in_features
    b = 1.0 / math.sqrt(H)

    def u(*shape, bound=b, g=1.0):
        return torch.from_numpy((rng.uniform(-bound, bound, size=shape) * g).astype(np.float32))

    sd: Dict[str, torch.Tensor] = {}
    sd["actor.decoder_start_input"] = u(H)
    if cfg.embedding_size:
        sd["actor.embedding1.weight"] = torch.from_numpy(
            rng.standard_normal((cfg.s_category, cfg.embedding_size)).astype(np.float32))
    sd["actor.embedding2.weight"] = u(H, Fin, bound=1.0 / math.sqrt(Fin))
    sd["actor.embedding2.bias"] = u(H, bound=1.0 / math.sqrt(Fin))
    for rnn in ("encoder", "decoder"):
        sd[f"actor.{rnn}.weight_ih_l0"] = u(4 * H, H, g=gain)
        sd[f"actor.{rnn}.weight_hh_l0"] = u(4 * H, H, g=gain)
        sd[f"actor.{rnn}.bias_ih_l0"] = u(4 * H)
        sd[f"actor.{rnn}.bias_hh_l0"] = u(4 * H)
    if cfg.attention == "Bahdanau":
        for att in ("pointer", "glimpse"):
            sd[f"actor.{att}.V"] = u(H)
            sd[f"actor.{att}.W_query.weight"] = u(H, H)
            sd[f"actor.{att}.W_query.bias"] = u(H)
            sd[f"actor.{att}.W_ref.weight"] = u(H, H, 1)
            sd[f"actor.{att}.W_ref.bias"] = u(H)
    return sd


# --------------------------------------------------------------------------
# building blocks
# --------------------------------------------------------------------------
def _lstm(sd, name: str, x: torch.Tensor, state=None):
    """``nn.LSTM(H, H, batch_first=True)`` (modelPN.py:157-158) through the same
    ATen entry point the module uses, gate order i,f,g,o, both biases."""
    w = [sd[f"actor.{name}.weight_ih_l0"], sd[f"actor.{name}.weight_hh_l0"],
         sd[f"actor.{name}.bias_ih_l0"], sd[f"actor.{name}.bias_hh_l0"]]
    B = x.shape[0]
    H = w[1].shape[1]
    if state is None:
        z = x.new_zeros(1, B, H)
        state = (z, z.clone())
    out, h, c = torch.lstm(x, state, w, True, 1, 0.0, False, False, True)
    return out, (h, c)


def lstm_cell_f64(w_ih, w_hh, b_ih, b_hh, x, h, c):
    """Manual float64 LSTM cell; analysis anchor only (how far is *anyone* from
    exact arithmetic), not part of the parity definition."""
    g = x.double() @ w_ih.double().T + h.double() @ w_hh.double().T + b_ih.double() + b_hh.double()
    i, f, gg, o = g.chunk(4, dim=-1)
    c2 = torch.sigmoid(f) * c.double() + torch.sigmoid(i) * torch.tanh(gg)
    return torch.sigmoid(o) * torch.tanh(c2), c2


def attention(sd, which: str, cfg: PNConfig, query: torch.Tensor, ref: torch.Tensor,
              use_tanh: bool, C: float):
    """modelPN.py:93-123.  Returns (ref as [B,H,L], logits [B,L])."""
    B, L, _ = ref.shape
    if cfg.attention == "Bahdanau":
        refp = ref.permute(0, 2, 1)
        q = F.linear(query, sd[f"actor.{which}.W_query.weight"], sd[f"actor.{which}.W_query.bias"]).unsqueeze(2)
        refp = F.conv1d(refp, sd[f"actor.{which}.W_ref.weight"], sd[f"actor.{which}.W_ref.bias"])
        v = sd[f"actor.{which}.V"].unsqueeze(0).unsqueeze(0).repeat(B, 1, 1)
        logits = torch.bmm(v, torch.tanh(q.repeat(1, 1, L) + refp)).squeeze(1)
    elif cfg.attention == "Dot":
        logits = torch.bmm(ref, query.unsqueeze(2)).squeeze(2)
        refp = ref.permute(0, 2, 1)
    else:
        raise NotImplementedError(cfg.attention)
    if use_tanh:
        logits = C * torch.tanh(logits)
    return refp, logits


def _visit(logits: torch.Tensor, mask: torch.Tensor, idxs: Optional[torch.Tensor]):
    """modelPN.py:165-173: cumulative visited mask, -inf written in place."""
    m = mask.clone()
    if idxs is not None:
        m[torch.arange(logits.shape[0]), idxs] = 1
        m = m.bool()
        logits[m] = -math.inf
    return logits, m


def embed_inputs(sd, cfg: PNConfig, inputs: torch.Tensor) -> torch.Tensor:
    """modelPN.py:183-190."""
    if cfg.embedding_size:
        cat = inputs[:, :, 0].long()
        e = F.embedding(cat, sd["actor.embedding1.weight"])
        x = torch.cat((e, inputs[:, :, 1:]), 2)
    else:
        x = inputs.clone()
    return F.linear(x, sd["actor.embedding2.weight"], sd["actor.embedding2.bias"])


# --------------------------------------------------------------------------
# PointerNet.forward  (modelPN.py:175-241)
# --------------------------------------------------------------------------
def pointer_forward(sd, cfg: PNConfig, inputs: torch.Tensor,
                    latent: Optional[Sequence[torch.Tensor]] = None,
                    sample: str = "sample",
                    forced_idxs: Optional[Sequence[torch.Tensor]] = None,
                    faithful_loops: bool = False,
                    generator: Optional[torch.Generator] = None,
                    return_internals: bool = False):
    """Returns (prev_probs, prev_idxs, prev_logits): K-lists of [B,L], [B] int64, [B,L].

    ``forced_idxs`` teacher-forces the selection (the returned idxs are still
    the free choice at every step) so a kernel can be compared step by step
    without one flipped pick cascading.
    """
    B, L, _ = inputs.shape
    assert L == cfg.seq_len
    N, K = cfg.s_number, cfg.s_category
    embedded = embed_inputs(sd, cfg, inputs)
    enc_out, (h, c) = _lstm(sd, "encoder", embedded)

    probs_l: List[torch.Tensor] = []
    idxs_l: List[torch.Tensor] = []
    logits_l: List[torch.Tensor] = []
    queries: List[torch.Tensor] = []
    mask = torch.zeros(B, L, dtype=torch.uint8)
    idxs = None
    dec_in = sd["actor.decoder_start_input"].unsqueeze(0).repeat(B, 1)
    rows = torch.arange(B)

    for k in range(K):
        _, (h, c) = _lstm(sd, "decoder", dec_in.unsqueeze(1), (h, c))
        query = h.squeeze(0)
        for _ in range(cfg.n_glimpses):
            refp, gl = attention(sd, "glimpse", cfg, query, enc_out, False, 10.0)
            gl, mask = _visit(gl, mask, idxs)
            query = torch.bmm(refp, F.softmax(gl, dim=1).unsqueeze(2)).squeeze(2)
        queries.append(query)
        _, logits = attention(sd, "pointer", cfg, query, enc_out, cfg.use_tanh, cfg.tanh_exploration)
        logits, mask = _visit(logits, mask, idxs)
        if latent:
            work = logits + cfg.alpha * latent[k]
        else:
            work = logits.clone()
        lo, hi = k * N, (k + 1) * N
        if faithful_loops:              # modelPN.py:220-222, one row at a time
            for p in range(len(work)):
                work[p][:lo] = -np.inf
                work[p][hi:] = -np.inf
        else:
            work[:, :lo] = -math.inf
            work[:, hi:] = -math.inf
        probs = F.softmax(work, dim=1)
        if sample == "greedy":
            _, idxs = torch.max(probs, dim=1)
        else:
            idxs = probs.multinomial(num_samples=1, generator=generator).squeeze(1)
        for old in idxs_l:               # modelPN.py:229-234 (unreachable under the window)
            hit = old.eq(idxs).any() if faithful_loops else bool((old == idxs).any())
            if hit:
                idxs = probs.multinomial(num_samples=1, generator=generator).squeeze(1)
                break
        free_idxs = idxs
        if forced_idxs is not None:
            idxs = forced_idxs[k].long()
        if faithful_loops:
            dec_in = embedded[[i for i in range(B)], idxs.data, :]
        else:
            dec_in = embedded[rows, idxs, :]
        probs_l.append(probs)
        idxs_l.append(free_idxs)
        logits_l.append(logits)
    if return_internals:
        return probs_l, idxs_l, logits_l, {"enc_out": enc_out, "queries": queries, "embedded": embedded}
    return probs_l, idxs_l, logits_l


# --------------------------------------------------------------------------
# CombinatorialRL.forward  (modelPN.py:282-306)
# --------------------------------------------------------------------------
def combinatorial_forward(sd, cfg: PNConfig, inputs: torch.Tensor, labs=None,
                          latent=None, sample: str = "sample", training: str = "RL",
                          level: str = "Low", faithful_loops: bool = False,
                          generator=None, quiet: bool = True):
    B = inputs.shape[0]
    probs, action_idxs, logits = pointer_forward(sd, cfg, inputs, latent, sample,
                                                 faithful_loops=faithful_loops, generator=generator)
    latent_p = list(logits)
    rows = [x for x in range(B)] if faithful_loops else torch.arange(B)
    actions = [inputs[rows, a, :] for a in action_idxs]
    action_probs = [p[rows, a] for p, a in zip(probs, action_idxs)]
    if training == "RL":
        R = reward(actions, labs, cfg.s_category, level=level,
                   embedding_size=cfg.embedding_size, quiet=quiet)
        return R, action_probs, actions, action_idxs, latent_p
    return probs, action_probs, actions, action_idxs, latent_p


# --------------------------------------------------------------------------
# reward / calc  (modelPN.py:15-72), vectorised over the batch in numpy fp32
# --------------------------------------------------------------------------
def composition_objective(actions: np.ndarray, tag: int = 0) -> Tuple[np.ndarray, np.ndarray]:
    """``actions`` fp32 [K,B,F].  Returns (violations int64 [B], objFunc fp32 [B]).

    Restates calc(): fp32 *sequential* products over the K chosen rows for the
    two constrained attributes (np.cumprod on a float32 array), bounds taken
    from the step-0 row (modelPN.py:51-54), strict comparisons, then
    ``(sum(q0)/#(q0>0) + 1 - min(q1)) / 2`` with numpy's float32 pairwise sum.
    """
    a = np.asarray(actions, dtype=np.float32)
    K, B, _ = a.shape
    q = a[:, :, tag:tag + QOS_NUM]                                  # [K,B,4]
    viol = np.zeros(B, dtype=np.int64)
    for i in range(CONS_NUM):
        prod = np.cumprod(q[:, :, 2 + i], axis=0, dtype=np.float32)[-1]      # [B]
        lo = a[0, :, tag + QOS_NUM + 2 * i]
        hi = a[0, :, tag + QOS_NUM + 2 * i + 1]
        viol += ((prod < lo) | (prod > hi)).astype(np.int64)
    n_used = (q[:, :, 0] > 0).sum(axis=0)
    obj = np.empty(B, dtype=np.float32)
    for b in range(B):                      # np.sum on a contiguous fp32 vector: numpy's pairwise order
        s = np.sum(np.ascontiguousarray(q[:, b, 0]))
        # serviceNum is a python int in the reference (modelPN.py:26-28): float32 arithmetic throughout
        obj[b] = (s / int(n_used[b]) + 1 - np.min(q[:, b, 1])) / 2
    return viol, obj


def reward(sample_solution, opt_solutions, s_category: int, level: str = "Low",
           embedding_size: int = 20, quiet: bool = True) -> torch.Tensor:
    """modelPN.py:35-72.  Low: #violations; High: round(#violations + objFunc, 5)."""
    tag = 0 if embedding_size == 0 else 1
    acts = np.stack([t.detach().cpu().numpy() for t in sample_solution]).astype(np.float32)
    viol, obj = composition_objective(acts, tag)
    if level == "Low":
        out = [int(v) for v in viol]
    else:
        out = [round(int(v) + float(o), 5) for v, o in zip(viol, obj)]
    if not quiet:
        print(f"{level}, {sum(1 for v in out if v >= 1)}, {np.average(out)}: ", out)
    return torch.FloatTensor(out)


# --------------------------------------------------------------------------
# convenience: the ML+2PN greedy decode of trainPNHigh.py:131-144
# --------------------------------------------------------------------------
def greedy_low_high(sd_low, sd_high, cfg: PNConfig, inputs: torch.Tensor,
                    faithful_loops: bool = False):
    """latent = Low(greedy, SL); High(greedy, latent).  Returns a dict of stacked results."""
    with torch.no_grad():
        _, _, _, idx_lo, latent = combinatorial_forward(
            sd_low, cfg, inputs, None, None, "greedy", "SL", "Low", faithful_loops)
        probs_hi, aprob_hi, actions, idx_hi, logits_hi = combinatorial_forward(
            sd_high, cfg, inputs, None, latent, "greedy", "SL", "High", faithful_loops)
    return {
        "idx_low": torch.stack(idx_lo), "latent": torch.stack(latent),
        "idx_high": torch.stack(idx_hi), "logits_high": torch.stack(logits_hi),
        "probs_high": torch.stack(probs_hi), "actions": torch.stack(actions),
        "action_probs": torch.stack(aprob_hi),
    }
