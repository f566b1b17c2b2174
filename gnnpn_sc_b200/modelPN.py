"""Drop-in replacement for the reference's ``src/models/modelPN.py`` on B200.

Same public names, constructor signatures, ``forward`` signatures, return tuples
and ``state_dict`` keys as the reference (modelPN.py:75-306, SURVEY 8b) -- the
trainers and ``main.py`` call it unchanged -- but ``forward`` runs the
hand-written sm_100a kernels of ``libgnnpn_b200.so``:

* encoder  : ``gnnpn_lstm_encode_f32``  (embedding2 folded into the LSTM input weights)
* decode   : ``gnnpn_pn_decode_greedy_f32`` (LSTM cell + window logits + C*tanh + latent +
             mask + softmax + first-max pick + next-input gather, K steps, whole batch)
* reward   : ``gnnpn_pn_reward_f32``

The reference returns K-long python lists of dense ``[B, L]`` tensors
(``prev_probs``, ``prev_logits``).  Only the window slice ``[k*N,(k+1)*N)`` of
step k ever influences a pick (modelPN.py:220-222), so the kernels keep the
compact ``[B, L]`` "window" form and the lists handed back are *lazy*: indexing
one materialises the reference's dense tensors (``gnnpn_pn_full_logits_f32``),
while passing one on as ``latent`` to the next network stays compact.

No CPU fallback: CUDA tensors only, and a missing extension raises.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Optional, Sequence

import torch
import torch.nn as nn

from . import ops

qosandcons = 8      # modelPN.py:10-12
qosNum = 4
consNum = 2

VERBOSE_REWARD = False     # the reference prints every batch's reward list (modelPN.py:67)


# --------------------------------------------------------------------------- lazy step lists
class _StepList(Sequence):
    """K-long, read-only, list-like view whose dense ``[K, B, L]`` backing tensor is built on first use."""

    def __init__(self, K: int, make_dense):
        self._K = K
        self._make = make_dense
        self._dense: Optional[torch.Tensor] = None

    def dense(self) -> torch.Tensor:
        if self._dense is None:
            self._dense = self._make()
        return self._dense

    def __len__(self):
        return self._K

    def __bool__(self):
        return self._K > 0

    def __getitem__(self, k):
        if isinstance(k, slice):
            return [self.dense()[i] for i in range(*k.indices(self._K))]
        if k < 0:
            k += self._K
        if not 0 <= k < self._K:
            raise IndexError(k)
        return self.dense()[k]

    def copy(self):
        return self


class WindowLogits(_StepList):
    """``prev_logits`` / ``latent_p``.  ``.window`` is the compact ``[B, L]`` tensor the decode kernel consumes."""

    def __init__(self, K, window: torch.Tensor, make_dense):
        super().__init__(K, make_dense)
        self.window = window


class _Last(dict):
    """Device-side results of the most recent forward.  ``["enc_out"]`` is the reference's ``[B, L, H]`` tensor
    (modelPN.py:191); when the kernels kept the encodings in the blocked layout it is converted on first use."""

    def __getitem__(self, key):
        if key == "enc_out" and not dict.__contains__(self, "enc_out"):
            B, L, H = dict.__getitem__(self, "enc_shape")
            dict.__setitem__(self, "enc_out", ops.enc_to_rowmajor(dict.__getitem__(self, "enc_buf"), B, L, H))
        if key in ("dec_h", "dec_q") and not dict.__contains__(self, key):
            # the fused decoder does not write its hidden states: replay the decode teacher-forced on the same picks
            # with the output enabled (same kernels, same arithmetic -> the states the picks were made from)
            dec_h = dict.__getitem__(self, "replay_dec_h")()
            dict.__setitem__(self, "dec_h", dec_h)
            dict.__setitem__(self, "dec_q", dec_h)
        return dict.__getitem__(self, key)


@dataclass
class _Encoded:
    """The handle ``PointerNet.encode`` returns for ``forward(..., encoded=handle)``.  ``path`` is the decode path of the
    batch (``PointerNet._path``), or "train" when the decode already ran with the BPTT's saves (``saves``)."""
    path: str
    x: torch.Tensor                         # the kernel input rows
    ws: Optional[torch.Tensor]              # tensor-core scratch (None: FFMA kernels)
    layout: int                             # ops.ENC_ROWMAJOR | ops.ENC_BLOCKED128
    enc_out: torch.Tensor
    c: Optional[torch.Tensor]               # encoder cell state, where the decoder starts
    range_flag: Optional[torch.Tensor]
    stream: torch.cuda.Stream               # the stream the encoder was enqueued on
    saves: Optional[dict] = None            # path == "train": ops.pn_train_forward's saves


def _window_of(latent, K: int, N: int) -> torch.Tensor:
    """Compact ``[B, L]`` latent from whatever the caller passed (our lazy list or the reference's dense list)."""
    if isinstance(latent, WindowLogits):
        return latent.window
    dense = torch.stack([t for t in latent])                       # [K, B, L]
    Kk, B, L = dense.shape
    assert Kk == K and L == K * N
    return dense.view(K, B, K, N).diagonal(dim1=0, dim2=2).permute(0, 2, 1).reshape(B, L).contiguous()


# --------------------------------------------------------------------------- reward
def reward(sample_solution, optSolutions, sCategory, USE_CUDA=False, level="Low", embedding_size=20):
    """modelPN.py:35-72 on the GPU: ``sample_solution`` is the K-list of chosen rows ``[B, F]``.

    Low -> number of violated global constraints; High -> round(violations + objFunc, 5).
    """
    acts = sample_solution if torch.is_tensor(sample_solution) else torch.stack(list(sample_solution))
    K, B, _ = acts.shape
    rows = acts.permute(1, 0, 2).contiguous()                      # [B, K, F]: pick k is row k
    idx = torch.arange(K, device=rows.device, dtype=torch.int32).view(K, 1).expand(K, B).contiguous()
    viol, _obj, rew = ops.pn_reward(rows, idx, tag=0 if embedding_size == 0 else 1)
    out = viol.float() if level == "Low" else rew
    if VERBOSE_REWARD:
        lst = out.tolist()
        print(f"{level}, {sum(1 for v in lst if v >= 1)}, {sum(lst) / max(len(lst), 1)}: ", lst)
    return out if USE_CUDA else out.cpu()


# --------------------------------------------------------------------------- Attention
class Attention(nn.Module):
    """modelPN.py:75-123.  Parameters exist exactly as in the reference (Bahdanau only)."""

    def __init__(self, hidden_size, use_tanh=False, C=10, name='Bahdanau', use_cuda=True):
        super().__init__()
        self.use_tanh = use_tanh
        self.C = C
        self.name = name
        if name == 'Bahdanau':
            self.W_query = nn.Linear(hidden_size, hidden_size)
            self.W_ref = nn.Conv1d(hidden_size, hidden_size, 1, 1)
            bound = 1.0 / math.sqrt(hidden_size)
            self.V = nn.Parameter(torch.empty(hidden_size).uniform_(-bound, bound))

    def block(self) -> torch.Tensor:
        """Bahdanau parameters packed for the kernels (``gnnpn_pn_att_block_floats`` layout)."""
        return ops.att_block(self.W_query.weight, self.W_query.bias, self.W_ref.weight, self.W_ref.bias, self.V)

    def forward(self, query, ref):
        """query [B,H], ref [B,L,H] -> (ref as [B,H,L] (Bahdanau: W_ref(ref)), logits [B,L])  (modelPN.py:93-123)."""
        B, L, H = ref.shape
        refc = ref.detach().float().contiguous()
        q = query.detach().float().contiguous()
        none_picked = torch.zeros(1, B, device=ref.device, dtype=torch.int32)
        if self.name == 'Dot':
            if H != 256:                                       # any-hidden-size kernels (strict fp32)
                logits = ops.pn_full_logits_anyh(refc, q.view(B, 1, H), none_picked, bool(self.use_tanh), float(self.C))[0]
            else:
                logits = ops.pn_full_logits(refc, q.view(B, 1, H), none_picked, "Dot", None, bool(self.use_tanh),
                                            float(self.C))[0]
            return ref.permute(0, 2, 1), logits
        if self.name != 'Bahdanau':
            raise NotImplementedError(self.name)
        blk = self.block()
        E = ops.pn_ref_transform(refc, blk)
        qw = ops.pn_query_transform(q, blk)
        logits = ops.pn_full_logits_bahdanau(E, qw.view(B, 1, H), blk, none_picked, bool(self.use_tanh), float(self.C))[0]
        return E.permute(0, 2, 1), logits

    def torch_rows(self, query, rows):
        """Differentiable torch evaluation on a subset of positions: rows [B,l,H] -> (ref' [B,l,H], logits [B,l])."""
        if self.name == 'Dot':
            logits = torch.bmm(rows, query.unsqueeze(2)).squeeze(2)
            refp = rows
        else:
            refp = torch.nn.functional.linear(rows, self.W_ref.weight.squeeze(2), self.W_ref.bias)
            logits = torch.tanh(self.W_query(query).unsqueeze(1) + refp) @ self.V
        if self.use_tanh:
            logits = self.C * torch.tanh(logits)
        return refp, logits


# --------------------------------------------------------------------------- PointerNet
class PointerNet(nn.Module):
    """modelPN.py:126-241."""

    def __init__(self, embedding_size, hidden_size, seq_len, n_glimpses, tanh_exploration, use_tanh,
                 attention, sNumber, sCategory, use_cuda=True, level="low", mask=False):
        super().__init__()
        self.embedding_size = embedding_size
        self.hidden_size = hidden_size
        self.n_glimpses = n_glimpses
        self.seq_len = seq_len
        self.use_cuda = use_cuda
        self.level = level
        self.serNumber = sNumber
        self.serCategory = sCategory
        self.alpha = torch.ones(1)                # plain tensor, not in state_dict (modelPN.py:151)
        self.mask = mask
        if embedding_size != 0:
            self.embedding1 = nn.Embedding(sCategory, embedding_size)
        self.embedding2 = nn.Linear(embedding_size + qosandcons, hidden_size)
        self.encoder = nn.LSTM(hidden_size, hidden_size, batch_first=True)
        self.decoder = nn.LSTM(hidden_size, hidden_size, batch_first=True)
        self.pointer = Attention(hidden_size, use_tanh=use_tanh, C=tanh_exploration, name=attention, use_cuda=use_cuda)
        self.glimpse = Attention(hidden_size, use_tanh=False, name=attention, use_cuda=use_cuda)
        bound = 1.0 / math.sqrt(hidden_size)
        self.decoder_start_input = nn.Parameter(torch.empty(hidden_size).uniform_(-bound, bound))
        self._weights_key = None
        self._weights_cache = None
        self.last = None                          # device-side results of the most recent forward
        self.impl = None                          # None -> ops.DEFAULT_IMPL ("tc"); "ffma" = strict-fp32 kernels
        self.generator = None                     # optional torch.Generator (cuda) for sample="sample"
        self.force_general = False                # route a fast-path configuration through the general kernels (tests)
        self.check_inputs = True                  # range-check the raw rows of every batch (one tiny kernel + one sync)
        self.enc_buffer = None                    # optional caller-owned encodings buffer (reused when large enough)
        self.defer_range_check = False            # True: forward leaves the range flag in ``last["range_flag"]`` (no sync);
                                                  # the caller reads it with ``raise_if_out_of_range`` when convenient
        self.replay_impl = "own"                  # REINFORCE gradient: "own" = library kernels (fast configuration), "torch"
        self._train_saves = None                  # (saves, inputs, latent window) of a training-mode forward, consumed by the replay
        self.last_rollouts = None                 # (encoded handle, latent window) of the most recent decode_rollouts

    # -- the kernels' weights are a cache over the parameters; rebuilt when any of them changes
    def _weights(self):
        """(encoder, decoder) weights in the form the kernels of this hidden size take: the packed LSTM blocks
        (``ops.pack_lstm``) for H = 256, else the folded ``(w_cat, bias, bias0)`` triples of the any-hidden-size kernels
        (``ops.anyh_fold``; the encoder's bias0 is None)."""
        ps = [self.embedding2.weight, self.embedding2.bias, self.decoder_start_input]
        for rnn in (self.encoder, self.decoder):
            ps += [rnn.weight_ih_l0, rnn.weight_hh_l0, rnn.bias_ih_l0, rnn.bias_hh_l0]
        key = tuple((p.data_ptr(), p._version) for p in ps)
        if key != self._weights_key:
            make = ops.pack_lstm if self.hidden_size == 256 else ops.anyh_fold
            with torch.no_grad():
                e, d = self.encoder, self.decoder
                we, be = self.embedding2.weight, self.embedding2.bias
                enc = make(e.weight_ih_l0, e.weight_hh_l0, e.bias_ih_l0, e.bias_hh_l0, we, be, None)
                dec = make(d.weight_ih_l0, d.weight_hh_l0, d.bias_ih_l0, d.bias_hh_l0, we, be, self.decoder_start_input)
            self._weights_cache, self._weights_key = (enc, dec), key
        return self._weights_cache

    def _packed_weights(self):
        """(encoder, decoder) packed LSTM blocks of the hidden_size = 256 kernels."""
        assert self.hidden_size == 256, "packed LSTM blocks exist for hidden_size = 256 only"
        return self._weights()

    @property
    def _impl(self) -> str:
        """``impl`` resolved: "tc" (tensor-core recurrence, the default) or "ffma" (strict-fp32 kernels)."""
        return self.impl or ops.DEFAULT_IMPL

    def _kernel_inputs(self, inputs):
        """Raw rows the LSTM kernels consume: with a category embedding (modelPN.py:183-188) column 0 is replaced by
        its ``embedding1`` row (``gnnpn_embed_concat_f32``), giving 20 + 8 = 28 columns."""
        x = inputs.detach().float().contiguous()
        if self.embedding_size == 0:
            return x
        B, L, C = x.shape
        return ops.embed_concat(x.view(B * L, C), self.embedding1.weight.detach()).view(B, L, -1)

    def _path(self, F: int) -> str:
        """Decode path of a batch of F kernel input columns: "anyh" for a hidden size other than the shipped 256 (the
        strict-fp32 any-hidden-size kernels, ``gnnpn_*_anyh_f32``), "fast" for the fused / scan kernels (Dot attention,
        no glimpses, no category embedding, at most 32 candidates per window and 8 columns), else "general"
        (``gnnpn_pn_decode_general_f32``; ``force_general`` sends a fast configuration there too)."""
        if self.hidden_size != 256:
            return "anyh"
        if (not self.force_general and self.embedding_size == 0 and self.n_glimpses == 0 and self.pointer.name == "Dot"
                and self.serNumber <= 32 and F <= 8):
            return "fast"
        return "general"

    def _decodes_with_saves(self, inputs, forced) -> bool:
        """A REINFORCE forward whose decode runs with the BPTT's saves enabled (``gnnpn_pn_train_forward_f32`` on the
        tensor-core column-split scan), so ``replay_action_probs`` needs no second forward."""
        return (forced is None and self.training and torch.is_grad_enabled() and self.replay_impl != "torch"
                and self._impl != "ffma" and inputs.is_cuda and self._path(inputs.shape[2]) == "fast")

    def enc_layout(self, n: int, F: int) -> int:
        """Layout of the encodings ``encode`` writes for n rows of F kernel input columns (``ops.pn_enc_layout``)."""
        if self._path(F) != "fast":
            return ops.ENC_ROWMAJOR
        has_ws = self._impl == "tc"                           # ops.pn_workspace: the tensor-core kernels' scratch
        return ops.pn_enc_layout(n, self.seq_len, F, self.serCategory, self.serNumber, has_ws)

    def own_enc_buffer(self, x) -> None:
        """Gives this network a persistent ``enc_buffer`` for batches shaped like the rows ``x`` (kept across calls: a
        4.6 GB block per network at n = 18,944 that would otherwise go through the caching allocator -- per stream, with
        deferred frees for buffers that crossed streams -- on every call).  A caller-set larger buffer is left alone.
        Does nothing with a category embedding, the FFMA kernels or a hidden size other than 256."""
        n, L, F = x.shape
        if self.embedding_size != 0 or self._impl == "ffma" or self._path(F) == "anyh":
            return
        need = ops.enc_out_floats(n, L, self.hidden_size, self.enc_layout(n, F))
        if self.enc_buffer is None or self.enc_buffer.numel() < need:
            self.enc_buffer = None                            # release the old block before asking for the larger one
            self.enc_buffer = torch.empty(need, device=x.device, dtype=torch.float32)

    def encode(self, inputs):
        """The encoder half of ``forward`` (modelPN.py:183-191: embedding + encoder LSTM), enqueued on the CURRENT stream.
        Returns an opaque handle for ``forward(..., encoded=handle)``.  The two networks of the ML+2PN decode read the
        same rows and their encoders are independent, so a caller can run them concurrently on two streams (batches
        that do not fill the machine finish in the time of one encoder; gnnpn_sc_b200.pipeline does)."""
        return self._encode(inputs)

    def _encode(self, inputs, train=None):
        """``encode``.  With ``train = (latent window, uniforms)`` the decode runs as well, free-running (greedy, or sampled
        with the uniforms) with every per-step save of the BPTT (``gnnpn_pn_train_forward_f32`` on the column-split
        cluster scan): path "train".  That returns None when the batch does not fit that scan; any other failure raises."""
        B, L, _ = inputs.shape
        assert L == self.seq_len
        if not inputs.is_cuda:
            raise RuntimeError("PointerNet.forward needs CUDA tensors: the B200 path has no CPU fallback")
        K, N, H = self.serCategory, self.serNumber, self.hidden_size
        x = self._kernel_inputs(inputs)
        path = "train" if train is not None else self._path(x.shape[2])
        if path == "anyh" and (self.n_glimpses != 0 or self.pointer.name != "Dot" or N > 32):
            raise NotImplementedError(
                f"hidden_size = {H}: the any-hidden-size kernels cover Dot attention without glimpses and "
                "windows of at most 32 candidates (Bahdanau / glimpses / wider windows need hidden_size = 256)")
        range_flag = None
        if self.check_inputs and path != "anyh" and self._impl != "ffma":
            range_flag = ops.pn_check_inputs(x)
        enc_w, dec_w = self._weights()
        ws, layout, c, saves = None, ops.ENC_ROWMAJOR, None, None
        with torch.no_grad():
            if path == "anyh":
                w_cat, bias, _ = enc_w
                enc_out, c = ops.lstm_encode_anyh(x, w_cat, bias, H)
            elif path == "train":
                lat, uniform = train
                saves = ops.pn_train_forward(x, enc_w, dec_w, None, K, N, latent_win=lat, alpha=float(self.alpha),
                                             use_tanh=bool(self.pointer.use_tanh), C=float(self.pointer.C), hidden=H,
                                             impl="tc", sample_uniform=uniform)
                if saves is None:
                    return None
                enc_out = saves["enc_out"]
            else:
                ws = ops.pn_workspace(B, H, x.device, self._impl)
                layout = self.enc_layout(B, x.shape[2])
                buf = None
                if self.enc_buffer is not None:
                    # a caller-owned buffer (e.g. shared by PNLow and PNHigh at the scale-up size, where one network's
                    # encodings are ~100 GB and the caching allocator would fragment)
                    need = ops.enc_out_floats(B, L, H, layout)
                    if self.enc_buffer.numel() >= need:
                        buf = self.enc_buffer.view(-1)[:need]
                        if layout == ops.ENC_ROWMAJOR:
                            buf = buf.view(B, L, H)
                enc_out, c = ops.lstm_encode(x, enc_w, H, enc_out=buf, workspace=ws, layout=layout)
        return _Encoded(path, x, ws, layout, enc_out, c, range_flag, torch.cuda.current_stream(x.device), saves)

    def forward(self, inputs, latent, sample="sample", forced_idxs=None, encoded=None):
        """inputs [B, L, F] -> (prev_probs, prev_idxs, prev_logits), K-long each (modelPN.py:241)."""
        B, L, _ = inputs.shape
        assert L == self.seq_len
        if self.pointer.name not in ("Dot", "Bahdanau"):
            raise NotImplementedError(self.pointer.name)
        K, N = self.serCategory, self.serNumber
        use_tanh, C = bool(self.pointer.use_tanh), float(self.pointer.C)
        with torch.no_grad():
            lat = _window_of(latent, K, N) if latent else None
            forced = None if forced_idxs is None else torch.stack([t.to(torch.int32) for t in forced_idxs])
            # sample != "greedy": multinomial draw per step (modelPN.py:227-228) as an inverse-CDF pick in the kernel
            uniform = None if sample == "greedy" else torch.rand(K, B, device=inputs.device, generator=self.generator)
        self._train_saves = None
        if encoded is None:
            if self._decodes_with_saves(inputs, forced):
                # None: the batch does not fit the column-split scan; it decodes normally and replays teacher-forced
                encoded = self._encode(inputs, train=(lat, uniform))
            if encoded is None:
                encoded = self.encode(inputs)
        else:
            self._join(encoded)
        path, x, ws, layout, enc_out, c = encoded.path, encoded.x, encoded.ws, encoded.layout, encoded.enc_out, encoded.c
        _, dec_w = self._weights()
        att = self.pointer.name
        with torch.no_grad():
            ptr_blk = qw = None
            replay = None
            if path == "train":
                sv = encoded.saves
                dec_h = dec_q = sv["dec_h"]
                idx, win_logits, win_probs = sv["idx"], sv["win_logits"], sv["win_probs"]
                self._train_saves = (sv, inputs, lat)
            elif path == "anyh":
                w_cat, bias, bias0 = dec_w
                dec_h, idx, win_logits, win_probs = ops.pn_decode_anyh(
                    x, enc_out, c, w_cat, bias, bias0, K, N, latent_win=lat, alpha=float(self.alpha), use_tanh=use_tanh, C=C,
                    forced_idx=forced, sample_uniform=uniform)
                dec_q = dec_h
            elif path == "fast":
                lazy_h = layout == ops.ENC_BLOCKED128          # fused decoder: hidden states stay on chip
                c_enc = c.clone() if lazy_h else None
                kw = dict(latent_win=lat, alpha=float(self.alpha), attention="Dot", use_tanh=use_tanh, C=C,
                          workspace=ws, sample_uniform=uniform, enc_layout=layout, hidden=self.hidden_size)
                dec_h, idx, win_logits, win_probs = ops.pn_decode_greedy(x, enc_out, c, dec_w, K, N, forced_idx=forced,
                                                                         want_dec_h=not lazy_h, **kw)
                dec_q = dec_h
                if lazy_h:
                    fed_picks = idx if forced is None else forced

                    def replay():
                        with torch.no_grad():
                            return ops.pn_decode_greedy(x, enc_out, c_enc.clone(), dec_w, K, N, forced_idx=fed_picks,
                                                        want_dec_h=True, **kw)[0]
            else:
                blocks = None
                if att == "Bahdanau":
                    ptr_blk = self.pointer.block()
                    blocks = torch.cat([ptr_blk, self.glimpse.block()]) if self.n_glimpses else ptr_blk
                dec_h, dec_q, qw, idx, win_logits, win_probs = ops.pn_decode_general(
                    x, enc_out, c, dec_w, K, N, latent_win=lat, alpha=float(self.alpha), attention=att,
                    att_params=blocks, n_glimpses=self.n_glimpses, use_tanh=use_tanh, C=C, forced_idx=forced,
                    sample_uniform=uniform, use_tc=ws is not None)
        if not self.defer_range_check:
            self.raise_if_out_of_range(encoded.range_flag)
        idx64 = idx.long()
        self.last = _Last({"idx": idx, "win_logits": win_logits, "win_probs": win_probs, "latent_win": lat,
                           "enc_buf": enc_out, "enc_layout": layout, "enc_shape": (B, L, self.hidden_size),
                           "range_flag": encoded.range_flag})
        if layout == ops.ENC_ROWMAJOR:
            self.last["enc_out"] = enc_out
        if dec_h is not None:
            self.last["dec_h"], self.last["dec_q"] = dec_h, dec_q
        else:
            self.last["replay_dec_h"] = replay
        last = self.last

        fed = idx if forced is None else forced.contiguous()     # the picks the visited mask follows

        def dense_logits():
            if path == "anyh":
                return ops.pn_full_logits_anyh(last["enc_out"], last["dec_h"], fed, use_tanh, C)
            if att == "Dot":
                return ops.pn_full_logits(last["enc_out"], last["dec_q"], fed, "Dot", None, use_tanh, C)
            return ops.pn_full_logits_bahdanau(ops.pn_ref_transform(last["enc_out"], ptr_blk), qw, ptr_blk, fed,
                                               use_tanh, C)

        def dense_probs():      # exactly zero outside window k (SURVEY 3.4)
            out = torch.zeros(K, B, L, device=x.device, dtype=torch.float32)
            out.view(K, B, K, N).diagonal(dim1=0, dim2=2).copy_(win_probs.view(B, K, N).permute(0, 2, 1))
            return out

        prev_probs = _StepList(K, dense_probs)
        prev_probs.window = win_probs
        prev_logits = WindowLogits(K, win_logits, dense_logits)
        return prev_probs, list(idx64.unbind(0)), prev_logits


    @staticmethod
    def _join(encoded):
        """Orders the current stream after an ``encode`` enqueued on another stream and keeps its buffers alive."""
        cur = torch.cuda.current_stream(encoded.x.device)
        if encoded.stream != cur:
            cur.wait_stream(encoded.stream)
            for t in (encoded.x, encoded.ws, encoded.enc_out, encoded.c):
                if t is not None:
                    t.record_stream(cur)

    def decode_rollouts(self, inputs, latent, rollouts: int, encoded=None):
        """``rollouts`` decodes of every instance from ONE encoder pass (``gnnpn_pn_decode_rollouts_f32``): rollout 0 is the
        greedy decode (``forward(..., sample="greedy")``), rollouts 1.. draw every pick from the window distribution with
        uniforms from ``self.generator``, as ``sample="sample"`` does.  ``encoded``: optional handle from ``encode``.
        Returns (idx int32 [R, K, B], win_logits [R, B, L], win_probs [R, B, L]) and leaves the handle in
        ``self.last_rollouts``.  The fast configuration only (hidden_size 256, Dot attention, no glimpses, no category
        embedding, at most 32 candidates per window, the tensor-core kernels): anything else raises NotImplementedError."""
        B, L, F = inputs.shape
        assert L == self.seq_len
        if int(rollouts) != rollouts or rollouts < 1:
            raise ValueError(f"decode_rollouts: rollouts must be an integer >= 1, got {rollouts!r}")
        if self._path(F) != "fast" or self._impl != "tc":
            raise NotImplementedError(
                "best-of-R decoding runs on the fused scan kernels only: hidden_size = 256, Dot attention, n_glimpses = 0, "
                f"embedding_size = 0, at most 32 candidates per window and 8 input columns, impl 'tc' (this network: "
                f"hidden_size = {self.hidden_size}, attention = {self.pointer.name}, n_glimpses = {self.n_glimpses}, "
                f"embedding_size = {self.embedding_size}, {self.serNumber} candidates, {F} columns, impl {self._impl!r})")
        K, N = self.serCategory, self.serNumber
        R = int(rollouts)
        if encoded is None:
            encoded = self.encode(inputs)
        else:
            self._join(encoded)
        _, dec_w = self._weights()
        with torch.no_grad():
            lat = _window_of(latent, K, N) if latent else None
            uniform = torch.rand(R - 1, K, B, device=inputs.device, generator=self.generator) if R > 1 else None
            _, idx, win_logits, win_probs = ops.pn_decode_rollouts(
                encoded.x, encoded.enc_out, encoded.c, dec_w, K, N, R, sample_uniform=uniform, latent_win=lat,
                alpha=float(self.alpha), use_tanh=bool(self.pointer.use_tanh), C=float(self.pointer.C),
                enc_layout=encoded.layout, hidden=self.hidden_size)
        if not self.defer_range_check:
            self.raise_if_out_of_range(encoded.range_flag)
        self.last_rollouts = (encoded, lat)
        return idx, win_logits, win_probs

    @staticmethod
    def raise_if_out_of_range(range_flag):
        """Reads the device flag ``gnnpn_pn_check_inputs_f32`` wrote (one 4-byte device->host read = one sync)."""
        if range_flag is not None and int(range_flag.item()):
            raise ops.GnnpnError(
                "PointerNet.forward: an input value is NaN / inf or |x| >= 65504 -- outside the range of the fp16-split "
                "tensor-core LSTM (GNNPN_ERANGE).  Normalise the QoS columns (the reference's data is min-max scaled) "
                "or set actor.impl = 'ffma' for the strict-fp32 kernels.")

    def replay_action_probs(self, inputs, idx, latent_win=None):
        """Differentiable probabilities of the picks ``idx`` [K,B] (REINFORCE needs d log p / d theta).

        The decode itself runs in the CUDA kernels without autograd; this replays it with torch ops restricted to
        the windows -- outside window k the reference's probabilities are exactly 0 and carry no gradient
        (modelPN.py:220-224) -- so the gradient equals the reference's.  Encoder via nn.LSTM (cuDNN), K cell steps;
        glimpses (when configured) attend over all positions with the cumulative visited mask as in modelPN.py:208-211."""
        saves, self._train_saves = self._train_saves, None
        if self.replay_impl != "torch" and self._path(inputs.shape[2]) == "fast":
            # the library's own forward-with-saves + BPTT kernels (Dot attention, no glimpse, embedding_size = 0).  When the
            # forward of THIS batch already ran with the saves enabled (same inputs / latent objects) they are used as is
            sv = saves[0] if (saves is not None and saves[1] is inputs and saves[2] is latent_win) else None
            e, d = self.encoder, self.decoder
            probs = _ReplayFn.apply(self, inputs.detach().float().contiguous(), idx.to(torch.int32).contiguous(),
                                    latent_win, sv, self.embedding2.weight, self.embedding2.bias, self.decoder_start_input,
                                    e.weight_ih_l0, e.weight_hh_l0, e.bias_ih_l0, e.bias_hh_l0,
                                    d.weight_ih_l0, d.weight_hh_l0, d.bias_ih_l0, d.bias_hh_l0)
            return list(probs.unbind(0))
        # torch replay (every other variant: Bahdanau, glimpses, category embedding).  Strict fp32 (set process-wide in
        # gnnpn_sc_b200/__init__.py: cuDNN's TF32 default would put ~5e-4 relative error into the nn.LSTM calls below)
        B, L, _ = inputs.shape
        K, N = self.serCategory, self.serNumber
        rows = torch.arange(B, device=inputs.device)
        x = inputs.float()
        if self.embedding_size != 0:
            x = torch.cat((self.embedding1(x[:, :, 0].long()), x[:, :, 1:]), 2)
        emb = self.embedding2(x)
        enc_out, (h, c) = self.encoder(emb)
        dec_in = self.decoder_start_input.unsqueeze(0).expand(B, -1)
        visited = torch.zeros(B, L, dtype=torch.bool, device=inputs.device)
        out = []
        for k in range(K):
            _, (h, c) = self.decoder(dec_in.unsqueeze(1), (h, c))
            query = h[0]
            for _ in range(self.n_glimpses):
                refp, gl = self.glimpse.torch_rows(query, enc_out)
                gl = gl.masked_fill(visited, float("-inf"))
                query = torch.bmm(refp.transpose(1, 2), torch.softmax(gl, dim=1).unsqueeze(2)).squeeze(2)
            _, logits = self.pointer.torch_rows(query, enc_out[:, k * N:(k + 1) * N, :])
            if latent_win is not None:
                logits = logits + float(self.alpha) * latent_win[:, k * N:(k + 1) * N]
            p = torch.softmax(logits, dim=1)
            out.append(p.gather(1, (idx[k] - k * N).unsqueeze(1)).squeeze(1))
            dec_in = emb[rows, idx[k]]
            visited = visited.clone()
            visited[rows, idx[k]] = True
        return out


# --------------------------------------------------------------------------- REINFORCE replay on the library's kernels
class _ReplayFn(torch.autograd.Function):
    """Probabilities of the sampled picks, differentiable w.r.t. every actor parameter, on this library's kernels
    (``gnnpn_pn_train_forward_f32`` / ``gnnpn_pn_train_backward_f32`` + ``gnnpn_gemm_f32_bias_act`` for the weight-gradient
    contractions): the gradient trainPNLow.py:88-96 obtains from torch autograd over its K-step python graph.
    Layout shuffles (transposes, shifts) are torch copy kernels; every contraction and the BPTT run in the library."""

    @staticmethod
    def forward(ctx, actor, x, idx, latent_win, sv, emb_w, emb_b, start, e_ih, e_hh, e_bih, e_bhh, d_ih, d_hh, d_bih, d_bhh):
        K, N = actor.serCategory, actor.serNumber
        use_tanh, C = bool(actor.pointer.use_tanh), float(actor.pointer.C)
        if sv is None:                             # teacher-forced replay of the picks (no saves from the decode itself)
            enc_w, dec_w = actor._packed_weights()
            sv = ops.pn_train_forward(x, enc_w, dec_w, idx, K, N, latent_win=latent_win, alpha=float(actor.alpha),
                                      use_tanh=use_tanh, C=C, hidden=actor.hidden_size, impl=actor._impl)
        ctx.sv, ctx.x, ctx.cfg = sv, x, (K, N, use_tanh, C)
        ctx.save_for_backward(emb_w, emb_b, start, e_ih, e_hh, d_ih, d_hh)
        return sv["win_probs"].gather(1, idx.t().long()).t().contiguous()            # [K, B]

    @staticmethod
    def backward(ctx, grad_p):
        emb_w, emb_b, start, e_ih, e_hh, d_ih, d_hh = ctx.saved_tensors
        sv, x = ctx.sv, ctx.x
        K, N, use_tanh, C = ctx.cfg
        n, L, H = sv["enc_out"].shape
        F = x.shape[2]
        idx = sv["idx"].long()                                                       # [K, n]
        dGe, dGd = ops.pn_train_backward(sv, grad_p.contiguous(), e_hh.detach(), d_hh.detach(), K, N,
                                         use_tanh, C)
        mm = lambda a, w: ops.gemm_bias_act(a, w, impl="ffma")                       # a @ w.T (small operands)
        rows = torch.arange(n, device=x.device)
        enc_lnh = sv["enc_out"].permute(1, 0, 2)                                     # [L, n, H]
        dec_knh = sv["dec_h"].permute(1, 0, 2)                                       # [K, n, H]

        def contract(dG_T, h_prev, x_in):
            """One tensor-core GEMM per LSTM: dG_T [4H, T*n] against the step inputs [h(t-1) | x(t) | 1] laid out
            [H + F + 1 (padded to 16), T*n]  ->  dW_hh [4H, H], dM = d(W_ih . W_emb) [4H, F], db = row sums [4H]."""
            T = h_prev.shape[0]
            ops_in = torch.zeros(H + 16, T * n, device=x.device)
            ops_in[:H] = h_prev.reshape(T * n, H).t()
            ops_in[H:H + F] = x_in.reshape(T * n, F).t()
            ops_in[H + F] = 1.0
            out = ops.gemm_bias_act(dG_T, ops_in, impl="tc")                         # [4H, H + 16]
            return out[:, :H].contiguous(), out[:, H:H + F].contiguous(), out[:, H + F].contiguous()

        h_prev_e = torch.cat([torch.zeros_like(enc_lnh[:1]), enc_lnh[:-1]])          # [L, n, H]
        dWhh_e, dM_e, db_e = contract(dGe, h_prev_e, x.permute(1, 0, 2))
        h_prev_d = torch.cat([enc_lnh[-1:], dec_knh[:-1]])                           # [K, n, H]
        x_d = torch.cat([torch.zeros(1, n, F, device=x.device), x[rows.unsqueeze(0), idx[:-1]]])   # step 0: no input term
        dWhh_d, dM_d, db_dec = contract(dGd, h_prev_d, x_d)
        s0, db_d = dGd[:, :n].sum(1), dGd[:, n:].sum(1)                              # step 0 uses the start-token bias
        # unfold M = W_ih . W_emb,  b = b_ih + b_hh + W_ih . b_emb,  start bias = b_ih + b_hh + W_ih . start
        e_ih_t, d_ih_t = e_ih.t().contiguous(), d_ih.t().contiguous()                # [H, 4H]
        dWih_e = mm(dM_e, emb_w) + torch.outer(db_e, emb_b)
        dWih_d = mm(dM_d, emb_w) + torch.outer(db_d, emb_b) + torch.outer(s0, start)
        d_emb_w = mm(e_ih_t, dM_e.t().contiguous()) + mm(d_ih_t, dM_d.t().contiguous())
        d_emb_b = (mm(e_ih_t, db_e.view(1, -1)) + mm(d_ih_t, db_d.view(1, -1))).view(-1)
        d_start = mm(d_ih_t, s0.view(1, -1)).view(-1)
        return (None, None, None, None, None, d_emb_w, d_emb_b, d_start, dWih_e, dWhh_e, db_e, db_e, dWih_d, dWhh_d, db_dec, db_dec)


# --------------------------------------------------------------------------- CombinatorialRL
class CombinatorialRL(nn.Module):
    """modelPN.py:244-306."""

    def __init__(self, embedding_size, hidden_size, seq_len, n_glimpses, tanh_exploration, use_tanh, reward,
                 attention, sNumber, sCategory, use_cuda=True, level="Low", mask=False):
        super().__init__()
        self.reward = reward
        self.use_cuda = use_cuda
        self.level = level
        self.embedding_size = embedding_size
        self.sNumber = sNumber
        self.serCategory = sCategory
        self.actor = PointerNet(embedding_size, hidden_size, seq_len, n_glimpses, tanh_exploration, use_tanh,
                                attention, sNumber, sCategory, use_cuda, level=level, mask=mask)

    def forward(self, inputs, labs, latent=None, sample="sample", training="RL", encoded=None):
        """-> (R | probs, action_probs, actions, action_idxs, latent_p), lists of length K (modelPN.py:282-306).
        ``encoded``: optional handle from ``self.actor.encode(inputs)`` (encoder already enqueued, maybe on another stream)."""
        probs, action_idxs, logits = self.actor(inputs, latent, sample=sample, encoded=encoded)
        latent_p = logits.copy()
        idx = torch.stack(action_idxs)                                              # [K, B] int64
        B = inputs.shape[0]
        rows = torch.arange(B, device=inputs.device)
        actions = list(inputs[rows.unsqueeze(0), idx].unbind(0))                    # K x [B, F]
        if self.training and torch.is_grad_enabled():                               # REINFORCE: differentiable replay
            action_probs = self.actor.replay_action_probs(inputs, idx, self.actor.last["latent_win"])
        else:
            action_probs = list(probs.window.gather(1, idx.t()).t().unbind(0))      # K x [B]
        if training == "RL":
            R = self.reward(actions, labs, self.serCategory, USE_CUDA=self.use_cuda, level=self.level,
                            embedding_size=self.embedding_size)
            return R, action_probs, actions, action_idxs, latent_p
        return probs, action_probs, actions, action_idxs, latent_p

    @torch.no_grad()
    def best_of(self, inputs, labs, latent=None, rollouts: int = 16, encoded=None):
        """Best-of-M sampled decoding (the "Sampling" inference of a REINFORCE-trained pointer network): ``rollouts`` decodes
        of every instance (``PointerNet.decode_rollouts``: rollout 0 greedy, the others sampled) scored by this module's
        reward -- "Low": violated constraints, "High": round(viol + objFunc, 5) (``gnnpn_pn_best_rollout_f32``, the
        arithmetic of ``reward``) -- keeping the lowest, the lowest rollout on a tie, so the result is never worse than
        the greedy decode and ``rollouts=1`` is the greedy decode.  Returns (R_best [B], actions K x [B, F], action_idxs
        K x [B], rollout int32 [B]); ``self.actor.last`` then holds the chosen rollout's picks, window logits and
        probabilities.  ``labs`` is unused, as in ``reward``."""
        actor = self.actor
        idx_all, wl_all, wp_all = actor.decode_rollouts(inputs, latent, rollouts, encoded=encoded)
        encoded, lat = actor.last_rollouts
        x = encoded.x
        idx, R_best, rollout, _ = ops.pn_best_rollout(x, idx_all, level="Low" if self.level == "Low" else "High")
        B, L, _ = inputs.shape
        rows = torch.arange(B, device=inputs.device)
        chosen = rollout.long()
        win_logits, win_probs = wl_all[chosen, rows], wp_all[chosen, rows]
        K, N = self.serCategory, self.sNumber
        _, dec_w = actor._weights()
        kw = dict(latent_win=lat, alpha=float(actor.alpha), attention="Dot", use_tanh=bool(actor.pointer.use_tanh),
                  C=float(actor.pointer.C), workspace=encoded.ws, enc_layout=encoded.layout, hidden=actor.hidden_size)

        def replay():       # the chosen rollout's decoder states: the decode teacher-forced on its picks
            return ops.pn_decode_greedy(x, encoded.enc_out, encoded.c.clone(), dec_w, K, N, forced_idx=idx, want_dec_h=True,
                                        **kw)[0]
        actor.last = _Last({"idx": idx, "win_logits": win_logits, "win_probs": win_probs, "latent_win": lat,
                            "enc_buf": encoded.enc_out, "enc_layout": encoded.layout,
                            "enc_shape": (B, L, actor.hidden_size), "range_flag": encoded.range_flag,
                            "replay_dec_h": replay})
        if encoded.layout == ops.ENC_ROWMAJOR:
            actor.last["enc_out"] = encoded.enc_out
        idx64 = idx.long()
        actions = list(inputs[rows.unsqueeze(0), idx64].unbind(0))
        return (R_best if self.use_cuda else R_best.cpu()), actions, list(idx64.unbind(0)), rollout
