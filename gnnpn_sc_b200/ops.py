"""Torch-tensor front end of the C ABI: allocates outputs with torch, passes raw
device pointers + the current CUDA stream.  Plumbing only -- all arithmetic
happens in ``libgnnpn_b200.so``.  Every function requires CUDA tensors."""
from __future__ import annotations

from typing import Optional

import torch

from ._lib import GnnpnError, check, get_option, lib, set_option  # noqa: F401  (re-exported)

ACT = {None: 0, "none": 0, "relu": 1, "sigmoid": 2}
# "tc": tcgen05 recurrence / node transform (default);  "ffma": strict-fp32 CUDA-core kernels
DEFAULT_IMPL = "tc"
TC_GEMM_MIN_ROWS = 512          # below this the tile pipeline cannot fill; the FFMA kernel is used
ATT = {"Dot": 0, "Bahdanau": 1}
CSR_PLAIN, CSR_GCN_NORM = 0, 1
ENC_ROWMAJOR, ENC_BLOCKED128 = 0, 1     # include/gnnpn_b200.h: layouts of the encoder -> decoder encodings buffer


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _f32(t: torch.Tensor, name: str) -> torch.Tensor:
    if not t.is_cuda:
        raise RuntimeError(f"{name}: expected a CUDA tensor (the B200 path has no CPU fallback)")
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


# ------------------------------------------------------------------ pointer network
def packed_lstm_floats(hidden: int, in_features: int) -> int:
    return int(lib().gnnpn_pn_packed_lstm_floats(hidden, in_features))


def pack_lstm(w_ih, w_hh, b_ih, b_hh, w_embed, b_embed, start_input=None) -> torch.Tensor:
    """Folded + gate-interleaved LSTM block (see ``gnnpn_pn_pack_lstm_f32``)."""
    H = w_hh.shape[1]
    F = w_embed.shape[1]
    args = [_f32(t, "weight") for t in (w_ih, w_hh, b_ih, b_hh, w_embed, b_embed)]
    st = None if start_input is None else _f32(start_input, "start_input")
    out = torch.empty(packed_lstm_floats(H, F), device=args[0].device, dtype=torch.float32)
    check(lib().gnnpn_pn_pack_lstm_f32(*[a.data_ptr() for a in args], _ptr(st), H, F, out.data_ptr(), _stream()),
          "pn_pack_lstm")
    return out


def pn_workspace(n: int, hidden: int = 256, device=None, impl: Optional[str] = None) -> Optional[torch.Tensor]:
    """Scratch for the tensor-core recurrence, or None when the FFMA kernels are selected."""
    if (impl or DEFAULT_IMPL) != "tc":
        return None
    nbytes = int(lib().gnnpn_pn_workspace_bytes(n, hidden))
    return torch.empty(nbytes, device=device, dtype=torch.uint8)


def _ws(ws):
    return (None, 0) if ws is None else (ws.data_ptr(), ws.numel())


def _decode_inputs(n: int, L: int, K: int, latent_win, forced_idx, sample_uniform):
    """The optional inputs of a decode as the kernels take them: ``latent_win`` fp32 [n, L], ``forced_idx`` int32 [K, n],
    ``sample_uniform`` fp32 [K, n], contiguous (None stays None)."""
    if latent_win is not None:
        latent_win = _f32(latent_win, "latent_win")
        assert latent_win.shape == (n, L)
    if forced_idx is not None:
        forced_idx = forced_idx.to(torch.int32).contiguous()
        assert forced_idx.shape == (K, n)
    if sample_uniform is not None:
        sample_uniform = _f32(sample_uniform, "sample_uniform")
        assert sample_uniform.shape == (K, n)
    return latent_win, forced_idx, sample_uniform


def _decode_outputs(n: int, L: int, K: int, device):
    """(idx int32 [K, n], win_logits [n, L], win_probs [n, L]) of a decode."""
    return (torch.empty(K, n, device=device, dtype=torch.int32), torch.empty(n, L, device=device, dtype=torch.float32),
            torch.empty(n, L, device=device, dtype=torch.float32))


def pn_check_inputs(inputs: torch.Tensor) -> torch.Tensor:
    """int32 [1] device flag: 1 when a raw input value is NaN / inf / outside the fp16-split range of the LSTM kernels
    (``gnnpn_pn_input_limit()``).  Asynchronous; the caller decides when to read it."""
    x = _f32(inputs, "inputs")
    flag = torch.zeros(1, device=x.device, dtype=torch.int32)
    check(lib().gnnpn_pn_check_inputs_f32(x.data_ptr(), x.numel(), flag.data_ptr(), _stream()), "pn_check_inputs")
    return flag


def pn_enc_layout(n: int, L: int, F: int, K: int, N: int, has_workspace: bool = True) -> int:
    """Layout the dispatcher wants for the (lstm_encode, pn_decode_greedy) pair of a batch: ``ENC_BLOCKED128`` when the
    batch runs on the persistent CTA-pair scan (pointer dots fused into the decoder's cell epilogue), else row-major."""
    return int(lib().gnnpn_pn_enc_layout(n, L, F, K, N, int(bool(has_workspace))))


def enc_out_floats(n: int, L: int, hidden: int, layout: int) -> int:
    """Floats an encodings buffer of this layout holds (the blocked layout pads n to whole groups of 128)."""
    if layout == ENC_ROWMAJOR:
        return n * L * hidden
    return int(lib().gnnpn_pn_enc_out_floats(n, L, hidden, layout))


def enc_out_empty(n: int, L: int, hidden: int, layout: int, device) -> torch.Tensor:
    """Encodings buffer for ``lstm_encode``: ``[n, L, H]`` (row-major) or the flat blocked buffer."""
    if layout == ENC_ROWMAJOR:
        return torch.empty(n, L, hidden, device=device, dtype=torch.float32)
    return torch.empty(enc_out_floats(n, L, hidden, layout), device=device, dtype=torch.float32)


def enc_to_rowmajor(enc_blocked: torch.Tensor, n: int, L: int, hidden: int = 256) -> torch.Tensor:
    """Blocked encodings -> the reference's ``[n, L, H]`` tensor (modelPN.py:191)."""
    out = torch.empty(n, L, hidden, device=enc_blocked.device, dtype=torch.float32)
    check(lib().gnnpn_pn_enc_to_rowmajor_f32(enc_blocked.data_ptr(), n, L, hidden, out.data_ptr(), _stream()),
          "enc_to_rowmajor")
    return out


def lstm_encode(inputs: torch.Tensor, packed: torch.Tensor, hidden: int = 256,
                enc_out: Optional[torch.Tensor] = None, c_state: Optional[torch.Tensor] = None,
                workspace: Optional[torch.Tensor] = None, layout: int = ENC_ROWMAJOR):
    x = _f32(inputs, "inputs")
    n, L, F = x.shape
    if enc_out is None:
        enc_out = enc_out_empty(n, L, hidden, layout, x.device)
    if c_state is None:
        c_state = torch.empty(n, hidden, device=x.device, dtype=torch.float32)
    check(lib().gnnpn_lstm_encode_f32(x.data_ptr(), n, L, F, hidden, packed.data_ptr(), enc_out.data_ptr(),
                                      c_state.data_ptr(), *_ws(workspace), int(layout), _stream()), "lstm_encode")
    return enc_out, c_state


def pn_decode_greedy(inputs, enc_out, c_state, packed_dec, K: int, N: int, latent_win=None, alpha: float = 1.0,
                     attention: str = "Dot", att_params=None, use_tanh: bool = True, C: float = 10.0,
                     forced_idx=None, out=None, workspace: Optional[torch.Tensor] = None,
                     sample_uniform: Optional[torch.Tensor] = None, enc_layout: int = ENC_ROWMAJOR, hidden: int = 256,
                     want_dec_h: bool = True):
    """Returns (dec_h [n,K,H] | None, idx int32 [K,n], win_logits [n,L], win_probs [n,L]).  ``c_state`` is updated in
    place.  ``enc_out`` is in ``enc_layout`` (as produced by ``lstm_encode(..., layout=enc_layout)``).  With blocked
    encodings the decoder hidden states need not be written to memory: ``want_dec_h=False`` (or ``out[0] is None``)."""
    x = _f32(inputs, "inputs")
    n, L, F = x.shape
    H = enc_out.shape[2] if enc_layout == ENC_ROWMAJOR else hidden
    dev = x.device
    if out is None:
        dec_h = torch.empty(n, K, H, device=dev, dtype=torch.float32) if (want_dec_h or enc_layout == ENC_ROWMAJOR) else None
        idx, wl, wp = _decode_outputs(n, L, K, dev)
    else:
        dec_h, idx, wl, wp = out
    latent_win, forced_idx, sample_uniform = _decode_inputs(n, L, K, latent_win, forced_idx, sample_uniform)
    check(lib().gnnpn_pn_decode_greedy_f32(
        x.data_ptr(), enc_out.data_ptr(), c_state.data_ptr(), _ptr(latent_win), float(alpha),
        packed_dec.data_ptr(), ATT[attention], _ptr(att_params), int(bool(use_tanh)), float(C),
        n, L, F, H, K, N, _ptr(dec_h), idx.data_ptr(), wl.data_ptr(), wp.data_ptr(),
        _ptr(forced_idx), _ptr(sample_uniform), *_ws(workspace), int(enc_layout), _stream()), "pn_decode_greedy")
    return dec_h, idx, wl, wp


def pn_decode_rollouts(inputs, enc_out, c_state, packed_dec, K: int, N: int, rollouts: int, sample_uniform=None,
                       latent_win=None, alpha: float = 1.0, use_tanh: bool = True, C: float = 10.0,
                       enc_layout: int = ENC_ROWMAJOR, hidden: int = 256, want_dec_h: bool = False):
    """``rollouts`` decodes of every instance from one set of encodings (``gnnpn_pn_decode_rollouts_f32``): rollout 0
    greedy, rollout r >= 1 drawn with ``sample_uniform[r-1]`` (fp32 [rollouts-1, K, n]).  ``c_state`` is read, not
    updated.  Returns (dec_h [R, n, K, H] | None, idx int32 [R, K, n], win_logits [R, n, L], win_probs [R, n, L]); dec_h
    is allocated when the decoder needs it (row-major encodings) or ``want_dec_h``."""
    x = _f32(inputs, "inputs")
    n, L, F = x.shape
    R = int(rollouts)
    if R < 1:
        raise ValueError(f"pn_decode_rollouts: rollouts must be >= 1, got {R}")
    dev = x.device
    dec_h = (torch.empty(R, n, K, hidden, device=dev, dtype=torch.float32)
             if (want_dec_h or enc_layout == ENC_ROWMAJOR) else None)
    idx = torch.empty(R, K, n, device=dev, dtype=torch.int32)
    wl = torch.empty(R, n, L, device=dev, dtype=torch.float32)
    wp = torch.empty(R, n, L, device=dev, dtype=torch.float32)
    if latent_win is not None:
        latent_win = _f32(latent_win, "latent_win")
        assert latent_win.shape == (n, L)
    if sample_uniform is not None:
        sample_uniform = _f32(sample_uniform, "sample_uniform")
        assert sample_uniform.shape == (R - 1, K, n)
    ws = torch.empty(int(lib().gnnpn_pn_rollouts_workspace_bytes(n, hidden, R)), device=dev, dtype=torch.uint8)
    check(lib().gnnpn_pn_decode_rollouts_f32(
        x.data_ptr(), enc_out.data_ptr(), c_state.data_ptr(), _ptr(latent_win), float(alpha), packed_dec.data_ptr(),
        ATT["Dot"], None, int(bool(use_tanh)), float(C), n, L, F, hidden, K, N, _ptr(dec_h), idx.data_ptr(),
        wl.data_ptr(), wp.data_ptr(), _ptr(sample_uniform), *_ws(ws), int(enc_layout), R, _stream()),
        "pn_decode_rollouts")
    return dec_h, idx, wl, wp


def pn_best_rollout(inputs, idx, level: str = "High", tag: int = 0, want_rollout_rewards: bool = False):
    """Best rollout of picks ``idx`` int32 [R, K, n] by the reward of ``level`` ("Low": violations, "High":
    round(viol + obj, 5)), lowest rollout on a tie (``gnnpn_pn_best_rollout_f32``).  Returns (best picks int32 [K, n],
    best reward fp32 [n], chosen rollout int32 [n], every rollout's reward fp32 [R, n] | None)."""
    x = _f32(inputs, "inputs")
    n, L, F = x.shape
    idx = idx.to(torch.int32).contiguous()
    R, K, _ = idx.shape
    if level not in ("Low", "High"):
        raise ValueError(f"pn_best_rollout: level must be 'Low' or 'High', got {level!r}")
    best_idx = torch.empty(K, n, device=x.device, dtype=torch.int32)
    best_rew = torch.empty(n, device=x.device, dtype=torch.float32)
    best_r = torch.empty(n, device=x.device, dtype=torch.int32)
    rews = torch.empty(R, n, device=x.device, dtype=torch.float32) if want_rollout_rewards else None
    check(lib().gnnpn_pn_best_rollout_f32(x.data_ptr(), idx.data_ptr(), n, L, F, K, tag, int(level == "High"), R,
                                          best_idx.data_ptr(), best_rew.data_ptr(), best_r.data_ptr(), _ptr(rews),
                                          _stream()), "pn_best_rollout")
    return best_idx, best_rew, best_r, rews


# ------------------------------------------------------------------ any hidden size (strict fp32, per-step launches)
def anyh_fold(w_ih, w_hh, b_ih, b_hh, w_embed, b_embed, start_input=None):
    """Folded weights of the any-hidden-size kernels: ``w_cat [4H, H+F] = [W_hh | W_ih . W_emb]``, ``bias = b_ih + b_hh +
    W_ih . b_emb`` and, for a decoder, ``bias0 = b_ih + b_hh + W_ih . start``.  float64 products (as the H = 256 packer)."""
    wi, we = w_ih.detach().double(), w_embed.detach().double()
    b = b_ih.detach().double() + b_hh.detach().double()
    w_cat = torch.cat([w_hh.detach().double(), wi @ we], 1).float().contiguous()
    bias = (b + wi @ b_embed.detach().double()).float().contiguous()
    bias0 = None if start_input is None else (b + wi @ start_input.detach().double()).float().contiguous()
    return w_cat, bias, bias0


def _anyh_ws(n, H, F, device):
    return torch.empty(int(lib().gnnpn_pn_anyh_workspace_floats(n, H, F)), device=device, dtype=torch.float32)


def lstm_encode_anyh(inputs, w_cat, bias, hidden: int):
    x = _f32(inputs, "inputs")
    n, L, F = x.shape
    enc_out = torch.empty(n, L, hidden, device=x.device, dtype=torch.float32)
    c = torch.empty(n, hidden, device=x.device, dtype=torch.float32)
    ws = _anyh_ws(n, hidden, F, x.device)
    check(lib().gnnpn_lstm_encode_anyh_f32(x.data_ptr(), n, L, F, hidden, w_cat.data_ptr(), bias.data_ptr(), enc_out.data_ptr(),
                                           c.data_ptr(), ws.data_ptr(), ws.numel(), _stream()), "lstm_encode_anyh")
    return enc_out, c


def pn_decode_anyh(inputs, enc_out, c_state, w_cat, bias, bias0, K: int, N: int, latent_win=None, alpha: float = 1.0,
                   use_tanh: bool = True, C: float = 10.0, forced_idx=None, sample_uniform=None):
    """-> (dec_h [n,K,H], idx int32 [K,n], win_logits [n,L], win_probs [n,L]); ``c_state`` is updated in place."""
    x = _f32(inputs, "inputs")
    n, L, F = x.shape
    H = enc_out.shape[2]
    dev = x.device
    dec_h = torch.empty(n, K, H, device=dev, dtype=torch.float32)
    idx, wl, wp = _decode_outputs(n, L, K, dev)
    latent_win, forced_idx, sample_uniform = _decode_inputs(n, L, K, latent_win, forced_idx, sample_uniform)
    ws = _anyh_ws(n, H, F, dev)
    check(lib().gnnpn_pn_decode_anyh_f32(x.data_ptr(), enc_out.data_ptr(), c_state.data_ptr(), _ptr(latent_win), float(alpha),
                                         w_cat.data_ptr(), bias.data_ptr(), bias0.data_ptr(), int(bool(use_tanh)), float(C),
                                         n, L, F, H, K, N, dec_h.data_ptr(), idx.data_ptr(), wl.data_ptr(), wp.data_ptr(),
                                         _ptr(forced_idx), _ptr(sample_uniform), ws.data_ptr(), ws.numel(), _stream()),
          "pn_decode_anyh")
    return dec_h, idx, wl, wp


def pn_full_logits_anyh(enc_out, dec_h, idx, use_tanh: bool = True, C: float = 10.0) -> torch.Tensor:
    n, L, H = enc_out.shape
    K = dec_h.shape[1]
    out = torch.empty(K, n, L, device=enc_out.device, dtype=torch.float32)
    check(lib().gnnpn_pn_full_logits_anyh_f32(enc_out.data_ptr(), dec_h.data_ptr(), idx.contiguous().data_ptr(),
                                              int(bool(use_tanh)), float(C), n, L, H, K, out.data_ptr(), _stream()),
          "pn_full_logits_anyh")
    return out


def pn_train_forward(inputs, packed_enc, packed_dec, idx, K: int, N: int, latent_win=None, alpha: float = 1.0,
                     use_tanh: bool = True, C: float = 10.0, hidden: int = 256, impl: Optional[str] = None,
                     sample_uniform=None):
    """Forward half of the REINFORCE gradient (``gnnpn_pn_train_forward_f32``): runs the network saving what the BPTT
    needs.  Returns the dict of saves (``sv["idx"]``: the picks the steps were fed).

    ``impl="tc"`` (default) runs the tensor-core column-split cluster scan when it takes the batch
    (``gnnpn_pn_train_forward_workspace_bytes`` > 0): the kernels of the small-batch inference path with saves enabled;
    with ``idx=None`` and ``sample_uniform`` it IS the sampled decode (no replay needed).  ``impl="ffma"`` and larger
    batches replay the picks ``idx`` on the strict-fp32 per-step kernels; with ``idx=None`` they return None: decode
    first."""
    x = _f32(inputs, "inputs")
    n, L, F = x.shape
    dev, H = x.device, hidden
    lat, idx, uni = _decode_inputs(n, L, K, latent_win, idx, sample_uniform)
    ws = None
    if (impl or DEFAULT_IMPL) == "tc":
        nbytes = int(lib().gnnpn_pn_train_forward_workspace_bytes(n, L, F, H, K, N))
        ws = torch.empty(nbytes, device=dev, dtype=torch.uint8) if nbytes else None
    if idx is None and ws is None:
        return None
    f = lambda *shape: torch.empty(*shape, device=dev, dtype=torch.float32)
    idx_free, wl, wp = _decode_outputs(n, L, K, dev)
    sv = {"enc_out": f(n, L, H), "gates_e": f(L, n, 4 * H), "c_e": f(L, n, H), "dec_h": f(n, K, H),
          "gates_d": f(K, n, 4 * H), "c_d": f(K, n, H), "win_logits": wl, "win_probs": wp,
          "idx": idx_free if idx is None else idx}        # free-running (greedy / sampled): the picks ARE the fed picks
    check(lib().gnnpn_pn_train_forward_f32(
        x.data_ptr(), packed_enc.data_ptr(), packed_dec.data_ptr(), _ptr(idx), _ptr(uni), _ptr(lat), float(alpha),
        int(bool(use_tanh)), float(C), n, L, F, H, K, N, sv["enc_out"].data_ptr(), sv["gates_e"].data_ptr(),
        sv["c_e"].data_ptr(), sv["dec_h"].data_ptr(), sv["gates_d"].data_ptr(), sv["c_d"].data_ptr(),
        wl.data_ptr(), wp.data_ptr(), idx_free.data_ptr(), *_ws(ws), _stream()), "pn_train_forward")
    return sv


def pn_train_backward(sv, grad_p, w_hh_enc, w_hh_dec, K: int, N: int, use_tanh: bool = True, C: float = 10.0):
    """Backward half (``gnnpn_pn_train_backward_f32``): -> (dG_enc_T [4H, L*n], dG_dec_T [4H, K*n])."""
    n, L, H = sv["enc_out"].shape
    dev = sv["enc_out"].device
    dGe = torch.empty(4 * H, L * n, device=dev, dtype=torch.float32)
    dGd = torch.empty(4 * H, K * n, device=dev, dtype=torch.float32)
    nws = int(lib().gnnpn_pn_train_backward_workspace_floats(n, L, K, H))
    ws = torch.empty(nws, device=dev, dtype=torch.float32)
    gp = _f32(grad_p, "grad_p")
    check(lib().gnnpn_pn_train_backward_f32(
        sv["enc_out"].data_ptr(), sv["gates_e"].data_ptr(), sv["c_e"].data_ptr(), sv["dec_h"].data_ptr(),
        sv["gates_d"].data_ptr(), sv["c_d"].data_ptr(), sv["win_logits"].data_ptr(), sv["win_probs"].data_ptr(),
        sv["idx"].data_ptr(), gp.data_ptr(), _f32(w_hh_enc, "w_hh").data_ptr(), _f32(w_hh_dec, "w_hh").data_ptr(),
        int(bool(use_tanh)), float(C), n, L, H, K, N, dGe.data_ptr(), dGd.data_ptr(), ws.data_ptr(), ws.numel(),
        _stream()), "pn_train_backward")
    return dGe, dGd


def att_block(W_query_w, W_query_b, W_ref_w, W_ref_b, V) -> torch.Tensor:
    """One Attention module's Bahdanau parameters in the layout of ``gnnpn_pn_att_block_floats``."""
    H = V.numel()
    parts = [W_query_w.reshape(H * H), W_query_b.reshape(H), W_ref_w.reshape(H * H), W_ref_b.reshape(H), V.reshape(H)]
    out = torch.cat([_f32(t.detach(), "attention parameter") for t in parts])
    assert out.numel() == int(lib().gnnpn_pn_att_block_floats(H))
    return out


def pn_decode_general(inputs, enc_out, c_state, packed_dec, K: int, N: int, latent_win=None, alpha: float = 1.0,
                      attention: str = "Dot", att_params=None, n_glimpses: int = 0, use_tanh: bool = True,
                      C: float = 10.0, forced_idx=None, sample_uniform=None, use_tc: bool = True):
    """Every PointerNet variant (Bahdanau, glimpses, any window width, <= 32 raw columns).
    Returns (dec_h, dec_q, qw_pointer | None, idx int32 [K,n], win_logits [n,L], win_probs [n,L])."""
    x = _f32(inputs, "inputs")
    n, L, F = x.shape
    H = enc_out.shape[2]
    dev = x.device
    dec_h = torch.empty(n, K, H, device=dev, dtype=torch.float32)
    dec_q = torch.empty(n, K, H, device=dev, dtype=torch.float32) if n_glimpses > 0 else dec_h
    qw = torch.empty(n, K, H, device=dev, dtype=torch.float32) if attention == "Bahdanau" else None
    idx, wl, wp = _decode_outputs(n, L, K, dev)
    latent_win, forced_idx, sample_uniform = _decode_inputs(n, L, K, latent_win, forced_idx, sample_uniform)
    nbytes = int(lib().gnnpn_pn_decode_general_workspace_bytes(n, L, K, H, ATT[attention], n_glimpses, int(use_tc)))
    ws = torch.empty(nbytes, device=dev, dtype=torch.uint8)
    check(lib().gnnpn_pn_decode_general_f32(
        x.data_ptr(), enc_out.data_ptr(), c_state.data_ptr(), _ptr(latent_win), float(alpha), packed_dec.data_ptr(),
        ATT[attention], _ptr(att_params), int(n_glimpses), int(bool(use_tanh)), float(C), n, L, F, H, K, N,
        dec_h.data_ptr(), dec_q.data_ptr(), _ptr(qw), idx.data_ptr(), wl.data_ptr(), wp.data_ptr(),
        _ptr(forced_idx), _ptr(sample_uniform), int(use_tc), ws.data_ptr(), ws.numel(), _stream()), "pn_decode_general")
    return dec_h, dec_q, qw, idx, wl, wp


def pn_ref_transform(enc_out, block) -> torch.Tensor:
    """Bahdanau ``W_ref`` (Conv1d(H,H,1), modelPN.py:87,105) on every position: [.., H] -> [.., H]."""
    x = _f32(enc_out, "enc_out")
    H = x.shape[-1]
    out = torch.empty_like(x)
    check(lib().gnnpn_pn_ref_transform_f32(x.data_ptr(), block.data_ptr(), x.numel() // H, H, out.data_ptr(), _stream()),
          "pn_ref_transform")
    return out


def pn_query_transform(q, block) -> torch.Tensor:
    """Bahdanau ``W_query`` (modelPN.py:85,104): [rows, H] -> [rows, H]."""
    x = _f32(q, "query")
    rows, H = x.shape
    out = torch.empty_like(x)
    check(lib().gnnpn_pn_query_transform_f32(x.data_ptr(), H, block.data_ptr(), rows, H, out.data_ptr(), H, _stream()),
          "pn_query_transform")
    return out


def pn_full_logits_bahdanau(E, qw, block, idx, use_tanh: bool = True, C: float = 10.0) -> torch.Tensor:
    n, L, H = E.shape
    K = qw.shape[1]
    out = torch.empty(K, n, L, device=E.device, dtype=torch.float32)
    check(lib().gnnpn_pn_full_logits_bahdanau_f32(E.data_ptr(), qw.data_ptr(), block.data_ptr(), idx.data_ptr(),
                                                  int(bool(use_tanh)), float(C), n, L, H, K, out.data_ptr(), _stream()),
          "pn_full_logits_bahdanau")
    return out


def pn_full_logits(enc_out, dec_h, idx, attention: str = "Dot", att_params=None, use_tanh: bool = True,
                   C: float = 10.0) -> torch.Tensor:
    n, L, H = enc_out.shape
    K = dec_h.shape[1]
    out = torch.empty(K, n, L, device=enc_out.device, dtype=torch.float32)
    check(lib().gnnpn_pn_full_logits_f32(enc_out.data_ptr(), dec_h.data_ptr(), idx.data_ptr(), ATT[attention],
                                         _ptr(att_params), int(bool(use_tanh)), float(C), n, L, H, K,
                                         out.data_ptr(), _stream()), "pn_full_logits")
    return out


def pn_attention_windows(enc_out, dec_h, N: int, latent_win=None, alpha: float = 1.0, use_tanh: bool = True, C: float = 10.0,
                         out=None):
    """Window logits / probabilities / first-max picks of every decode step for GIVEN decoder states (row-major encodings
    ``[n, L, H]``, ``dec_h [n, K, H]``): ``gnnpn_pn_attention_windows_f32``.  Returns (idx int32 [K, n], win_logits, win_probs)."""
    n, L, H = enc_out.shape
    K = dec_h.shape[1]
    idx, wl, wp = _decode_outputs(n, L, K, enc_out.device) if out is None else out
    lat = None if latent_win is None else _f32(latent_win, "latent_win")
    check(lib().gnnpn_pn_attention_windows_f32(enc_out.data_ptr(), dec_h.data_ptr(), _ptr(lat), float(alpha), int(bool(use_tanh)),
                                               float(C), n, L, H, K, N, idx.data_ptr(), wl.data_ptr(), wp.data_ptr(), _stream()),
          "pn_attention_windows")
    return idx, wl, wp


def pn_reward(inputs, idx, tag: int = 0):
    """(violations int32 [n], objFunc fp32 [n], round(viol+obj,5) fp32 [n]) for picks ``idx`` int32 [K,n]."""
    x = _f32(inputs, "inputs")
    n, L, F = x.shape
    idx = idx.to(torch.int32).contiguous()
    K = idx.shape[0]
    viol = torch.empty(n, device=x.device, dtype=torch.int32)
    obj = torch.empty(n, device=x.device, dtype=torch.float32)
    rew = torch.empty(n, device=x.device, dtype=torch.float32)
    check(lib().gnnpn_pn_reward_f32(x.data_ptr(), idx.data_ptr(), n, L, F, K, tag, viol.data_ptr(),
                                    obj.data_ptr(), rew.data_ptr(), _stream()), "pn_reward")
    return viol, obj, rew


# ------------------------------------------------------------------ candidate selection (loadDataPN on the device)
def woa_fitness(qos: torch.Tensor, idx: torch.Tensor, bounds: torch.Tensor, klen: Optional[torch.Tensor] = None):
    """``ESWOA.calc`` (WOA.py:87-105) for a batch of positions: ``qos`` f64 [T,4], ``idx`` int32 [P,Kmax] rows of
    ``qos``, ``bounds`` f64 [P,4] (lo1,hi1,lo2,hi2), ``klen`` int32 [P] or None -> (viol int32 [P], obj f64 [P],
    fitness f64 [P]); float64 in numpy's operation order (bit-identical to the reference's values)."""
    if not (qos.is_cuda and idx.is_cuda and bounds.is_cuda):
        raise GnnpnError("woa_fitness needs CUDA tensors (no CPU fallback)")
    assert qos.dtype == torch.float64 and bounds.dtype == torch.float64 and idx.dtype == torch.int32
    qos, idx, bounds = qos.contiguous(), idx.contiguous(), bounds.contiguous()
    P, Kmax = idx.shape
    viol = torch.empty(P, device=idx.device, dtype=torch.int32)
    obj = torch.empty(P, device=idx.device, dtype=torch.float64)
    fit = torch.empty(P, device=idx.device, dtype=torch.float64)
    if klen is not None:
        assert klen.dtype == torch.int32 and klen.is_cuda
        klen = klen.contiguous()
    check(lib().gnnpn_woa_fitness_f64(qos.data_ptr(), qos.shape[0], idx.data_ptr(), idx.stride(0), _ptr(klen),
                                      bounds.data_ptr(), P, Kmax, viol.data_ptr(), obj.data_ptr(), fit.data_ptr(),
                                      _stream()), "woa_fitness")
    return viol, obj, fit


def ml2pn_score(qos: torch.Tensor, idx: torch.Tensor, bounds: torch.Tensor, klen: torch.Tensor):
    """``ML2PN.calc`` (ML2PN.py:6-12) for a batch of compositions, float64: same layout as :func:`woa_fitness`, the
    mean of q0 runs over all ``klen[p]`` picks.  -> (viol int32 [P], obj f64 [P], score f64 [P]): the score is obj
    with 1.0 added once per violated constraint, one add at a time as ``ML2PN.calc`` does."""
    if not (qos.is_cuda and idx.is_cuda and bounds.is_cuda and klen.is_cuda):
        raise GnnpnError("ml2pn_score needs CUDA tensors (no CPU fallback)")
    assert qos.dtype == torch.float64 and bounds.dtype == torch.float64
    assert idx.dtype == torch.int32 and klen.dtype == torch.int32
    qos, idx, bounds, klen = qos.contiguous(), idx.contiguous(), bounds.contiguous(), klen.contiguous()
    P, Kmax = idx.shape
    viol = torch.empty(P, device=idx.device, dtype=torch.int32)
    obj = torch.empty(P, device=idx.device, dtype=torch.float64)
    score = torch.empty(P, device=idx.device, dtype=torch.float64)
    check(lib().gnnpn_ml2pn_score_f64(qos.data_ptr(), qos.shape[0], idx.data_ptr(), idx.stride(0), klen.data_ptr(),
                                      bounds.data_ptr(), P, Kmax, viol.data_ptr(), obj.data_ptr(), score.data_ptr(),
                                      _stream()), "ml2pn_score")
    return viol, obj, score


def woa_search(qos, base, size, klen, bounds, pops, best_fit, best_ref, best_vec, seeds, traj):
    """Device-resident ESWOA search (``gnnpn_woa_search_f64``): all tensors CUDA, updated in place (see the header)."""
    I, P, KM = pops.shape
    for x, dt in ((qos, torch.float64), (bounds, torch.float64), (best_fit, torch.float64), (traj, torch.float64),
                  (base, torch.int32), (size, torch.int32), (klen, torch.int32), (pops, torch.int32),
                  (best_ref, torch.int32), (best_vec, torch.int32), (seeds, torch.int64)):
        if not (x.is_cuda and x.is_contiguous() and x.dtype == dt):
            raise GnnpnError("woa_search needs contiguous CUDA tensors of the declared dtypes (no CPU fallback)")
    check(lib().gnnpn_woa_search_f64(qos.data_ptr(), qos.shape[0], base.data_ptr(), size.data_ptr(), klen.data_ptr(),
                                     bounds.data_ptr(), pops.data_ptr(), best_fit.data_ptr(), best_ref.data_ptr(),
                                     best_vec.data_ptr(), seeds.data_ptr(), traj.data_ptr(), I, P, KM, traj.shape[1],
                                     _stream()), "woa_search")


# gnnpn_woa_prepare_f64's flags: the host path raises for all but 8, which is input the device stage does not take
WOA_FLAGS = {1: "more seed rows than candidate lists", 2: "the reduct front replaces past the end of its list",
             4: "no feasible candidate for any task",
             8: "unsupported request: a category requested twice or outside the catalogue",
             16: "fewer seed rows than candidate lists (a requested category with a neutral pick)"}


def woa_prepare(svc_raw, svc_round, cat_ptr, req_cat, n_req, local_bounds, global_bounds, seed_rows, seed_ids, seeds,
                popSize: int, reduct: float):
    """Candidate lists, seed, initial population and best state of the ESWOA stage on the device
    (``gnnpn_woa_prepare_f64``), in the layouts :func:`woa_search` takes.  Returns a dict of CUDA tensors: qos, ids,
    base, size, klen, list_cat, pops, best_fit, best_ref, best_vec, flags (see the header)."""
    n, K = req_cat.shape
    for x, dt in ((svc_raw, torch.float64), (svc_round, torch.float64), (cat_ptr, torch.int32), (req_cat, torch.int32),
                  (n_req, torch.int32), (local_bounds, torch.float64), (global_bounds, torch.float64),
                  (seed_rows, torch.float32), (seed_ids, torch.int32), (seeds, torch.int64)):
        if not (x.is_cuda and x.is_contiguous() and x.dtype == dt):
            raise GnnpnError("woa_prepare needs contiguous CUDA tensors of the declared dtypes (no CPU fallback)")
    assert cat_ptr.numel() == K + 1 and local_bounds.shape == (n, K, 4) and seed_rows.shape == (n, K, 4)
    S = svc_raw.shape[0]
    dev = req_cat.device
    rows = int(lib().gnnpn_woa_prepare_rows(n, S, K))
    i32 = lambda *s: torch.empty(s, device=dev, dtype=torch.int32)
    o = {"qos": torch.empty(rows, 4, device=dev, dtype=torch.float64), "ids": i32(rows), "base": i32(n, K),
           "size": i32(n, K), "klen": i32(n), "list_cat": i32(n, K), "pops": i32(n, popSize, K),
           "best_fit": torch.empty(n, device=dev, dtype=torch.float64), "best_ref": i32(n), "best_vec": i32(n, K),
           "flags": i32(n)}
    check(lib().gnnpn_woa_prepare_f64(
        svc_raw.data_ptr(), svc_round.data_ptr(), cat_ptr.data_ptr(), S, K, req_cat.data_ptr(), n_req.data_ptr(),
        local_bounds.data_ptr(), global_bounds.data_ptr(), seed_rows.data_ptr(), seed_ids.data_ptr(), seeds.data_ptr(),
        n, popSize, float(reduct), o["qos"].data_ptr(), o["ids"].data_ptr(), o["base"].data_ptr(), o["size"].data_ptr(),
        o["klen"].data_ptr(), o["list_cat"].data_ptr(), o["pops"].data_ptr(), o["best_fit"].data_ptr(),
        o["best_ref"].data_ptr(), o["best_vec"].data_ptr(), o["flags"].data_ptr(), _stream()), "woa_prepare")
    return o


def raise_if_woa_flagged(flags) -> None:
    """Raises naming every instance whose ``woa_prepare`` flags are set: the host path raises for them too, or (flag 8)
    the request is one the device stage does not take."""
    import numpy as np
    f = np.asarray(flags.cpu() if torch.is_tensor(flags) else flags)
    bad = np.nonzero(f)[0]
    if len(bad):
        why = "; ".join(f"{msg}: instances {np.nonzero(f & bit)[0].tolist()}" for bit, msg in WOA_FLAGS.items()
                        if (f & bit).any())
        raise GnnpnError(f"ESWOA stage cannot run {len(bad)} instance(s) of the batch: {why}")


def select_candidates(scores, svc_qos, cat_ptr, local_bounds, used, global_bounds, N: int, with_category: bool = False,
                      return_picked: bool = False, max_category_size: Optional[int] = None):
    """ML scores ``[n, S]`` -> PN input rows ``[n, K*N, 8(+1)]`` (see ``gnnpn_select_candidates_f32``).
    ``max_category_size``: the largest category (static per dataset); None reads it from ``cat_ptr`` -- one host sync."""
    if not (scores.is_cuda and scores.dtype == torch.float32 and scores.stride(1) == 1):
        scores = _f32(scores, "scores")                    # rows may be padded (stride(0) > S): no copy then
    n, S = scores.shape
    K = cat_ptr.numel() - 1
    svc_qos = _f32(svc_qos, "svc_qos")
    assert svc_qos.shape == (S, 4) and local_bounds.shape == (n, K, 4) and used.shape == (n, K)
    cat_ptr = cat_ptr.to(torch.int32).contiguous()
    if max_category_size is None:
        max_category_size = int((cat_ptr[1:] - cat_ptr[:-1]).max().item())
    max_size = int(max_category_size)
    rows = torch.empty(n, K * N, 9 if with_category else 8, device=scores.device, dtype=torch.float32)
    picked = torch.empty(n, K * N, device=scores.device, dtype=torch.int32) if return_picked else None
    check(lib().gnnpn_select_candidates_f32(
        scores.data_ptr(), scores.stride(0), svc_qos.data_ptr(), cat_ptr.data_ptr(), max_size,
        _f32(local_bounds, "local_bounds").data_ptr(), used.to(torch.uint8).contiguous().data_ptr(),
        _f32(global_bounds, "global_bounds").data_ptr(), n, K, N, int(with_category), rows.data_ptr(), _ptr(picked),
        _stream()), "select_candidates")
    return (rows, picked) if return_picked else rows


# ------------------------------------------------------------------ graph ops
def csr_build(edge_index: torch.Tensor, edge_weight: Optional[torch.Tensor], n_nodes: int, mode: int = CSR_PLAIN):
    """Destination-major CSR, stable in edge order.  Returns (rowptr int64 [n+1], col int32 [nnz], val fp32 [nnz] | None)."""
    if not edge_index.is_cuda:
        raise RuntimeError("csr_build: expected CUDA tensors")
    ei = edge_index.to(torch.int64).contiguous()
    E = ei.shape[1]
    w = None if edge_weight is None else _f32(edge_weight, "edge_weight")
    dev = ei.device
    cap = E + (n_nodes if mode == CSR_GCN_NORM else 0)
    rowptr = torch.empty(n_nodes + 1, device=dev, dtype=torch.int64)
    col = torch.empty(max(cap, 1), device=dev, dtype=torch.int32)
    need_val = mode == CSR_GCN_NORM or w is not None
    val = torch.empty(max(cap, 1), device=dev, dtype=torch.float32) if need_val else None
    nnz = torch.zeros(1, device=dev, dtype=torch.int64)
    import ctypes
    nbytes = ctypes.c_size_t(0)
    check(lib().gnnpn_csr_build_workspace_bytes(n_nodes, E, mode, ctypes.byref(nbytes)), "csr_workspace")
    ws = torch.empty(nbytes.value, device=dev, dtype=torch.uint8)
    check(lib().gnnpn_csr_build(ei.data_ptr(), _ptr(w), E, n_nodes, mode, rowptr.data_ptr(), col.data_ptr(),
                                _ptr(val), nnz.data_ptr(), ws.data_ptr(), nbytes.value, _stream()), "csr_build")
    # plain mode adds nothing (no self loops): every valid edge is one entry, and entries with an out-of-range endpoint sort
    # behind rowptr[n] where no kernel reads them -- the count is E without asking the device.  gcn_norm's count depends on
    # the self loops already present: one 8-byte read (the static service graph is built once and cached).
    total = E if mode == CSR_PLAIN else int(nnz.item())
    return rowptr, col[:total], (None if val is None else val[:total])


def embed_concat(x: torch.Tensor, table: torch.Tensor, pad_to: int = 4) -> torch.Tensor:
    """``cat(table[x[:,0].long()], x[:,1:])`` zero-padded to a multiple of ``pad_to`` columns."""
    x = _f32(x, "x")
    table = _f32(table, "table")
    n, C = x.shape
    rows, E = table.shape
    ld = (E + C - 1 + pad_to - 1) // pad_to * pad_to
    out = torch.empty(n, ld, device=x.device, dtype=torch.float32)
    check(lib().gnnpn_embed_concat_f32(x.data_ptr(), n, C, table.data_ptr(), rows, E, out.data_ptr(), ld, _stream()),
          "embed_concat")
    return out


def spmm_csr(rowptr, col, val, x, n_rows: Optional[int] = None, self_scale: float = 0.0, mean: bool = False,
             bias=None, scale=None, shift=None, act=None, out=None, long_row_threshold: Optional[int] = None) -> torch.Tensor:
    """CSR aggregation (``gnnpn_spmm_csr_f32``).  ``long_row_threshold``: rows with more edges are split into chunks (hub
    destinations of a skewed graph); None = the library's choice by edge count and feature width; 0 = never split."""
    x = _f32(x, "x")
    F = x.shape[1]
    assert F % 4 == 0, "feature dim must be padded to a multiple of 4"
    n_rows = rowptr.numel() - 1 if n_rows is None else n_rows
    y = torch.empty(n_rows, F, device=x.device, dtype=torch.float32) if out is None else out
    nnz = int(col.numel())
    T = -1 if long_row_threshold is None else int(long_row_threshold)
    need = int(lib().gnnpn_spmm_csr_workspace_bytes(nnz, F, T))
    ws = torch.empty(need, device=x.device, dtype=torch.uint8) if need > 0 else None
    check(lib().gnnpn_spmm_csr_f32(rowptr.data_ptr(), col.data_ptr(), _ptr(val), x.data_ptr(), x.stride(0), y.data_ptr(),
                                   y.stride(0), n_rows, nnz, F, float(self_scale), int(mean), _ptr(bias), _ptr(scale),
                                   _ptr(shift), ACT[act], T, _ptr(ws), need, _stream()), "spmm_csr")
    return y


def gemm_bias_act(a, w, bias=None, scale=None, shift=None, act=None, out=None, impl: Optional[str] = None,
                  pad_ld: bool = False) -> torch.Tensor:
    """``act((a @ w.T + bias) * scale + shift)`` with ``w`` in nn.Linear layout [N,K].

    ``impl="tc"`` (default for M >= TC_GEMM_MIN_ROWS): the tensor-core kernels -- the persistent 3xFP16 node transform
    for K, N <= 256 (K % 4 == 0, N % 16 == 0, a 16-byte aligned with a.stride(0) % 4 == 0; inputs outside its fp16 range
    are recomputed in strict fp32), 3xTF32 for other shapes, and strict fp32 for a misaligned ``a`` of a node-transform
    shape.  ``"ffma"``: strict fp32 CUDA cores.
    ``pad_ld``: allocate the result with rows padded to a multiple of 8 floats and return the ``[:, :N]`` view (row stride
    != N): the tensor-core epilogue then writes whole 32-byte sectors -- for wide outputs whose N is not a multiple of 8."""
    a = _f32(a, "a")
    w = _f32(w, "w")
    M, K = a.shape
    N = w.shape[0]
    assert w.shape[1] == K
    if out is not None:
        c = out
    elif pad_ld and N % 8:
        c = torch.empty(M, (N + 7) // 8 * 8, device=a.device, dtype=torch.float32)[:, :N]
    else:
        c = torch.empty(M, N, device=a.device, dtype=torch.float32)
    impl = impl or (DEFAULT_IMPL if M >= TC_GEMM_MIN_ROWS else "ffma")
    ws = None
    if impl == "tc":
        ws = torch.empty(int(lib().gnnpn_gemm_workspace_bytes(M, N, K)), device=a.device, dtype=torch.uint8)
    check(lib().gnnpn_gemm_f32_bias_act(a.data_ptr(), a.stride(0), w.data_ptr(), w.stride(0), _ptr(bias),
                                        _ptr(scale), _ptr(shift), ACT[act], c.data_ptr(), c.stride(0),
                                        M, N, K, *_ws(ws), _stream()), "gemm_bias_act")
    return c


# ------------------------------------------------------------------ train-mode BatchNorm (+ReLU)
def bn_train_forward(y, gamma, beta, eps: float, momentum: float, relu: bool, running_mean=None, running_var=None):
    """-> (out [M,C], save_mean [C], save_rstd [C]); running statistics are updated in place (torch semantics)."""
    y = _f32(y, "y")
    M, Cc = y.shape
    out = torch.empty_like(y)
    mean = torch.empty(Cc, device=y.device, dtype=torch.float32)
    rstd = torch.empty(Cc, device=y.device, dtype=torch.float32)
    check(lib().gnnpn_bn_train_forward_f32(y.data_ptr(), y.stride(0), M, Cc, _ptr(gamma), _ptr(beta), float(eps),
                                           float(momentum), int(bool(relu)), out.data_ptr(), out.stride(0),
                                           mean.data_ptr(), rstd.data_ptr(), _ptr(running_mean), _ptr(running_var),
                                           _stream()), "bn_train_forward")
    return out, mean, rstd


def bn_train_backward(y, out, dout, gamma, mean, rstd, relu: bool):
    """-> (dx [M,C], dgamma [C], dbeta [C])."""
    dout = _f32(dout, "dout")
    M, Cc = y.shape
    dx = torch.empty_like(y)
    dg = torch.empty(Cc, device=y.device, dtype=torch.float32)
    db = torch.empty(Cc, device=y.device, dtype=torch.float32)
    check(lib().gnnpn_bn_train_backward_f32(y.data_ptr(), y.stride(0), out.data_ptr(), out.stride(0), dout.data_ptr(),
                                            dout.stride(0), M, Cc, _ptr(gamma), mean.data_ptr(), rstd.data_ptr(),
                                            int(bool(relu)), dx.data_ptr(), dx.stride(0), dg.data_ptr(), db.data_ptr(),
                                            _stream()), "bn_train_backward")
    return dx, dg, db
