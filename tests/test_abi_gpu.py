"""The C ABI itself on the GPU: argument validation (negative codes before any launch), empty and ragged batches,
the host-buffer entry point, determinism.  Calls go through ctypes exactly as a non-Python caller would bind them."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import pn_oracle as po

pytestmark = pytest.mark.gpu
K, N, H, F = 6, 4, 256, 8
L = K * N


def _packed(seed=3):
    from gnnpn_sc_b200 import ops
    cfg = po.PNConfig(seq_len=L, s_number=N, s_category=K)
    sd = {k: v.cuda() for k, v in po.make_state_dict(cfg, seed).items()}
    enc = ops.pack_lstm(sd["actor.encoder.weight_ih_l0"], sd["actor.encoder.weight_hh_l0"], sd["actor.encoder.bias_ih_l0"],
                        sd["actor.encoder.bias_hh_l0"], sd["actor.embedding2.weight"], sd["actor.embedding2.bias"])
    dec = ops.pack_lstm(sd["actor.decoder.weight_ih_l0"], sd["actor.decoder.weight_hh_l0"], sd["actor.decoder.bias_ih_l0"],
                        sd["actor.decoder.bias_hh_l0"], sd["actor.embedding2.weight"], sd["actor.embedding2.bias"],
                        sd["actor.decoder_start_input"])
    return enc, dec


def test_argument_errors_are_reported_before_any_launch():
    from gnnpn_sc_b200 import _lib
    lib = _lib.lib()
    enc, _ = _packed()
    n = 5
    x = torch.zeros(n, L, F, device="cuda")
    out = torch.empty(n, L, H, device="cuda")
    c = torch.empty(n, H, device="cuda")
    ws = torch.empty(lib.gnnpn_pn_workspace_bytes(n, H), dtype=torch.uint8, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    before = lib.gnnpn_launch_count()
    call = lambda **kw: lib.gnnpn_lstm_encode_f32(
        kw.get("x", x.data_ptr()), kw.get("n", n), L, kw.get("F", F), kw.get("H", H), enc.data_ptr(),
        kw.get("out", out.data_ptr()), c.data_ptr(), ws.data_ptr(), kw.get("wsb", ws.numel()), kw.get("layout", 0), st)
    assert call(x=None) == -1                                   # GNNPN_ENULL
    assert call(H=128) == -2                                    # GNNPN_ESHAPE: hidden_size != 256
    assert call(F=33) == -2                                     # more raw columns than the packed block holds
    assert call(out=out.data_ptr() + 4) == -3                   # GNNPN_EALIGN
    assert call(wsb=16) == -4                                   # GNNPN_EWORKSPACE
    assert call(n=1 << 31) == -5                                # GNNPN_ERANGE
    assert call(layout=7) == -2                                 # unknown encodings layout
    assert lib.gnnpn_launch_count() == before                   # nothing was launched
    assert call(n=0) == 0                                       # empty batch: success, no launch
    assert lib.gnnpn_launch_count() == before
    assert lib.gnnpn_error_string(-3).startswith(b"pointer")
    assert b"invalid" in lib.gnnpn_error_string(1).lower() or lib.gnnpn_error_string(1)   # positive = cudaError_t text
    torch.cuda.synchronize()


@pytest.mark.parametrize("n", [1, 127, 129, 257, 300])
def test_ragged_batches_equal_the_padded_batch(n):
    """A batch that does not fill its last CTA (pair) gives the same picks / logits as the same instances inside a
    bigger batch: no dependence on padding rows or on where an instance sits in its CTA."""
    from gnnpn_sc_b200 import modelPN as M
    from gnnpn_sc_b200.synth import pn_instances
    cfg = po.PNConfig(seq_len=L, s_number=N, s_category=K)
    m = M.CombinatorialRL(0, H, L, 0, 10, 1, M.reward, "Dot", N, K, level="Low")
    m.load_state_dict(po.make_state_dict(cfg, 9))
    m = m.cuda().eval()
    x = pn_instances(512, K, N, seed=2).cuda()
    with torch.no_grad():
        _, idx_all, lg_all = m.actor(x, None, sample="greedy")
        _, idx_n, lg_n = m.actor(x[:n], None, sample="greedy")
        _, idx_t, lg_t = m.actor(x[512 - n:], None, sample="greedy")        # same instances at other CTA rows
    assert torch.equal(torch.stack(idx_n), torch.stack(idx_all)[:, :n])
    assert torch.equal(lg_n.window, lg_all.window[:n])
    assert torch.equal(torch.stack(idx_t), torch.stack(idx_all)[:, 512 - n:])
    assert torch.equal(lg_t.window, lg_all.window[512 - n:])


def test_host_buffer_entry_point_equals_module_path():
    """gnnpn_pn_greedy_low_high_host (plain host pointers, what a non-torch caller binds) == the drop-in modules."""
    from gnnpn_sc_b200 import _lib, modelPN as M
    from gnnpn_sc_b200.synth import pn_instances
    lib = _lib.lib()
    cfg = po.PNConfig(seq_len=L, s_number=N, s_category=K)
    nets, packs = [], []
    for level, seed in (("Low", 1), ("High", 2)):
        m = M.CombinatorialRL(0, H, L, 0, 10, 1, M.reward, "Dot", N, K, level=level)
        m.load_state_dict(po.make_state_dict(cfg, seed))
        m = m.cuda().eval()
        nets.append(m)
        packs.append(torch.cat(m.actor._packed_weights()).cpu().contiguous())
    n = 9000                                                                 # > one 8192-instance chunk of the host entry
    x = pn_instances(n, K, N, seed=4)
    idx_lo = np.empty((K, n), dtype=np.int32)
    idx_hi = np.empty((K, n), dtype=np.int32)
    rew = np.empty(n, dtype=np.float32)
    xn = np.ascontiguousarray(x.numpy())
    rc = lib.gnnpn_pn_greedy_low_high_host(xn.ctypes.data, n, L, F, H, K, N, packs[0].data_ptr(), packs[1].data_ptr(),
                                           1, C.c_float(10.0), C.c_float(1.0), idx_lo.ctypes.data, idx_hi.ctypes.data,
                                           rew.ctypes.data)
    assert rc == 0
    with torch.no_grad():
        _, _, _, i_lo, lat = nets[0](x.cuda(), None, sample="greedy", training="SL")
        R, _, _, i_hi, _ = nets[1](x.cuda(), None, lat, sample="greedy", training="RL")
    assert np.array_equal(idx_lo, torch.stack(i_lo).cpu().numpy())
    assert np.array_equal(idx_hi, torch.stack(i_hi).cpu().numpy())
    # instances whose every category is neutral have no service with q0 > 0: 0/0 = nan in the reference's calc() too
    assert np.array_equal(rew, R.cpu().numpy(), equal_nan=True)


def test_argument_errors_of_the_anyh_and_training_forward_entry_points():
    """Any-hidden-size kernels and the training forward with saves (its workspace query and the refusals of
    gnnpn_pn_train_forward_f32): negative codes before any launch, n = 0 is a no-op."""
    from gnnpn_sc_b200 import _lib
    lib = _lib.lib()
    st = torch.cuda.current_stream().cuda_stream
    n, Hh = 5, 96
    x = torch.zeros(n, L, F, device="cuda")
    w = torch.zeros(4 * Hh, Hh + F, device="cuda")
    b = torch.zeros(4 * Hh, device="cuda")
    enc = torch.empty(n, L, Hh, device="cuda")
    c = torch.empty(n, Hh, device="cuda")
    wsf = lib.gnnpn_pn_anyh_workspace_floats(n, Hh, F)
    assert wsf == n * (Hh + F) + n * 4 * Hh
    ws = torch.empty(wsf, device="cuda")
    enc_p, dec_p = _packed()                                     # (two pack launches: before the counter is sampled)
    before = lib.gnnpn_launch_count()
    enc_call = lambda **kw: lib.gnnpn_lstm_encode_anyh_f32(
        kw.get("x", x.data_ptr()), kw.get("n", n), L, kw.get("F", F), kw.get("H", Hh), w.data_ptr(), b.data_ptr(),
        enc.data_ptr(), c.data_ptr(), ws.data_ptr(), kw.get("wsf", wsf), st)
    assert enc_call(x=None) == -1
    assert enc_call(H=0) == -2 and enc_call(F=33) == -2
    assert enc_call(wsf=8) == -4
    assert enc_call(n=0) == 0
    dec_h = torch.empty(n, K, Hh, device="cuda")
    idx = torch.empty(K, n, dtype=torch.int32, device="cuda")
    wl, wp = torch.empty(n, L, device="cuda"), torch.empty(n, L, device="cuda")
    dec_call = lambda **kw: lib.gnnpn_pn_decode_anyh_f32(
        x.data_ptr(), enc.data_ptr(), c.data_ptr(), None, C.c_float(1.0), w.data_ptr(), b.data_ptr(), kw.get("b0", b.data_ptr()),
        1, C.c_float(10.0), n, kw.get("L", L), F, Hh, kw.get("K", K), kw.get("N", N), dec_h.data_ptr(), idx.data_ptr(),
        wl.data_ptr(), wp.data_ptr(), None, None, ws.data_ptr(), wsf, st)
    assert dec_call(b0=None) == -1
    assert dec_call(K=1, N=40, L=40) == -2                       # windows wider than 32 need hidden_size = 256
    assert dec_call(K=5) == -2                                   # K * N != L
    assert lib.gnnpn_pn_full_logits_anyh_f32(enc.data_ptr(), dec_h.data_ptr(), None, 1, C.c_float(10.0), n, L, Hh, K,
                                             wl.data_ptr(), st) == -1
    # training forward: a batch beyond the column-split scan needs no workspace (the FFMA kernels replay forced picks);
    # a free-running call outside that scan, or without a workspace, is refused
    big = 8192
    assert lib.gnnpn_pn_train_forward_workspace_bytes(big, L, F, H, K, N) == 0
    wsb = lib.gnnpn_pn_train_forward_workspace_bytes(64, L, F, H, K, N)
    assert wsb > 0
    dummy = torch.empty(16, device="cuda")
    p = dummy.data_ptr()
    fwd = lambda n_, H_, ws_, wsb_: lib.gnnpn_pn_train_forward_f32(
        p, enc_p.data_ptr(), dec_p.data_ptr(), None, None, None, C.c_float(1.0), 1, C.c_float(10.0), n_, L, F, H_, K, N,
        p, p, p, p, p, p, p, p, p, ws_, wsb_, st)
    assert fwd(big, H, p, lib.gnnpn_pn_workspace_bytes(big, H)) == -6    # GNNPN_EUNSUPPORTED
    assert fwd(64, H, None, 0) == -6
    assert fwd(64, 128, p, wsb) == -2                                     # hidden_size != 256
    assert lib.gnnpn_launch_count() == before
    torch.cuda.synchronize()
