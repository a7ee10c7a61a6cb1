"""GPU suite (`-m gpu`): recurrent hidden sizes outside the multiples of 128 up to 640 (DESIGN.md §3.2, §9).

- the recurrent kernels at device hidden sizes 768 / 896 / 1024 (global exchange; at 1024 the weight slice is split between
  tensor memory and shared memory) against a float64 recurrence and its autograd BPTT, for every cell;
- CTC_Model / CTC_RNN at padded and large hidden sizes against the oracle, at the bf16 / x3 tolerances of DESIGN.md §4;
- zero padding is exact on the device: a model at H = 200 and one at H = 256 holding the same weights zero-padded produce the
  same bits;
- the public surface: torch-shaped state_dict / gradients, checkpoints, an optimizer, the documented x3 limit.
"""
import io

import pytest
import torch
import torch.nn as nn

from oracle import model_ref, packed_ref
from tests.test_hidden_pad_host import _pad_weight

pytestmark = pytest.mark.gpu

DEV = "cuda"


@pytest.fixture(scope="module", autouse=True)
def _need_cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from ctc_pytorch_b200 import _lib
    _lib.lib()


def relnorm(a, b):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


# ---- kernels vs float64 ---------------------------------------------------------------------------------------------------
def _recurrence_fp64(gx, W, T, N, H, cell):
    """hout [T*N, 2H] of the bias-free bidirectional recurrence in float64 from the packed pre-activations gx [T*N, 8H] and the
    torch-ordered recurrent weights W[d] [G*H, H]; differentiable w.r.t. gx (its gradient is the kernels' dG)."""
    from ctc_pytorch_b200.model import _gate_row_perm
    G = W[0].shape[0] // H
    perm = _gate_row_perm(H, gx.device)[:G * H]
    outs = []
    for d in range(2):
        g = gx[:, d * 4 * H + perm].view(T, N, G * H)
        h = torch.zeros(N, H, dtype=torch.float64, device=gx.device)
        c = torch.zeros_like(h)
        hs = [None] * T
        for t in (range(T) if d == 0 else range(T - 1, -1, -1)):
            rec = h @ W[d].t()
            if cell == 0:
                i, f, gg, o = (g[t] + rec).split(H, 1)
                c = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(gg)
                h = torch.sigmoid(o) * torch.tanh(c)
            elif cell == 1:
                gr, gz, gn = g[t].split(H, 1)
                rr, rz, rn = rec.split(H, 1)
                r, z = torch.sigmoid(gr + rr), torch.sigmoid(gz + rz)
                h = (1 - z) * torch.tanh(gn + r * rn) + z * h
            else:
                h = torch.relu(g[t] + rec) if cell == 3 else torch.tanh(g[t] + rec)
            hs[t] = h
        outs.append(torch.stack(hs, 0))
    return torch.cat(outs, -1).reshape(T * N, 2 * H)


@pytest.mark.parametrize("H", [768, 896, 1024])
@pytest.mark.parametrize("N", [4, 21])
@pytest.mark.parametrize("cell", [0, 1, 2])
def test_recurrent_kernels_vs_fp64(H, N, cell):
    from ctc_pytorch_b200 import _lib
    L = _lib.lib()
    G = (4, 3, 1, 1)[cell]
    T, I = 6, 8
    R = T * N
    torch.manual_seed(H + N + cell)
    wih = [0.2 * torch.randn(G * H, I, device=DEV) for _ in range(2)]
    whh = [(0.7 / H ** 0.5) * torch.randn(G * H, H, device=DEV) for _ in range(2)]
    wih_p = torch.empty(8 * H, I, dtype=torch.bfloat16, device=DEV)
    wihT_p = torch.empty(I, 8 * H, dtype=torch.bfloat16, device=DEV)
    whh_p = torch.empty(8 * H, H, dtype=torch.bfloat16, device=DEV)
    whhT_p = torch.empty(8 * H, H, dtype=torch.bfloat16, device=DEV)
    L.call("ctcb200_pack_lstm_weights", _lib.ptr(wih[0]), _lib.ptr(whh[0]), _lib.ptr(wih[1]), _lib.ptr(whh[1]),
           _lib.ptr(wih_p), _lib.ptr(wihT_p), _lib.ptr(whh_p), _lib.ptr(whhT_p), H, I, I, 0, G, _lib.stream())
    gx = torch.randn(R, 8 * H, device=DEV)
    scratch = torch.empty(L.dll.ctcb200_lstm_scratch_bytes(N, H), dtype=torch.uint8, device=DEV)
    hout = torch.zeros(R, 2 * H, device=DEV)
    c_save = torch.zeros(R, 2 * H, device=DEV)
    gates = torch.zeros(R, 2 * H, 4, dtype=torch.float16, device=DEV)
    L.call("ctcb200_lstm_fwd", _lib.ptr(gx), _lib.ptr(whh_p), None, _lib.ptr(hout), _lib.ptr(c_save), _lib.ptr(gates),
           _lib.ptr(scratch), T, N, H, 0, cell, _lib.stream())
    dh = torch.randn(R, 2 * H, device=DEV)
    dg = torch.zeros(R, 8 * H, dtype=torch.bfloat16, device=DEV)
    dg_rec = torch.zeros(R, 8 * H, dtype=torch.bfloat16, device=DEV) if cell == 1 else None
    L.call("ctcb200_lstm_bwd", _lib.ptr(dh), _lib.ptr(whhT_p), None, _lib.ptr(c_save), _lib.ptr(gates), _lib.ptr(dg), None,
           _lib.ptr(dg_rec), None, _lib.ptr(scratch), T, N, H, 0, cell, None, None, None, None, _lib.stream())
    torch.cuda.synchronize()
    # the reference sees the bf16 weights the kernels hold
    W = [w.to(torch.bfloat16).double() for w in whh]
    gx64 = gx.double().requires_grad_(True)
    ref = _recurrence_fp64(gx64, W, T, N, H, cell)
    (ref * dh.double()).sum().backward()
    e_h = relnorm(hout, ref.detach())
    e_g = relnorm(dg.float(), gx64.grad)
    print("HIDDEN_KERNEL", dict(H=H, N=N, cell=cell, hout_rel_l2=e_h, dg_rel_l2=e_g))
    assert e_h < 1e-2 and e_g < 3e-2, (e_h, e_g)


# ---- model vs oracle ------------------------------------------------------------------------------------------------------
# H = 1 runs in x3 mode: a one-unit layer's weight gradients are sums with heavy cancellation over the frames, where bf16 operand
# rounding alone reaches ~3e-2 (measured 3.3e-2 on one matrix); that padding adds no error of its own is what
# test_padded_model_is_bitwise_the_zero_padded_model shows. The ReLU RNN runs in x3 mode for the same reason: without BatchNorm
# its gradients through three unbounded layers amplify the bf16 rounding (measured 8e-2 at H = 1000).
MODEL_CASES = [
    # H, precision, rnn_type, nonlinearity, bidirectional, batch_norm, dropout
    (200, "bf16", nn.LSTM, None, True, True, 0.2),
    (300, "bf16", nn.GRU, None, True, True, 0.0),
    (700, "bf16", nn.LSTM, None, False, True, 0.0),
    (768, "bf16", nn.LSTM, None, True, True, 0.2),
    (1000, "bf16", nn.RNN, None, True, False, 0.0),
    (1024, "bf16", nn.LSTM, None, True, False, 0.0),
    (1024, "bf16", nn.GRU, None, True, True, 0.0),
    (1, "x3", nn.LSTM, None, True, True, 0.0),
    (50, "x3", nn.LSTM, None, True, True, 0.2),
    (200, "x3", nn.GRU, None, False, True, 0.0),
    (200, "x3", nn.RNN, "relu", True, False, 0.0),
    (520, "x3", nn.LSTM, None, True, False, 0.0),
]


@pytest.mark.parametrize("H,precision,rnn_type,nonlin,bidir,bn,p_drop", MODEL_CASES)
def test_model_vs_oracle_any_hidden(H, precision, rnn_type, nonlin, bidir, bn, p_drop):
    from ctc_pytorch_b200.model import CTC_Model
    from ctc_pytorch_b200.loss import CTCLoss
    T, N, F, L, C = 16, 5, 40, 3, 12
    torch.manual_seed(H + L)
    rnn_param = {"rnn_input_size": F, "rnn_hidden_size": H, "rnn_layers": L, "rnn_type": rnn_type, "bidirectional": bidir,
                 "batch_norm": bn}
    m = CTC_Model(rnn_param=rnn_param, num_class=C, drop_out=p_drop)
    ref = model_ref.RefAcousticModel(F, H, L, C, batch_norm=bn, dropout=p_drop, bidirectional=bidir, rnn_type=rnn_type)
    if nonlin == "relu":
        for model_ in (m, ref):
            for blk in model_.rnns.children():
                old = blk.rnn
                blk.rnn = nn.RNN(input_size=old.input_size, hidden_size=H, bidirectional=bidir, bias=False,
                                 nonlinearity="relu")
    ref.load_state_dict(m.state_dict())
    m = m.to(DEV)
    m.precision = precision
    gen = torch.Generator().manual_seed(99)
    masks = []

    def source(shape, p_, dev):
        k = (torch.rand(shape, generator=gen) >= p_).to(torch.uint8)
        masks.append(k)
        return k
    m.mask_source = source
    x, frac, tg, tl = model_ref.synthetic_batch(T, N, F, C, 5, H)
    il = (frac * T).long()
    m.train(); ref.train()
    out = m(x.to(DEV))
    loss = CTCLoss(reduction="sum")(out, tg.to(DEV), il.to(DEV), tl.to(DEV)) / N
    loss.backward()
    if p_drop > 0:
        assert len(masks) == L
        for blk, k in zip(ref.rnns.children(), masks):
            blk.fixed_mask = k
    rout = ref(x)
    rloss = nn.CTCLoss(reduction="sum")(rout, tg, il, tl) / N
    rloss.backward()
    tol_l, tol_g = (2e-3, 3e-2) if precision == "bf16" else (1e-4, 1e-3)
    e_loss = abs(loss.item() - rloss.item()) / abs(rloss.item())
    rp = dict(ref.named_parameters())
    errs = {k: relnorm(p.grad, rp[k].grad) for k, p in m.named_parameters()}
    print("HIDDEN_MODEL", dict(H=H, precision=precision, cell=rnn_type.__name__, loss_rel=e_loss,
                               grad_rel_l2_worst=max(errs.values())))
    assert e_loss < tol_l, e_loss
    for k, e in errs.items():
        assert e < tol_g, (k, e)


def test_packed_863_default_model_vs_oracle():
    """CTC_RNN() with the 863 recipe's defaults (rnn_hidden_size = 768, 5 layers) on a ragged PackedSequence batch."""
    from ctc_pytorch_b200.packed import CTC_RNN
    m = CTC_RNN()
    H, L, F_, C = m.rnn_hidden_size, m.rnn_layers, m.rnn_input_size, m.num_class
    assert (H, L) == (768, 5)
    torch.manual_seed(3)
    ref = packed_ref.RefPackedModel(F_, H, L, True, C)
    ref.load_state_dict(m.state_dict())
    m = m.to(DEV)
    T, N = 24, 6
    x, lens, targets, tsz = packed_ref.synthetic_packed_batch(T, N, F_, C, 4, 1)
    m.train(); ref.train()
    act = m(nn.utils.rnn.pack_padded_sequence(x.to(DEV), lens))
    from ctc_pytorch_b200.packed import WarpCTCLoss
    loss = WarpCTCLoss()(act, targets.to(DEV), lens, tsz)
    loss.backward()
    ract = ref(x, lens)
    rloss = packed_ref.warp_ctc_loss(ract, targets, lens, tsz)
    rloss.backward()
    for n, Ln in enumerate(lens):
        assert act[Ln:, n].abs().sum().item() == 0.0
    rp = dict(ref.named_parameters())
    worst = max(relnorm(p.grad, rp[k].grad) for k, p in m.named_parameters())
    e_loss = abs(loss.item() - rloss.item()) / abs(rloss.item())
    print("HIDDEN_863", dict(loss_rel=e_loss, grad_rel_l2_worst=worst))
    assert e_loss < 2e-3 and worst < 3e-2, (e_loss, worst)


# ---- zero padding is exact on the device -----------------------------------------------------------------------------------
def _make(H, F=40, L=2, C=12, rnn_type=nn.LSTM):
    from ctc_pytorch_b200.model import CTC_Model
    return CTC_Model(rnn_param={"rnn_input_size": F, "rnn_hidden_size": H, "rnn_layers": L, "rnn_type": rnn_type,
                                "bidirectional": True, "batch_norm": True}, num_class=C, drop_out=0.0)


@pytest.mark.parametrize("precision", ["bf16", "x3"])
def test_padded_model_is_bitwise_the_zero_padded_model(precision):
    """H = 200 runs at 256 device units; a model AT 256 whose weights are the H = 200 model's, zero-padded, runs the same
    launches on the same operands: log-probs, loss and the real part of every gradient agree bit for bit."""
    from ctc_pytorch_b200.loss import CTCLoss
    from ctc_pytorch_b200.model import unit_cols
    H, Hp, T, N, C = 200, 256, 30, 7, 12
    torch.manual_seed(21)
    a, b = _make(H), _make(Hp)
    cols = unit_cols(H, Hp, 2, "cpu")
    rows4 = unit_cols(H, Hp, 4, "cpu")
    sa, sb = a.state_dict(), {}
    for k, v in b.state_dict().items():
        w = sa[k]
        if "rnn.weight_ih" in k:
            sb[k] = _pad_weight(w, H, Hp, 4) if k.startswith("rnns.0.") else _pad_weight(w, H, Hp, 4, cols, 2 * Hp)
        elif "rnn.weight_hh" in k:
            sb[k] = _pad_weight(w, H, Hp, 4, torch.arange(H), Hp)
        elif k == "fc.1.weight":
            sb[k] = torch.zeros_like(v).index_copy_(1, cols, w)
        elif v.dim() == 1 and v.numel() == 2 * Hp:
            sb[k] = torch.full_like(v, 1.0 if k.endswith("running_var") else 0.0).index_copy_(0, cols, w)
        else:
            sb[k] = w.clone()
    b.load_state_dict(sb)
    x, frac, tg, tl = model_ref.synthetic_batch(T, N, 40, C, 5, 4)
    il = (frac * T).long()
    res = []
    for m in (a, b):
        m = m.to(DEV)
        m.precision = precision
        m.train()
        out = m(x.to(DEV))
        loss = CTCLoss(reduction="sum")(out, tg.to(DEV), il.to(DEV), tl.to(DEV)) / N
        loss.backward()
        res.append((out.detach().cpu(), loss.detach().cpu(), {k: p.grad.cpu() for k, p in m.named_parameters()}))
    assert torch.equal(res[0][0], res[1][0]), (res[0][0] - res[1][0]).abs().max()
    assert torch.equal(res[0][1], res[1][1])
    for k, ga in res[0][2].items():
        gb = res[1][2][k]
        if "rnn.weight_ih" in k:
            gb = gb[rows4] if k.startswith("rnns.0.") else gb[rows4][:, cols]
        elif "rnn.weight_hh" in k:
            gb = gb[rows4][:, :H]
        elif k == "fc.1.weight":
            gb = gb[:, cols]
        elif gb.dim() == 1 and gb.numel() == 2 * Hp:
            gb = gb[cols]
        assert torch.equal(ga, gb), (k, (ga - gb).abs().max())


# ---- public surface ---------------------------------------------------------------------------------------------------------
def test_state_dict_checkpoint_and_training_at_h200():
    from ctc_pytorch_b200.model import CTC_Model
    from ctc_pytorch_b200.loss import CTCLoss
    H, T, N, F, C = 200, 40, 8, 40, 12
    torch.manual_seed(5)
    m = _make(H).to(DEV)
    ref = model_ref.RefAcousticModel(F, H, 2, C, batch_norm=True)
    assert {k: v.shape for k, v in m.state_dict().items()} == {k: v.shape for k, v in ref.state_dict().items()}
    x, frac, tg, tl = model_ref.synthetic_batch(T, N, F, C, 5, 6)
    il = (frac * T).long()
    xd, tgd, ild, tld = x.to(DEV), tg.to(DEV), il.to(DEV), tl.to(DEV)
    opt = torch.optim.Adam(m.parameters(), lr=3e-3)
    losses = []
    m.train()
    for _ in range(6):
        opt.zero_grad()
        loss = CTCLoss(reduction="sum")(m(xd), tgd, ild, tld) / N
        loss.backward()
        for p in m.parameters():
            assert p.grad.shape == p.shape
        opt.step()
        losses.append(loss.item())
    assert losses[-1] < losses[0], losses
    # checkpoint round trip: a fresh model loaded from the package computes the same bits
    buf = io.BytesIO()
    torch.save(CTC_Model.save_package(m, optimizer=opt), buf)
    buf.seek(0)
    pkg = torch.load(buf, weights_only=False)
    m2 = CTC_Model(rnn_param=pkg["rnn_param"], num_class=pkg["num_class"], drop_out=pkg["_drop_out"]).to(DEV)
    m2.load_state_dict(pkg["state_dict"])
    m.eval(); m2.eval()
    with torch.no_grad():
        assert torch.equal(m(xd), m2(xd))


def test_x3_above_640_refuses_before_any_launch():
    from ctc_pytorch_b200 import _lib
    m = _make(700).to(DEV)
    m.precision = "x3"
    x = torch.randn(3, 10, 40, device=DEV)
    before = _lib.lib().launches
    with pytest.raises(RuntimeError, match="x3"):
        m(x)
    assert _lib.lib().launches == before
