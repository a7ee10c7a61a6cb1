"""CPU suite: hidden sizes that are not a multiple of 128 run at Hp = 128 * ceil(H / 128) device units with zero padding
(ctc_pytorch_b200/model.py: device_hidden, unit_cols, _gate_row_perm; DESIGN.md §3.2).

Two levels, neither needs a GPU:
- the padding argument itself, in float64 torch layers built through the product's index maps: the padded layer reproduces the
  unpadded one (to float64 round-off), its padding units stay exactly zero and so does every gradient entry that touches them;
- the host-side orchestration of a padded model against the torch-CPU emulation of the C ABI (tests/emu_lib.py, extended here by
  the padded packing entry point, restated as "pack the zero-padded torch weights at Hp") and the oracle, in every mode.
"""
import pytest
import torch
import torch.nn as nn

from ctc_pytorch_b200 import synth
from ctc_pytorch_b200.model import CTC_Model, _gate_row_perm, check_hidden, device_hidden, unit_cols
from oracle import model_ref, packed_ref
from tests import emu_lib
from tests.emu_lib import emulated

HIDDEN = [1, 50, 200, 300, 700]
CELLS = [(nn.LSTM, {}), (nn.GRU, {}), (nn.RNN, {"nonlinearity": "tanh"}), (nn.RNN, {"nonlinearity": "relu"})]


def _gates(rnn_type):
    return {nn.LSTM: 4, nn.GRU: 3, nn.RNN: 1}[rnn_type]


def _pad_weight(w, H, Hp, G, in_cols=None, in_width=None):
    """torch weight [G*H, K] -> [G*Hp, K'] with the rows of unit u of gate g at g*Hp + u (unit_cols over G gate blocks) and
    the columns at in_cols (None: columns unchanged)."""
    rows = unit_cols(H, Hp, G, "cpu")
    K = w.shape[1] if in_cols is None else in_width
    out = torch.zeros(G * Hp, K, dtype=w.dtype)
    cidx = torch.arange(w.shape[1]) if in_cols is None else in_cols
    out[rows.view(-1, 1), cidx.view(1, -1)] = w
    return out


def _stack(rnn_type, kw, F, H, D, dtype=torch.float64):
    return [rnn_type(F, H, bidirectional=D == 2, bias=False, **kw).to(dtype),
            rnn_type(D * H, H, bidirectional=D == 2, bias=False, **kw).to(dtype)]


@pytest.mark.parametrize("H", HIDDEN)
@pytest.mark.parametrize("cell", range(len(CELLS)))
def test_zero_padding_is_exact_float64(H, cell):
    rnn_type, kw = CELLS[cell]
    G = _gates(rnn_type)
    T, N, F, D = 5, 3, 7, 2
    Hp = device_hidden(H)
    assert Hp % 128 == 0 and H <= Hp < H + 128
    torch.manual_seed(H + 17 * cell)
    ref = _stack(rnn_type, kw, F, H, D)
    pad = _stack(rnn_type, kw, F, Hp, D)
    cols = unit_cols(H, Hp, D, "cpu")
    with torch.no_grad():
        for li, (r, p) in enumerate(zip(ref, pad)):
            for sfx in ("", "_reverse"):
                wi, wh = getattr(r, "weight_ih_l0" + sfx), getattr(r, "weight_hh_l0" + sfx)
                getattr(p, "weight_ih_l0" + sfx).copy_(
                    _pad_weight(wi, H, Hp, G) if li == 0 else _pad_weight(wi, H, Hp, G, cols, D * Hp))
                getattr(p, "weight_hh_l0" + sfx).copy_(_pad_weight(wh, H, Hp, G, torch.arange(H), Hp))
    x = torch.randn(T, N, F, dtype=torch.float64)
    y_ref = ref[1](ref[0](x)[0])[0]
    y_pad = pad[1](pad[0](x)[0])[0]
    # the real units: the unpadded layer (to float64 round-off: BLAS sums the longer K = Hp products in another order, the
    # added terms themselves are exact zeros)
    assert torch.allclose(y_pad[..., cols], y_ref, rtol=1e-12, atol=1e-15)
    pad_mask = torch.ones(D * Hp, dtype=torch.bool)
    pad_mask[cols] = False
    assert (y_pad[..., pad_mask] == 0).all()                          # the padding units: exactly zero
    # backward: the same upstream gradient on the real units, none on the padding (the next layer's / fc's zero columns)
    g = torch.randn(T, N, D * H, dtype=torch.float64)
    gp = torch.zeros(T, N, D * Hp, dtype=torch.float64)
    gp[..., cols] = g
    (y_ref * g).sum().backward()
    (y_pad * gp).sum().backward()
    rows = unit_cols(H, Hp, G, "cpu")
    for li, (r, p) in enumerate(zip(ref, pad)):
        for name, rp in r.named_parameters():
            gpad = dict(p.named_parameters())[name].grad
            kc = (cols if (li > 0 and "ih" in name) else torch.arange(H) if "hh" in name else torch.arange(gpad.shape[1]))
            got = gpad[rows.view(-1, 1), kc.view(1, -1)]
            assert torch.allclose(got, rp.grad, rtol=1e-12, atol=1e-12), (li, name)
            rest = gpad.clone()
            rest[rows.view(-1, 1), kc.view(1, -1)] = 0
            assert (rest == 0).all(), (li, name)                      # every padded row / column: exactly zero


@pytest.mark.parametrize("H", HIDDEN)
def test_gate_row_gather_works_at_the_padded_size(H):
    """_gate_row_perm(H) picks torch row g*H + u out of a product whose rows follow the kernels' packed gate order at Hp."""
    Hp = device_hidden(H)
    perm = _gate_row_perm(H, torch.device("cpu"))
    packed_to_torch_at_hp = torch.tensor([emu_lib._orig_row(p, Hp) for p in range(4 * Hp)])
    want = unit_cols(H, Hp, 4, "cpu")                                  # g*Hp + u in the padded torch order
    assert torch.equal(packed_to_torch_at_hp[perm], want)


def test_hidden_size_limits():
    assert check_hidden(1, False) == 128 and check_hidden(768, False) == 768 and check_hidden(1000, False) == 1024
    assert check_hidden(520, True) == 640
    with pytest.raises(RuntimeError, match="x3"):
        check_hidden(700, True)
    with pytest.raises(RuntimeError, match="up to 1024"):
        check_hidden(1025, False)


# ---- the padded model's orchestration against the emulated C ABI and the oracle -------------------------------------------
def _emu_pack_padded(self, wih_f, whh_f, wih_r, whh_r, wih_p, wihT_p, whh_p, whhT_p, H, Hp, I, i_blk, i_blk_p, Ipad, part,
                     gates, stream):
    """ctcb200_pack_lstm_weights_padded restated: the unpadded packing of the zero-padded torch weights at Hp."""
    icols = (torch.arange(I) // i_blk) * i_blk_p + torch.arange(I) % i_blk
    I_dev = (I // i_blk) * i_blk_p
    pw = [_pad_weight(w.detach(), H, Hp, gates, icols, I_dev) for w in (wih_f, wih_r)]
    ph = [_pad_weight(w.detach(), H, Hp, gates, torch.arange(H), Hp) for w in (whh_f, whh_r)]
    self.pack_lstm_weights(pw[0], ph[0], pw[1], ph[1], wih_p, wihT_p, whh_p, whhT_p, Hp, I_dev, Ipad, part, gates, stream)


@pytest.fixture
def emu_padded(monkeypatch):
    monkeypatch.setattr(emu_lib.Emu, "pack_lstm_weights_padded", _emu_pack_padded, raising=False)


def _relnorm(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / (b.norm() + 1e-30))


def _ctc(out, tg, il, tl, N):
    return nn.CTCLoss(reduction="sum")(out, tg, il, tl) / N


@pytest.mark.parametrize("H,precision,rnn_type,nonlin,bidir,bn,p_drop", [
    (50, "x3", nn.LSTM, None, True, True, 0.0),
    (200, "x3", nn.LSTM, None, True, True, 0.25),
    (200, "x3", nn.LSTM, None, False, True, 0.25),
    (50, "x3", nn.GRU, None, True, True, 0.0),
    (50, "x3", nn.RNN, "relu", True, False, 0.0),
    (1, "x3", nn.LSTM, None, True, True, 0.0),
    (200, "bf16", nn.LSTM, None, True, True, 0.0),
])
def test_padded_model_orchestration(emu_padded, H, precision, rnn_type, nonlin, bidir, bn, p_drop):
    T, N, F, L, C = 9, 3, 24, 3, 7
    torch.manual_seed(H)
    rnn_param = {"rnn_input_size": F, "rnn_hidden_size": H, "rnn_layers": L, "rnn_type": rnn_type, "bidirectional": bidir,
                 "batch_norm": bn}
    m = CTC_Model(rnn_param=rnn_param, num_class=C, drop_out=p_drop)
    ref = model_ref.RefAcousticModel(F, H, L, C, batch_norm=bn, dropout=p_drop, bidirectional=bidir, rnn_type=rnn_type)
    if nonlin == "relu":
        for model_ in (m, ref):
            for blk in model_.rnns.children():
                old = blk.rnn
                blk.rnn = nn.RNN(input_size=old.input_size, hidden_size=H, bidirectional=bidir, bias=False, nonlinearity="relu")
    ref.load_state_dict(m.state_dict())
    m.precision, m.overlap_wgrad = precision, False
    masks = []
    gen = torch.Generator().manual_seed(5)

    def source(shape, p_, dev):
        k = (torch.rand(shape, generator=gen) >= p_).to(torch.uint8)
        masks.append(k)
        return k
    m.mask_source = source
    x, frac, tg, tl = synth.synthetic_batch(T, N, F, C, 3, 7)
    il = (frac * T).long()
    m.train(); ref.train()
    with emulated():
        xm = x.clone().requires_grad_(True)
        out = m(xm)
        loss = _ctc(out, tg, il, tl, N)
        loss.backward()
    if p_drop > 0:
        assert len(masks) == L and all(k.shape == (T * N, (2 if bidir else 1) * H) for k in masks)   # torch's shape
        for blk, k in zip(ref.rnns.children(), masks):
            blk.fixed_mask = k
    xr = x.clone().requires_grad_(True)
    rout = ref(xr)
    rloss = _ctc(rout, tg, il, tl, N)
    rloss.backward()
    rp, rb = dict(ref.named_parameters()), dict(ref.named_buffers())
    for k, p in m.named_parameters():
        assert p.grad.shape == p.shape == rp[k].shape, k
    worst = max(_relnorm(p.grad, rp[k].grad) for k, p in m.named_parameters())
    e_loss = abs(loss.item() - rloss.item()) / abs(rloss.item())
    if precision == "x3":
        assert e_loss < 1e-5 and worst < 3e-4 and _relnorm(xm.grad, xr.grad) < 3e-4, (e_loss, worst)
    else:
        assert e_loss < 2e-3 and worst < 3e-2, (e_loss, worst)
    for k, b in m.named_buffers():
        assert b.shape == rb[k].shape, k
        if "running" in k:
            assert _relnorm(b, rb[k]) < (1e-4 if precision == "x3" else 2e-2), k


@pytest.mark.parametrize("precision", ["x3", "bf16"])
def test_padded_packed_model_orchestration(emu_padded, precision):
    from ctc_pytorch_b200.packed import CTC_RNN
    T, N, F_, H, L, C = 12, 4, 24, 60, 3, 9
    torch.manual_seed(6)
    m = CTC_RNN(rnn_input_size=F_, rnn_hidden_size=H, rnn_layers=L, rnn_type=nn.LSTM, bidirectional=True, batch_norm=True,
                num_class=C, drop_out=0.0)
    ref = packed_ref.RefPackedModel(F_, H, L, True, C)
    ref.load_state_dict(m.state_dict())
    m.precision = precision
    x, lens, targets, tsz = packed_ref.synthetic_packed_batch(T, N, F_, C, 3, 8)
    m.train(); ref.train()
    with emulated():
        act = m(nn.utils.rnn.pack_padded_sequence(x, lens))
        loss = packed_ref.warp_ctc_loss(act, targets, lens, tsz)
        loss.backward()
    ract = ref(x, lens)
    rloss = packed_ref.warp_ctc_loss(ract, targets, lens, tsz)
    rloss.backward()
    rp = dict(ref.named_parameters())
    worst = max(_relnorm(p.grad, rp[k].grad) for k, p in m.named_parameters())
    tol = (1e-5, 3e-4) if precision == "x3" else (2e-3, 3e-2)
    assert abs(loss.item() - rloss.item()) < tol[0] * abs(rloss.item()) and worst < tol[1], worst


@pytest.mark.parametrize("precision", ["x3", "bf16"])
def test_padded_model_equals_the_zero_padded_model_bitwise(emu_padded, precision):
    """A model at H = 200 and one at H = 256 holding the same weights zero-padded run the same emulated launches on the same
    operands: identical log-probs, loss and real-part gradients, bit for bit."""
    T, N, F, L, C, H, Hp = 8, 3, 24, 2, 7, 200, 256
    torch.manual_seed(11)

    def make(h):
        return CTC_Model(rnn_param={"rnn_input_size": F, "rnn_hidden_size": h, "rnn_layers": L, "rnn_type": nn.LSTM,
                                    "bidirectional": True, "batch_norm": True}, num_class=C, drop_out=0.0)
    a, b = make(H), make(Hp)
    cols = unit_cols(H, Hp, 2, "cpu")
    sa = a.state_dict()
    sb = {}
    for k, v in b.state_dict().items():
        w = sa[k]
        if "rnn.weight_ih" in k:
            sb[k] = _pad_weight(w, H, Hp, 4) if k.startswith("rnns.0.") else _pad_weight(w, H, Hp, 4, cols, 2 * Hp)
        elif "rnn.weight_hh" in k:
            sb[k] = _pad_weight(w, H, Hp, 4, torch.arange(H), Hp)
        elif k == "fc.1.weight":
            sb[k] = torch.zeros_like(v).index_copy_(1, cols, w)
        elif v.dim() == 1 and v.numel() == 2 * Hp:
            fill = 1.0 if k.endswith("running_var") else 0.0
            sb[k] = torch.full_like(v, fill).index_copy_(0, cols, w)
        else:
            sb[k] = w.clone()
    b.load_state_dict(sb)
    x, frac, tg, tl = synth.synthetic_batch(T, N, F, C, 3, 2)
    il = (frac * T).long()
    res = []
    for m in (a, b):
        m.precision, m.overlap_wgrad = precision, False
        m.train()
        with emulated():
            out = m(x)
            loss = _ctc(out, tg, il, tl, N)
            loss.backward()
        res.append((out.detach(), loss.detach(), {k: p.grad for k, p in m.named_parameters()}))
    assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][1], res[1][1])
    for k, ga in res[0][2].items():
        gb = res[1][2][k]
        if "rnn.weight_ih" in k:
            gb = gb[unit_cols(H, Hp, 4, "cpu")] if k.startswith("rnns.0.") else gb[unit_cols(H, Hp, 4, "cpu")][:, cols]
        elif "rnn.weight_hh" in k:
            gb = gb[unit_cols(H, Hp, 4, "cpu")][:, :H]
        elif k == "fc.1.weight":
            gb = gb[:, cols]
        elif gb.dim() == 1 and gb.numel() == 2 * Hp:
            gb = gb[cols]
        assert torch.equal(ga, gb), k
