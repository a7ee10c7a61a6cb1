"""CPU suite: pins the oracle (oracle/*.py) against (a) the committed golden vectors generated from the
unmodified reference, (b) what the reference itself returned on the inputs of the `*_reference_live` tests
(tests/golden/reference_live.*, recorded by oracle/make_golden_live.py), (c) torch's own CPU kernels, which is where the
reference's arithmetic for the model and the loss lives."""
import json
import os

import numpy as np
import pytest
import torch
import torch.nn as nn

from oracle import ctc_ref, decode_ref, model_ref


@pytest.fixture(scope="module")
def reference_live(golden_dir):
    """(json, npz) of the reference's recorded answers."""
    meta = json.load(open(os.path.join(golden_dir, "reference_live.json")))
    return meta, np.load(os.path.join(golden_dir, "reference_live.npz"))


# ---------------------------------------------------------------------------------------------- CTC
def test_ctc_oracle_matches_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "ctc_small.npz"))
    feas = g["feasible"]
    w = feas.astype(np.float64)
    nll, grad = ctc_ref.ctc_loss_and_grad(g["log_probs"], g["targets"], g["input_lengths"], g["target_lengths"], 0, w)
    assert np.isinf(nll[~feas]).all() and np.isinf(g["nll"][~feas]).all()
    np.testing.assert_allclose(nll[feas], g["nll"][feas], rtol=1e-5)
    gm = np.broadcast_to(feas[None, :, None], grad.shape)
    np.testing.assert_allclose(grad[gm], g["grad_feasible"][gm], atol=2e-4)
    assert np.isinf(g["loss_sum"])  # the reference's reduction='sum' is inf when one utterance is infeasible


@pytest.mark.parametrize("T,N,C,S,seed", [(25, 4, 7, 5, 0), (60, 3, 20, 12, 1), (12, 2, 5, 1, 2)])
def test_ctc_oracle_matches_torch_cpu(T, N, C, S, seed):
    g = torch.Generator().manual_seed(seed)
    lp = torch.log_softmax(torch.randn(T, N, C, generator=g) * 3, -1)
    tl = torch.randint(0, S + 1, (N,), generator=g)
    tg = torch.randint(1, C, (N, S), generator=g)
    il = torch.randint(2 * S + 1, T + 1, (N,), generator=g)
    lpr = lp.clone().requires_grad_(True)
    ref = torch.nn.functional.ctc_loss(lpr, tg, il, tl, reduction="none")
    ref.sum().backward()
    nll, grad = ctc_ref.ctc_loss_and_grad(lp.numpy(), tg.numpy(), il.numpy(), tl.numpy())
    np.testing.assert_allclose(nll, ref.detach().numpy(), rtol=2e-5)
    np.testing.assert_allclose(grad, lpr.grad.numpy(), atol=2e-4)  # torch accumulates in fp32, the oracle in fp64


def test_ctc_oracle_empty_target_and_short_input():
    lp = np.log(np.full((3, 1, 4), 0.25, dtype=np.float32))
    nll, _ = ctc_ref.ctc_loss_and_grad(lp, np.zeros((1, 1), dtype=np.int64), [3], [0])
    np.testing.assert_allclose(nll, [-3 * np.log(0.25)], rtol=1e-6)
    nll, _ = ctc_ref.ctc_loss_and_grad(lp, np.array([[1, 1, 2]]), [3], [3])  # needs 4 frames
    assert np.isinf(nll[0])


# ------------------------------------------------------------------------------------------- decoding
def test_collapse_and_edit_distance():
    assert decode_ref.collapse([1, 1, 0, 1, 2, 2, 0, 0, 3]) == [1, 1, 2, 3]
    assert decode_ref.collapse([0, 0, 0]) == []
    assert decode_ref.collapse([5]) == [5]
    assert decode_ref.levenshtein("kitten", "sitting") == 3
    assert decode_ref.levenshtein([], [1, 2]) == 2
    assert decode_ref.wer("a b c", "a c") == 1
    assert decode_ref.cer(" a b", " a c") == 1


def test_greedy_oracle_matches_golden(golden_dir):
    for name in ("rnn_bn", "rnn_nobn", "cnn_rnn"):
        meta = json.load(open(os.path.join(golden_dir, "model_%s.json" % name)))
        g = np.load(os.path.join(golden_dir, "model_%s.npz" % name))
        C = meta["cfg"]["C"]
        int2char = {i: ("blank" if i == 0 else "u%d" % i) for i in range(C)}
        assert decode_ref.greedy_strings(g["out_eval"], g["input_lengths"], int2char) == meta["greedy"]
        idx = g["out_train"].argmax(-1)
        assert (idx == g["argmax"]).all()
        errs, toks = decode_ref.batch_errors(idx.T, g["input_lengths"], g["targets"], g["target_lengths"])
        assert (errs, toks) == (meta_wer(g))


def meta_wer(g):
    return int(g["wer_errs"]), int(g["wer_toks"])


def test_beam_oracle_matches_golden(golden_dir):
    meta = json.load(open(os.path.join(golden_dir, "beam_small.json")))
    arrs = np.load(os.path.join(golden_dir, "beam_small.npz"))
    assert meta["all_blank_error"] == "IndexError"
    for case in meta["cases"]:
        lm = decode_ref.BigramLM(os.path.join(golden_dir, case["arpa"]))
        probs = arrs["%s/probs" % case["tag"]]
        _, strings = decode_ref.beam_search(probs, case["lens"], case["units"], case["beam_width"], lm, case["lm_alpha"])
        assert strings == case["strings"], (case["tag"], case["beam_width"], case["lm_alpha"])


def test_beam_oracle_all_blank_raises_like_reference(golden_dir):
    lm = decode_ref.BigramLM(os.path.join(golden_dir, "lm_c8.arpa"))
    probs = np.tile(np.array([0.97, 0.01, 0.01, 0.01], dtype=np.float32), (1, 6, 1))
    with pytest.raises(IndexError):
        decode_ref.beam_search(probs, [6], ["blank", "UNK", "a", "b"], 3, lm, 0.1)


def test_lm_oracle_backoff(golden_dir):
    lm = decode_ref.BigramLM(os.path.join(golden_dir, "lm_c8.arpa"))
    tab = lm.table(["blank", "UNK", "a", "b", "c", "d", "e", "f"])
    assert np.isnan(tab[0]).all() and np.isnan(tab[:, 0]).all()  # 'blank' is not an LM unit -> KeyError in the reference
    assert tab[2, 3] == lm.bigram("a", "b")
    assert tab[8, 2] == lm.bigram("", "a") and tab[2, 8] == lm.bigram("a", "")
    key = "a b"
    if key not in lm.bi:
        assert lm.bigram("a", "b") == lm.uni["a"][1] + lm.uni["b"][0]


def test_decode_oracle_matches_reference_live(golden_dir, reference_live):
    """Bigram table, beam / greedy strings and wer / cer of the oracle equal what the reference's LanguageModel, BeamDecoder,
    GreedyDecoder and Decoder returned on the same log-probs."""
    meta, arrs = reference_live
    rec = meta["decode"]
    units = rec["units"]
    int2char = dict(enumerate(units))
    lm = decode_ref.BigramLM(os.path.join(golden_dir, rec["arpa"]))
    words = rec["words"]
    for i, w1 in enumerate(words):
        for j, w2 in enumerate(words):
            assert lm.bigram(w1, w2) == rec["bigram"][i][j]
    assert len(rec["cases"]) == 6
    for case in rec["cases"]:
        lp = torch.from_numpy(arrs["decode/lp%d" % case["seed"]])
        lens = case["lens"]
        assert len(case["beams"]) == 2
        for beam in case["beams"]:
            probs = torch.exp(lp.transpose(0, 1)).numpy()
            _, got = decode_ref.beam_search(probs, lens, units, beam["beam_width"], lm, beam["lm_alpha"])
            assert got == beam["strings"]
        assert decode_ref.greedy_strings(lp.numpy(), lens, int2char) == case["greedy"]
    a, b, want = rec["cer"]
    assert decode_ref.cer(a, b) == want
    a, b, want = rec["wer"]
    assert decode_ref.wer(a, b) == want


# ---------------------------------------------------------------------------------------------- model
def _build_oracle(cfg):
    from oracle.make_golden import model_args
    args = model_args(cfg)
    return model_ref.RefAcousticModel(cfg["F"], cfg["H"], cfg["L"], cfg["C"], batch_norm=cfg["bn"],
                                      cnn_layers=args["cnn_param"]["layer"] if cfg["cnn"] else None, cnn_batch_norm=cfg["bn"])


@pytest.mark.parametrize("name", ["rnn_bn", "rnn_nobn", "cnn_rnn", "cnn_pool"])
def test_model_oracle_matches_golden(golden_dir, name):
    meta = json.load(open(os.path.join(golden_dir, "model_%s.json" % name)))
    g = np.load(os.path.join(golden_dir, "model_%s.npz" % name))
    cfg = meta["cfg"]
    torch.manual_seed(cfg["seed"])
    m = _build_oracle(cfg)  # same creation order as the reference -> same initial weights under the seed
    for k, v in m.state_dict().items():
        assert abs(float(v.double().abs().sum()) - meta["checksum"][k]) <= 1e-9 * max(1.0, meta["checksum"][k]), k
    x = torch.from_numpy(g["x"])
    m.train()
    out = m(x)
    np.testing.assert_allclose(out.detach().numpy(), g["out_train"], atol=1e-6)
    loss = nn.CTCLoss(reduction="sum")(out, torch.from_numpy(g["targets"]), torch.from_numpy(g["input_lengths"]),
                                       torch.from_numpy(g["target_lengths"])) / cfg["N"]
    assert abs(float(loss.detach()) - float(g["loss"])) < 1e-5 * abs(float(g["loss"]))
    loss.backward()
    for k, p in m.named_parameters():
        step = meta["grad_step"][k]
        vals = p.grad.reshape(-1)[::step][:256].numpy()
        np.testing.assert_allclose(vals, g["gradvals/" + k], atol=1e-5 * max(1.0, meta["grad_norm"][k]))
    m.eval()
    with torch.no_grad():
        np.testing.assert_allclose(m(x).numpy(), g["out_eval"], atol=1e-6)


def test_model_oracle_matches_reference_live(reference_live):
    """The oracle, with the reference's weights (re-created from the seed, verified by checksum), gives the reference
    CTC_Model's outputs in train mode and then in eval mode."""
    from oracle.make_golden import MODEL_CASES
    meta, arrs = reference_live
    assert sorted(meta["model"]["checksum"]) == sorted(MODEL_CASES)
    for name, cfg in MODEL_CASES.items():
        torch.manual_seed(cfg["seed"])
        om = _build_oracle(cfg)
        want_sum = meta["model"]["checksum"][name]
        assert list(om.state_dict()) == list(want_sum)
        for k, v in om.state_dict().items():
            assert abs(float(v.double().abs().sum()) - want_sum[k]) <= 1e-9 * max(1.0, want_sum[k]), (name, k)
        x, *_ = model_ref.synthetic_batch(cfg["T"], cfg["N"], cfg["F"], cfg["C"], cfg["S"], cfg["seed"])
        assert np.array_equal(x.numpy(), arrs["model/%s/x" % name])
        for mode in ("train", "eval"):
            getattr(om, mode)()
            a, b = torch.from_numpy(arrs["model/%s/%s" % (name, mode)]), om(x)
            # same library kernels, different reduction order inside BatchNorm -> float32 round-off only
            assert torch.allclose(a, b, atol=2e-6, rtol=0), (name, mode, (a - b).abs().max())


# ------------------------------------------------------------------- packed / variable-length semantics (N1)
def _packed_golden(golden_dir):
    from oracle import packed_ref
    meta = json.load(open(os.path.join(golden_dir, "packed_rnn.json")))
    g = np.load(os.path.join(golden_dir, "packed_rnn.npz"))
    cfg = meta["cfg"]
    torch.manual_seed(cfg["seed"])
    m = packed_ref.RefPackedModel(cfg["F"], cfg["H"], cfg["L"], True, cfg["C"])
    for k, v in m.state_dict().items():   # same construction order as the reference => same weights from the seed
        if k in meta["checksum"]:
            assert abs(float(v.double().abs().sum()) - meta["checksum"][k]) <= 1e-6 * max(1.0, meta["checksum"][k]), k
    return packed_ref, meta, g, m


def test_packed_oracle_matches_golden(golden_dir):
    """The mask formulation of oracle/packed_ref.py reproduces what the unmodified 863 CTC_RNN computed on a
    pack_padded_sequence batch (tests/golden/packed_rnn.*): activations, warp-ctc style loss, gradients, eval log-probs."""
    packed_ref, meta, g, m = _packed_golden(golden_dir)
    x, lens = torch.from_numpy(g["x"]), g["lengths"].tolist()
    m.train()
    act = m(x, lens)
    np.testing.assert_allclose(act.detach().numpy(), g["act_train"], atol=5e-6)
    # padded frames are exactly zero after pad_packed_sequence
    for n, l in enumerate(lens):
        assert np.all(g["act_train"][l:, n] == 0.0) and torch.all(act[l:, n] == 0.0)
    loss = packed_ref.warp_ctc_loss(act, torch.from_numpy(g["targets"]), lens, g["target_sizes"].tolist())
    assert abs(float(loss) - float(g["loss"])) < 1e-5 * abs(float(g["loss"]))
    loss.backward()
    for k, p in m.named_parameters():
        step = meta["grad_step"][k]
        vals = p.grad.reshape(-1)[::step][:256].numpy()
        np.testing.assert_allclose(vals, g["gradvals/" + k], atol=2e-5 * max(1.0, meta["grad_norm"][k]))
        assert abs(float(p.grad.norm()) - meta["grad_norm"][k]) < 1e-4 * max(1.0, meta["grad_norm"][k])
    for k, v in m.named_buffers():
        if "running" in k:
            np.testing.assert_allclose(v.numpy(), g["buffer/" + k], atol=1e-6)
    m.eval()
    with torch.no_grad():
        np.testing.assert_allclose(m(x, lens).numpy(), g["logp_eval"], atol=5e-6)


def test_packed_oracle_matches_reference_live(reference_live):
    """The packed oracle, with the unmodified 863 CTC_RNN's weights (re-created from the seed, verified by checksum), gives its
    activations, loss and gradients (a fixed sample of 1024 entries per parameter, plus every gradient's norm)."""
    from oracle import packed_ref
    from oracle.make_golden_live import PACKED_CASES, grad_sample_index
    meta, arrs = reference_live
    cases = meta["packed"]["cases"]
    assert [(c["T"], c["N"], c["H"], c["L"], c["bn"]) for c in cases] == [tuple(c) for c in PACKED_CASES]
    for case in cases:
        seed, T, N, H, L, bn = case["seed"], case["T"], case["N"], case["H"], case["L"], case["bn"]
        torch.manual_seed(100 + seed)
        mine = packed_ref.RefPackedModel(40, H, L, bn, 9)
        assert list(mine.state_dict()) == list(case["checksum"])
        for k, v in mine.state_dict().items():
            assert abs(float(v.double().abs().sum()) - case["checksum"][k]) <= 1e-9 * max(1.0, case["checksum"][k]), k
        x, lens, tg, tsz = packed_ref.synthetic_packed_batch(T, N, 40, 9, 3, seed)
        mine.train()
        a = torch.from_numpy(arrs["packed/%d/act" % seed])
        b = mine(x, lens)
        assert (a - b).abs().max().item() < 5e-6
        la = case["loss"]
        lb = packed_ref.warp_ctc_loss(b, tg, lens, tsz); lb.backward()
        assert abs(la - lb.item()) < 1e-5 * abs(la)
        for k, p in mine.named_parameters():
            want, g = case["grads"][k], p.grad.reshape(-1)
            tol = 2e-5 * max(1.0, want["maxabs"])
            got = g[torch.from_numpy(grad_sample_index(g.numel(), k))]
            assert (got - torch.from_numpy(arrs["packed/%d/grad/%s" % (seed, k)])).abs().max().item() < tol, k
            assert abs(g.abs().max().item() - want["maxabs"]) < tol, k
            assert abs(g.norm().item() - want["norm"]) < 1e-4 * max(1.0, want["norm"]), k


# ------------------------------------------------------------------- host batch assembly (N2)
def _batch_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "batch_small.npz"))
    n = int(g["n"])
    feats = [g["feat/%d" % i] for i in range(n)]
    labs = [g["label/%d" % i] for i in range(n)]
    return g, feats, labs


def test_batch_oracle_matches_golden(golden_dir):
    from oracle import batch_ref
    g, feats, labs = _batch_golden(golden_dir)
    for ci, (left, right, skip, down) in enumerate(g["cases"].tolist()):
        x, isz, tg, tsz = batch_ref.batch(feats, labs, left, right, skip, down)
        assert np.array_equal(x, g["case%d/x" % ci]) and np.array_equal(isz, g["case%d/input_sizes" % ci])
        assert np.array_equal(tg, g["case%d/targets" % ci]) and np.array_equal(tsz, g["case%d/target_sizes" % ci])


def test_batch_oracle_matches_reference_live(reference_live):
    """Splicing and frame skipping of the oracle equal the reference's utils/tools.py make_context + skip_feat."""
    from oracle import batch_ref
    meta, arrs = reference_live
    assert meta["batch"]["cases"] == [[0, 0, 1], [4, 0, 1], [0, 3, 2], [2, 2, 5], [7, 7, 3]]
    rng = np.random.RandomState(3)
    for ci, (left, right, skip) in enumerate(meta["batch"]["cases"]):
        f = rng.randn(rng.randint(1, 30), 5).astype(np.float32)
        assert np.array_equal(f, arrs["batch/%d/feat" % ci])
        a = arrs["batch/%d/out" % ci]
        b = batch_ref.skipped(batch_ref.spliced(f, left, right), skip)
        assert a.shape == b.shape and np.array_equal(a, b)


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_alignment_design_reproduces_packed_semantics(seed):
    """DESIGN.md §9 (N1): full-length scans over a left-aligned (forward) and a right-aligned (reverse) batch, with arbitrary
    finite garbage in the padding rows, give exactly the packed bidirectional LSTM — outputs and every gradient."""
    from oracle import packed_ref
    torch.manual_seed(seed)
    T, N, I, H = 17, 4, 6, 5
    lengths = [17, 12, 12, 3]
    rnn = nn.LSTM(I, H, bidirectional=True, bias=False).double()
    x = torch.randn(T, N, I, dtype=torch.float64)
    for n, L in enumerate(lengths):
        x[L:, n] = 0.0
    x.requires_grad_(True)
    # reference formulation: each utterance alone through torch's LSTM on its valid slice
    want = torch.zeros(T, N, 2 * H, dtype=torch.float64)
    for n, L in enumerate(lengths):
        y, _ = rnn(x[:L, n:n + 1])
        want[:L, n] = y[:, 0]
    w = torch.randn(T, N, 2 * H, dtype=torch.float64)
    gw = torch.autograd.grad((want * w).sum(), [x] + list(rnn.parameters()))
    got = packed_ref.aligned_bilstm(rnn, x, lengths, garbage=3.0 * torch.randn(T, N, I, dtype=torch.float64))
    gg = torch.autograd.grad((got * w).sum(), [x] + list(rnn.parameters()))
    assert (got - want).abs().max().item() < 1e-12
    for a, b in zip(gg, gw):
        assert (a - b).abs().max().item() < 1e-11
    # and the padding rows of the input receive no gradient at all
    for n, L in enumerate(lengths):
        assert gg[0][L:, n].abs().max().item() == 0.0 if L < T else True


def test_alignment_design_full_model_matches_packed_oracle(golden_dir):
    """The whole planned N1 composition (column-sum BatchNorm with the valid-frame count, aligned recurrent scans with garbage
    in the padding, output layer on all rows with re-zeroed padding) equals the packed oracle — and therefore the unmodified 863
    model, to which that oracle is pinned — in activations, loss, gradients, running statistics and eval log-probs."""
    import copy
    packed_ref, meta, g, m = _packed_golden(golden_dir)
    m = m.double()
    m2 = copy.deepcopy(m)
    x, lens = torch.from_numpy(g["x"]).double(), g["lengths"].tolist()
    tg, tsz = torch.from_numpy(g["targets"]), g["target_sizes"].tolist()
    m.train(); m2.train()
    a = m(x, lens)
    b = packed_ref.aligned_model_forward(m2, x, lens, garbage_scale=2.0)
    assert (a - b).abs().max().item() < 1e-10
    la = packed_ref.warp_ctc_loss(a, tg, lens, tsz); la.backward()
    lb = packed_ref.warp_ctc_loss(b, tg, lens, tsz); lb.backward()
    assert abs(la.item() - lb.item()) < 1e-10 * abs(la.item())
    for (k, p), (_, q) in zip(m.named_parameters(), m2.named_parameters()):
        assert (p.grad - q.grad).abs().max().item() < 1e-9 * max(1.0, p.grad.abs().max().item()), k
    for (k, u), (_, v) in zip(m.named_buffers(), m2.named_buffers()):
        assert torch.allclose(u.double(), v.double(), atol=1e-12), k
    m.eval(); m2.eval()
    with torch.no_grad():
        assert (m(x, lens) - packed_ref.aligned_model_forward(m2, x, lens)).abs().max().item() < 1e-10
