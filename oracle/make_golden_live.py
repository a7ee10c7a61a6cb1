"""ORACLE — test infrastructure only. Records what the UNMODIFIED reference returns on the inputs of the CPU tests that pin the
oracle and the host-side mirrors to it (tests/test_oracle.py, tests/test_abi_host.py, tests/test_train_host.py), so that those
comparisons run wherever the repository is checked out:

    python -m oracle.make_golden_live          # needs the reference tree (oracle/ref_shim.py, my_863_corpus for the packed case)

Writes tests/golden/reference_live.json (strings, scalars, LM tables, schedule traces, checkpoint layout) and
tests/golden/reference_live.npz (inputs and outputs). Large gradients are stored as a seeded sample of 1024 entries plus their
norm and largest magnitude; weights are not stored but re-created from the seed and verified by checksum.
"""
import json
import os
import sys
import types

import numpy as np
import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_shim  # noqa: E402
from oracle.make_golden import MODEL_CASES, model_args  # noqa: E402
from oracle.model_ref import synthetic_batch  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
REF_TREE = os.path.dirname(ref_shim.REF_ROOT)   # the reference repository (timit/ and my_863_corpus/)

UNITS8 = ["blank", "UNK", "a", "b", "c", "d", "e", "f"]
DECODE_SEEDS = range(6)
DECODE_BEAMS = ((2, 0.05), (8, 0.2))
PACKED_CASES = [(18, 3, 128, 2, True), (25, 4, 128, 3, True), (12, 2, 128, 2, False)]
BATCH_SPLICE = [(0, 0, 1), (4, 0, 1), (0, 3, 2), (2, 2, 5), (7, 7, 3)]
SCHEDULE_SEEDS = range(12)
CHECKPOINT_RNN_PARAM = {"rnn_input_size": 40, "rnn_hidden_size": 128, "rnn_layers": 2, "rnn_type": nn.LSTM,
                        "bidirectional": True, "batch_norm": True}
CKPT_SEED = 7
GRAD_SAMPLE = 1024


def checksum(sd):
    return {k: float(v.double().abs().sum()) for k, v in sd.items()}


def grad_sample_index(numel, key):
    """Fixed, seeded positions of the stored gradient entries of one parameter (all of them when it has few)."""
    if numel <= GRAD_SAMPLE:
        return np.arange(numel)
    rng = np.random.RandomState(sum(key.encode()) + numel)
    return np.sort(rng.choice(numel, GRAD_SAMPLE, replace=False))


def gen_decode(ref, meta, arrays):
    """Bigram table, beam and greedy strings, wer / cer of the reference's LanguageModel / BeamDecoder / GreedyDecoder / Decoder."""
    int2char = dict(enumerate(UNITS8))
    arpa = os.path.join(OUT, "lm_c8.arpa")
    rlm = ref.LanguageModel(arpa_file=arpa)
    words = UNITS8[1:] + [""]
    cases = []
    for seed in DECODE_SEEDS:
        g = torch.Generator().manual_seed(100 + seed)
        T, N, C = 24, 3, 8
        logits = 2.5 * torch.randn(T, N, C, generator=g)
        logits[:, :, 0] += 1.5
        lp = torch.log_softmax(logits, -1)
        lens = [T, T - 5, T // 2]
        arrays["decode/lp%d" % seed] = lp.numpy()
        beams = []
        for width, alpha in DECODE_BEAMS:
            dec = ref.BeamDecoder(int2char, beam_width=width, blank_index=0, space_idx=-1, lm_path=arpa, lm_alpha=alpha)
            beams.append(dict(beam_width=width, lm_alpha=alpha, strings=dec.decode(lp, lens)))
        greedy = ref.GreedyDecoder(int2char, space_idx=-1, blank_index=0).decode(lp, lens)
        cases.append(dict(seed=seed, lens=lens, beams=beams, greedy=greedy))
    d = ref.Decoder(int2char, space_idx=-1, blank_index=0)
    meta["decode"] = dict(units=UNITS8, arpa="lm_c8.arpa", words=words,
                          bigram=[[rlm.get_bi_prob(w1, w2) for w2 in words] for w1 in words], cases=cases,
                          cer=[" a b c", " a c", d.cer(" a b c", " a c")], wer=["a b c d", "a c d e", d.wer("a b c d", "a c d e")])


def gen_model(ref, meta, arrays):
    """Outputs of the reference CTC_Model in train and then eval mode for every MODEL_CASES entry."""
    out = {}
    for name, cfg in MODEL_CASES.items():
        torch.manual_seed(cfg["seed"])
        rm = ref.CTC_Model(**model_args(cfg))
        out[name] = checksum(rm.state_dict())   # taken before any forward pass
        x, *_ = synthetic_batch(cfg["T"], cfg["N"], cfg["F"], cfg["C"], cfg["S"], cfg["seed"])
        arrays["model/%s/x" % name] = x.numpy()
        for mode in ("train", "eval"):
            getattr(rm, mode)()
            with torch.no_grad():
                arrays["model/%s/%s" % (name, mode)] = rm(x).numpy()
    meta["model"] = dict(checksum=out)


def gen_packed(meta, arrays):
    """The unmodified 863 CTC_RNN on pack_padded_sequence batches: activations, warp-ctc style loss, gradient samples."""
    sys.path.insert(0, os.path.join(REF_TREE, "my_863_corpus", "steps"))
    import model as m863  # noqa: E402  (the reference's module, imported in place)
    from oracle import packed_ref
    cases = []
    for seed, (T, N, H, L, bn) in enumerate(PACKED_CASES):
        torch.manual_seed(100 + seed)
        net = m863.CTC_RNN(rnn_input_size=40, rnn_hidden_size=H, rnn_layers=L, rnn_type=nn.LSTM, bidirectional=True,
                           batch_norm=bn, num_class=9, drop_out=0.0)
        torch.manual_seed(100 + seed)
        mine = packed_ref.RefPackedModel(40, H, L, bn, 9)
        sd = {k: v.clone() for k, v in net.state_dict().items()}   # before the forward pass updates the running statistics
        for k, v in mine.state_dict().items():   # the oracle re-creates exactly these weights from the seed
            assert torch.equal(v, sd[k]), k
        x, lens, tg, tsz = packed_ref.synthetic_packed_batch(T, N, 40, 9, 3, seed)
        net.train()
        a = net(nn.utils.rnn.pack_padded_sequence(x, lens))
        loss = packed_ref.warp_ctc_loss(a, tg, lens, tsz)
        loss.backward()
        arrays["packed/%d/act" % seed] = a.detach().numpy()
        grads = {}
        for k, p in net.named_parameters():
            g = p.grad.detach().reshape(-1)
            arrays["packed/%d/grad/%s" % (seed, k)] = g[torch.from_numpy(grad_sample_index(g.numel(), k))].numpy()
            grads[k] = dict(norm=float(g.norm()), maxabs=float(g.abs().max()))
        cases.append(dict(seed=seed, T=T, N=N, H=H, L=L, bn=bn, loss=float(loss), checksum=checksum(sd), grads=grads))
    meta["packed"] = dict(cases=cases, grad_sample=GRAD_SAMPLE)


def gen_batch(meta, arrays):
    """utils/tools.py make_context + skip_feat of the reference on seeded feature matrices."""
    sys.path.insert(0, os.path.join(REF_TREE, "timit"))
    sys.path.insert(0, os.path.join(REF_TREE, "timit", "utils"))
    sys.modules.setdefault("kaldiio", types.ModuleType("kaldiio"))
    import tools  # noqa: E402
    rng = np.random.RandomState(3)
    for ci, (left, right, skip) in enumerate(BATCH_SPLICE):
        f = rng.randn(rng.randint(1, 30), 5).astype(np.float32)
        arrays["batch/%d/feat" % ci] = f
        arrays["batch/%d/out" % ci] = tools.skip_feat(tools.make_context(f, left, right), skip)
    meta["batch"] = dict(cases=[list(c) for c in BATCH_SPLICE])


def gen_schedule(meta):
    """The reference's own `while not stop_train:` loop (oracle/train_live.py) on the scripted dev-loss sequences."""
    from oracle import train_live, train_ref
    traces = []
    for seed in SCHEDULE_SEEDS:
        losses, accs = train_ref.scripted_sequence(seed, 120)
        losses[0] = 30.0
        live, final = train_live.reference_schedule_trace(losses, accs, 1e-3, 0.5, 0.05, 100)
        traces.append(dict(seed=seed, lr=[r["lr"] for r in live], rollback=[r["rollback"] for r in live],
                           final={k: final[k] for k in ("loss_best", "acc_best", "epochs")}))
    meta["schedule"] = dict(init_lr=1e-3, decay=0.5, end_adjust_acc=0.05, num_epoches=100, first_loss=30.0, traces=traces)


def gen_checkpoint(ref, meta):
    """Layout of the reference's save_package: keys, constructor fields, state_dict names / shapes, weights by checksum."""
    torch.manual_seed(CKPT_SEED)
    theirs = ref.CTC_Model(rnn_param=CHECKPOINT_RNN_PARAM, num_class=11, drop_out=0.1)
    pkg = ref.CTC_Model.save_package(theirs, epoch={"epoch": 1})
    fields = {k: v for k, v in pkg.items() if k != "state_dict"}
    fields["rnn_param"] = dict(fields["rnn_param"], rnn_type=fields["rnn_param"]["rnn_type"].__name__)
    sd = pkg["state_dict"]
    meta["checkpoint"] = dict(seed=CKPT_SEED, fields=fields, keys=sorted(pkg.keys()), state_dict=[[k, list(v.shape)] for k, v in sd.items()],
                              checksum=checksum(sd))


def gen_host(ref, meta):
    """Decoder string helpers and the LanguageModel tables of both committed ARPA files."""
    int2char = {0: "_", 1: "a", 2: "b", 3: "c"}
    d = ref.Decoder(int2char, space_idx=-1, blank_index=0)
    strings = []
    for seq in (["a", "a", "_", "b", "b", "c"], ["_", "_"], ["c"]):
        for rr in (True, False):
            strings.append([seq, rr, d._process_string(seq, rr)])
    lms = {}
    for name in ("lm_c8.arpa", "lm_c62.arpa"):
        lm = ref.LanguageModel(arpa_file=os.path.join(OUT, name))
        lms[name] = dict(unigram=lm.unigram, bigram=lm.bigram)
    meta["host"] = dict(int2char=int2char, process_string=strings, wer=["a b c d", "b c e", d.wer("a b c d", "b c e")],
                        cer=[" a b", " b", d.cer(" a b", " b")], lm=lms)


def main():
    torch.set_num_threads(4)
    ref = ref_shim.load()
    meta, arrays = {}, {}
    gen_decode(ref, meta, arrays)
    gen_model(ref, meta, arrays)
    gen_packed(meta, arrays)
    gen_batch(meta, arrays)
    gen_schedule(meta)
    gen_checkpoint(ref, meta)
    gen_host(ref, meta)
    meta = json.loads(json.dumps(meta))   # plain JSON types only (tuples -> lists), as the tests read it back
    np.savez_compressed(os.path.join(OUT, "reference_live.npz"), **arrays)
    with open(os.path.join(OUT, "reference_live.json"), "w") as fh:
        json.dump(meta, fh, indent=1)
    print("reference_live: %d arrays, sections %s" % (len(arrays), sorted(meta)))


if __name__ == "__main__":
    main()
