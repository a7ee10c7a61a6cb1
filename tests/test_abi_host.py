"""CPU suite: the C-ABI library loads and exports exactly what include/ctcb200.h declares, the host-side mirrors of
the reference's classes behave like the reference, and the product path refuses to run without CUDA."""
import ctypes
import json
import os

import numpy as np
import pytest
import torch
import torch.nn as nn

from ctc_pytorch_b200 import _build, _lib
from ctc_pytorch_b200.decoder import Decoder, collapse_frames, edit_distance
from ctc_pytorch_b200.lm import LanguageModel
from ctc_pytorch_b200.model import CTC_Model
from oracle import decode_ref


@pytest.fixture(scope="module")
def built_lib():
    path = _build.build()
    assert os.path.exists(path)
    return path


def test_library_exports_every_declared_symbol(built_lib):
    protos = _lib.parse_header()
    assert len(protos) >= 20
    dll = ctypes.CDLL(built_lib)  # must load without a GPU driver (no libcuda link dependency)
    for name in protos:
        assert hasattr(dll, name), "include/ctcb200.h declares %s but libctcb200.so does not export it" % name
    dll.ctcb200_version.restype = ctypes.c_int
    assert dll.ctcb200_version() >= 100
    dll.ctcb200_last_error.restype = ctypes.c_char_p
    assert isinstance(dll.ctcb200_last_error(), bytes)


def test_no_undeclared_exports(built_lib):
    import subprocess
    out = subprocess.run(["nm", "-D", "--defined-only", built_lib], capture_output=True, text=True).stdout
    exported = {l.split()[-1] for l in out.splitlines() if " T " in l}
    declared = set(_lib.parse_header())
    assert {e for e in exported if e.startswith("ctcb200_")} == declared


def test_workspace_size_queries_need_no_gpu(built_lib):
    L = _lib.lib()
    assert L.dll.ctcb200_ctc_workspace_floats(800, 32, 60) >= 32 * 800 * 4 * 32  # alpha history + log-scale offsets
    assert L.dll.ctcb200_lstm_scratch_bytes(32, 512) > 0
    assert L.dll.ctcb200_beam_workspace_bytes(800, 32, 62, 100) > 0


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_product_path_fails_loudly_without_cuda():
    from ctc_pytorch_b200.loss import CTCLoss
    from ctc_pytorch_b200.decoder import GreedyDecoder
    lp = torch.log_softmax(torch.randn(5, 2, 4), -1)
    with pytest.raises(RuntimeError, match="CUDA"):
        CTCLoss(reduction="sum")(lp, torch.ones(2, 2, dtype=torch.long), [5, 5], [2, 2])
    with pytest.raises(RuntimeError, match="CUDA"):
        GreedyDecoder({0: "_", 1: "a", 2: "b", 3: "c"}, space_idx=-1).decode(lp, [5, 5])
    m = CTC_Model(rnn_param={"rnn_input_size": 8, "rnn_hidden_size": 128, "rnn_layers": 1, "rnn_type": nn.LSTM,
                             "bidirectional": True, "batch_norm": False}, num_class=4, drop_out=0.0)
    with pytest.raises(RuntimeError, match="CUDA"):
        m(torch.randn(2, 5, 8))


def test_model_surface_and_state_dict_keys(golden_dir):
    with pytest.raises(ValueError):
        CTC_Model(rnn_param=None)
    for name in ("rnn_bn", "rnn_nobn", "cnn_rnn"):
        meta = json.load(open(os.path.join(golden_dir, "model_%s.json" % name)))
        from oracle.make_golden import model_args
        cfg = meta["cfg"]
        torch.manual_seed(cfg["seed"])
        m = CTC_Model(**model_args(cfg))
        sd = m.state_dict()
        assert list(sd.keys()) == list(meta["checksum"].keys())
        for k, v in sd.items():  # same creation order as the reference => identical initial weights under the seed
            assert abs(float(v.double().abs().sum()) - meta["checksum"][k]) <= 1e-9 * max(1.0, meta["checksum"][k]), k
        pkg = CTC_Model.save_package(m, epoch={"n_feats": 40})
        assert set(pkg) == {"rnn_param", "add_cnn", "cnn_param", "num_class", "_drop_out", "state_dict", "epoch"}


def test_compute_wer_matches_golden(golden_dir):
    m = CTC_Model(rnn_param={"rnn_input_size": 8, "rnn_hidden_size": 128, "rnn_layers": 1, "rnn_type": nn.LSTM,
                             "bidirectional": True, "batch_norm": False}, num_class=4, drop_out=0.0)
    for name in ("rnn_bn", "rnn_nobn", "cnn_rnn"):
        g = np.load(os.path.join(golden_dir, "model_%s.npz" % name))
        errs, toks = m.compute_wer(g["argmax"].T, g["input_lengths"], g["targets"], g["target_lengths"])
        assert (errs, toks) == (int(g["wer_errs"]), int(g["wer_toks"]))


def test_decoder_host_helpers():
    assert collapse_frames([3, 3, 0, 3, 1, 1, 0]) == [3, 3, 1]
    assert edit_distance("abc", "") == 3 and edit_distance([1, 2, 3], [1, 3]) == 1
    for a, b in (("kitten", "sitting"), ("", "x"), ("abcd", "abcd"), ([1, 2, 3, 4], [4, 3, 2, 1])):
        assert edit_distance(a, b) == decode_ref.levenshtein(a, b)
    d = Decoder({0: "_", 1: "a", 2: "b", 3: " "}, space_idx=-1, blank_index=0)
    assert d._process_string(["a", "a", "_", "b"], remove_rep=True) == " a b"
    assert d._process_string(["a", "a", "_", "b"], remove_rep=False) == " a a b"
    assert d._convert_to_strings([[1, 2, 1, 0, 3]]) == [["a", "b", "a", "_", " "]]
    d2 = Decoder({0: "_", 1: "a", 2: "b", 3: " "}, space_idx=3, blank_index=0)
    assert d2._process_string(list("ab a"), remove_rep=False) == "ab a"
    assert d.wer("a b c", "a c") == 1 and d.cer("abc", "abd") == 1
    assert d._unflatten_targets([1, 2, 3, 4, 5], [2, 3]) == [[1, 2], [3, 4, 5]]


def test_language_model_matches_oracle(golden_dir):
    arpa = os.path.join(golden_dir, "lm_c8.arpa")
    lm, olm = LanguageModel(arpa_file=arpa), decode_ref.BigramLM(arpa)
    units = ["UNK", "a", "b", "c", "d", "e", "f"]
    for w1 in units + [""]:
        for w2 in units + [""]:
            assert lm.get_bi_prob(w1, w2) == olm.bigram(w1, w2)
    with pytest.raises(KeyError):
        lm.get_bi_prob("nosuchunit", "a")
    classes = ["blank"] + units
    tab = lm.dense_table(classes)
    np.testing.assert_array_equal(tab, olm.table(classes))
    assert lm.score_bg("a b") == lm.get_bi_prob("<s>", "a") + lm.get_bi_prob("a", "b") + lm.get_bi_prob("b", "</s>")


def _reference_host(golden_dir):
    """What the reference's Decoder / LanguageModel returned (tests/golden/reference_live.json, oracle/make_golden_live.py)."""
    return json.load(open(os.path.join(golden_dir, "reference_live.json")))["host"]


def test_host_mirrors_match_reference_live(golden_dir):
    rec = _reference_host(golden_dir)
    int2char = {int(k): v for k, v in rec["int2char"].items()}
    assert int2char == {0: "_", 1: "a", 2: "b", 3: "c"}
    mine = Decoder(int2char, space_idx=-1, blank_index=0)
    assert len(rec["process_string"]) == 6
    for seq, rr, want in rec["process_string"]:
        assert mine._process_string(seq, rr) == want
    a, b, want = rec["wer"]
    assert mine.wer(a, b) == want
    a, b, want = rec["cer"]
    assert mine.cer(a, b) == want
    lm = LanguageModel(arpa_file=os.path.join(golden_dir, "lm_c62.arpa"))
    assert lm.unigram == rec["lm"]["lm_c62.arpa"]["unigram"] and lm.bigram == rec["lm"]["lm_c62.arpa"]["bigram"]


def test_product_path_never_imports_the_oracle():
    """oracle/ is test infrastructure: nothing under ctc_pytorch_b200/ may import it (DESIGN.md §1)."""
    import re
    pkg = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "ctc_pytorch_b200")
    for fn in sorted(os.listdir(pkg)):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), fn
            assert "/root/reference" not in src, fn


def test_integration_doc_names_every_entry_point():
    """INTEGRATION.md is the maintainer-facing map of the C ABI: every declared entry point appears in it."""
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    hdr = open(os.path.join(root, "include", "ctcb200.h")).read()
    doc = open(os.path.join(root, "INTEGRATION.md")).read()
    names = set(re.findall(r"\b(ctcb200_\w+)\s*\(", hdr)) - {"ctcb200_version"}
    assert names and not [n for n in sorted(names) if n not in doc]


def test_arpa_loader_tolerates_spaces_and_higher_orders(golden_dir, tmp_path):
    """N4: same tables as the reference's loader on its own tab-separated format, and the same tables again from a
    space-separated, CRLF-terminated copy with a trigram section (which the reference's loader cannot read)."""
    tab = os.path.join(golden_dir, "lm_c8.arpa")
    lm = LanguageModel(arpa_file=tab)
    rlm = _reference_host(golden_dir)["lm"]["lm_c8.arpa"]
    assert lm.unigram == rlm["unigram"] and lm.bigram == rlm["bigram"]
    text = open(tab).read().replace("\t", " ").replace("\\end\\", "\\3-grams:\n-0.5 a b c\n\n\\end\\")
    path = str(tmp_path / "spaces.arpa")
    with open(path, "w", newline="") as fh:
        fh.write(text.replace("\n", "\r\n"))
    lm2 = LanguageModel(arpa_file=path)
    assert lm2.unigram == lm.unigram and lm2.bigram == lm.bigram
    assert lm2.higher[3] == {"a b c": (-0.5, 0.0)}
    assert lm2.get_bi_prob("", "a") == lm.get_bi_prob("", "a") and lm2.get_bi_prob("f", "") == lm.get_bi_prob("f", "")


def test_readme_switches_exist_in_the_source():
    """Every CTCB200_* environment switch the README documents is read somewhere in the product or bench source, and the job
    script the README points at parses."""
    import re
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    readme = open(os.path.join(root, "README.md")).read()
    names = set(re.findall(r"`(CTCB200_[A-Z0-9_]+)", readme))
    assert len(names) >= 10
    src = ""
    for d, _, files in os.walk(os.path.join(root, "ctc_pytorch_b200")):
        if os.path.basename(d) == "build":
            continue
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                src += open(os.path.join(d, f), errors="ignore").read()
    src += open(os.path.join(root, "bench.py")).read()
    missing = sorted(n for n in names if n not in src)
    assert not missing, "documented but never read: %s" % missing
    assert subprocess.run(["bash", "-n", os.path.join(root, "tools", "gpu_job.sh")]).returncode == 0
