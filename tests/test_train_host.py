"""CPU tests of the training-loop services (ctc_pytorch_b200/train.py): the lr / rollback schedule against the oracle's
restatement of train_ctc.py:162-231 AND against what the reference's own loop source, exec'ed with stubs (oracle/train_live.py),
produced, and checkpoint interchange with the unmodified reference's package layout (both recorded in
tests/golden/reference_live.json by oracle/make_golden_live.py)."""
import json
import os

import pytest
import torch
import torch.nn as nn

from ctc_pytorch_b200.model import CTC_Model
from ctc_pytorch_b200.train import DevLossSchedule, load_package
from oracle import train_ref
from oracle.make_golden_live import CHECKPOINT_RNN_PARAM as RNN_PARAM


@pytest.fixture(scope="module")
def reference_live(golden_dir):
    return json.load(open(os.path.join(golden_dir, "reference_live.json")))


@pytest.mark.parametrize("seed", range(12))
def test_schedule_matches_reference_policy(seed):
    losses, accs = train_ref.scripted_sequence(seed, 120)
    init_lr, decay, eps, epochs = 1e-3, 0.5, 0.05, 100
    want, final = train_ref.schedule_trace(losses, accs, init_lr, decay, eps, epochs)
    sched = DevLossSchedule(init_lr, decay, eps)
    got, count = [], 0
    while not sched.stop and count < epochs and count < len(losses):
        count += 1
        sched.begin_epoch()
        act = sched.update(losses[count - 1], accs[count - 1])
        got.append(dict(act, lr=sched.learning_rate))
    assert len(got) == len(want) == final["epochs"]
    for g, w in zip(got, want):
        assert g == w
    assert sched.loss_best == final["loss_best"] and sched.acc_best == final["acc_best"]
    assert any(w["rollback"] for w in want)   # the sequences do exercise the halving path


@pytest.mark.parametrize("seed", range(12))
def test_schedule_pinned_to_the_reference_loop_source(seed, reference_live):
    """The policy's oracle is the reference's OWN statements: oracle/train_live.py cuts the `while not stop_train:` loop out of the
    unmodified steps/train_ctc.py (lines 159-231), execs it with stubs, and both the restatement (oracle/train_ref.py) and
    DevLossSchedule must reproduce its learning rates, roll-backs and final bookkeeping epoch by epoch."""
    rec = reference_live["schedule"]
    trace = rec["traces"][seed]
    assert trace["seed"] == seed
    losses, accs = train_ref.scripted_sequence(seed, 120)
    losses[0] = rec["first_loss"]   # below the initial loss_best = 1000 so that the counter is bound, as in any real run
    init_lr, decay, eps, epochs = 1e-3, 0.5, 0.05, 100
    assert (rec["init_lr"], rec["decay"], rec["end_adjust_acc"], rec["num_epoches"]) == (init_lr, decay, eps, epochs)
    live = [{"lr": lr, "rollback": rb} for lr, rb in zip(trace["lr"], trace["rollback"])]
    final = trace["final"]
    restated, rfinal = train_ref.schedule_trace(losses, accs, init_lr, decay, eps, epochs)
    sched = DevLossSchedule(init_lr, decay, eps)
    ours, count = [], 0
    while not sched.stop and count < epochs and count < len(losses):
        count += 1
        sched.begin_epoch()
        act = sched.update(losses[count - 1], accs[count - 1])
        ours.append(dict(act, lr=sched.learning_rate))
    assert len(live) == len(restated) == len(ours) == final["epochs"] == rfinal["epochs"]
    for a, b, c in zip(live, restated, ours):
        assert a["lr"] == pytest.approx(b["lr"], rel=0, abs=1e-18) and a["lr"] == pytest.approx(c["lr"], rel=0, abs=1e-18)
        assert a["rollback"] == b["rollback"] == c["rollback"]
    assert final["loss_best"] == rfinal["loss_best"] == sched.loss_best
    assert final["acc_best"] == rfinal["acc_best"] == sched.acc_best
    assert any(a["rollback"] for a in live)


def test_schedule_reproduces_the_unbound_counter_quirk():
    # first epoch inside the +-band around the initial 1000: the reference increments a variable it never assigned
    sched = DevLossSchedule(1e-3, 0.5, 0.05)
    with pytest.raises(UnboundLocalError):
        sched.update(1000.0, 0.1)
    with pytest.raises(UnboundLocalError):
        train_ref.schedule_trace([1000.0], [0.1], 1e-3, 0.5, 0.05, 5)


def test_package_roundtrip_cpu():
    m = CTC_Model(rnn_param=RNN_PARAM, num_class=11, drop_out=0.1)
    opt = torch.optim.Adam(m.parameters(), lr=1e-3)
    pkg = CTC_Model.save_package(m, optimizer=opt, epoch={"epoch": 3, "feature_type": "fbank", "n_feats": 40},
                                 loss_results=[3.0, 2.0, 1.5], dev_loss_results=[3.1, 2.2, 1.9], dev_cer_results=[0.1, 0.3, 0.4])
    m2, pkg2 = load_package(pkg, device="cpu")
    assert pkg2 is pkg and m2.num_class == 11 and m2.drop_out == 0.1
    for (k1, v1), (k2, v2) in zip(m.state_dict().items(), m2.state_dict().items()):
        assert k1 == k2 and torch.equal(v1, v2)


def test_checkpoint_interchange_with_reference(reference_live):
    """A package of ours has the reference's layout (keys, constructor fields, state_dict names and shapes, so the reference's
    constructor + load_state_dict accept it), and a package in the reference's layout, holding the reference's weights
    (re-created from the seed, verified by checksum), loads into ours unchanged."""
    rec = reference_live["checkpoint"]
    ours = CTC_Model(rnn_param=RNN_PARAM, num_class=11, drop_out=0.1)
    # ours -> reference (test_ctc.py:37-60 style)
    pkg = CTC_Model.save_package(ours, epoch={"epoch": 1})
    assert sorted(pkg.keys()) == rec["keys"]
    for k, v in rec["fields"].items():
        got = pkg[k]
        if k == "rnn_param":
            got = dict(got, rnn_type=got["rnn_type"].__name__)
        assert got == v, k
    assert [[k, list(v.shape)] for k, v in pkg["state_dict"].items()] == rec["state_dict"]
    # reference -> ours
    torch.manual_seed(rec["seed"])
    sd = CTC_Model(rnn_param=RNN_PARAM, num_class=11, drop_out=0.1).state_dict()
    for k, v in sd.items():
        assert abs(float(v.double().abs().sum()) - rec["checksum"][k]) <= 1e-9 * max(1.0, rec["checksum"][k]), k
    rpkg = dict(rec["fields"], state_dict=sd)
    rpkg["rnn_param"] = dict(rpkg["rnn_param"], rnn_type=getattr(nn, rpkg["rnn_param"]["rnn_type"]))
    m2, _ = load_package(rpkg, device="cpu")
    assert list(m2.state_dict()) == list(sd)
    for (k1, v1), (k2, v2) in zip(sd.items(), m2.state_dict().items()):
        assert k1 == k2 and torch.equal(v1, v2)
