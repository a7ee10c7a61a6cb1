"""TEST INFRASTRUCTURE ONLY — restatement of the learning-rate / rollback policy inside `main` of
timit/steps/train_ctc.py:162-231 as a pure function of the per-epoch (dev_loss, acc) sequence.

The reference's loop cannot be imported (it lives inside `main`, behind Visdom and the Kaldi data layer), so this is a
restatement; it is pinned by tests/test_train_host.py::test_schedule_pinned_to_the_reference_loop_source, which execs the
reference's own loop text with stubs (oracle/train_live.py) and compares epoch by epoch. Used to check
ctc_pytorch_b200.train.DevLossSchedule on random sequences.
"""


def schedule_trace(dev_losses, accs, init_lr, decay, end_adjust_acc, num_epoches):
    """Returns a list of per-epoch dicts: lr used, snapshot / best / rollback flags, and whether training stops after it."""
    count = 0
    learning_rate = init_lr          # train_ctc.py:163
    loss_best = 1000                 # :164
    loss_best_true = 1000            # :165
    adjust_rate_flag = False         # :166
    stop_train = False               # :167
    adjust_time = 0                  # :168
    acc_best = 0                     # :169
    trace = []
    while not stop_train:            # :175
        if count >= num_epoches:     # :176
            break
        if count >= len(dev_losses):
            break
        count += 1
        if adjust_rate_flag:         # :181
            learning_rate *= decay
            adjust_rate_flag = False
        dev_loss, acc = dev_losses[count - 1], accs[count - 1]
        ev = {"lr": learning_rate, "snapshot": False, "best": False, "rollback": False, "stop": False}
        if dev_loss < (loss_best - end_adjust_acc):          # :197
            loss_best = dev_loss
            loss_best_true = dev_loss
            adjust_rate_count = 0
            ev["snapshot"] = True
        elif dev_loss < loss_best + end_adjust_acc:          # :203
            adjust_rate_count += 1                           # UnboundLocalError if no epoch improved before
            if dev_loss < loss_best and dev_loss < loss_best_true:
                loss_best_true = dev_loss
                ev["snapshot"] = True
        else:                                                # :209
            adjust_rate_count = 10
        if acc > acc_best:                                   # :212
            acc_best = acc
            ev["best"] = True
        if adjust_rate_count == 10:                          # :220
            adjust_rate_flag = True
            adjust_time += 1
            adjust_rate_count = 0
            if loss_best > loss_best_true:
                loss_best = loss_best_true
            ev["rollback"] = True
        if adjust_time == 8:                                 # :230
            stop_train = True
            ev["stop"] = True
        trace.append(ev)
    return trace, {"loss_best": loss_best, "acc_best": acc_best, "epochs": count}


def scripted_sequence(seed, n):
    """Seeded per-epoch (dev loss, accuracy) sequence mixing improvements, plateaus inside the +-end_adjust_acc band and
    divergences, so that every branch of the policy is exercised."""
    import random
    rng = random.Random(seed)
    loss, out_l, out_a = 40.0 + rng.random() * 10, [], []
    for i in range(n):
        r = rng.random()
        if r < 0.45:
            loss -= rng.random() * 2.0          # clear improvement
        elif r < 0.8:
            loss += (rng.random() - 0.5) * 0.02  # plateau inside the +-end_adjust_acc band
        else:
            loss += rng.random() * 3.0          # divergence -> immediate halving
        out_l.append(loss)
        out_a.append(rng.random())
    return out_l, out_a
