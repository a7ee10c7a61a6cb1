"""GPU suite, multi-rank (`-m gpu`, needs >= 2 CUDA devices; skipped on a 1-GPU box): SURVEY.md §8(e)'s data-parallel
contract on real devices over NCCL — rank r of G takes utterances [r N/G, (r+1) N/G) of the padded batch, BatchNorm statistics
stay per rank, the per-layer in-backward all-reduces (dist.GradSync) must leave every rank with the MEAN OF THE PER-SHARD
gradients. The oracle is run on every shard separately on the CPU and averaged, exactly as §8(e) prescribes.
"""
import json
import os
import socket

import pytest
import torch
import torch.nn as nn

pytestmark = pytest.mark.gpu

from oracle import model_ref  # noqa: E402


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


CASE = dict(T=40, N=12, F=40, H=256, L=3, C=20, S=6, seed=17)


def _rank_main(rank, world, port, out, precision):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from ctc_pytorch_b200.model import CTC_Model
    from ctc_pytorch_b200.loss import CTCLoss
    from ctc_pytorch_b200.dist import GradSync, shard_range
    c = CASE
    torch.manual_seed(c["seed"])
    rnn_param = {"rnn_input_size": c["F"], "rnn_hidden_size": c["H"], "rnn_layers": c["L"], "rnn_type": nn.LSTM,
                 "bidirectional": True, "batch_norm": True}
    m = CTC_Model(rnn_param=rnn_param, num_class=c["C"], drop_out=0.0).to("cuda:%d" % rank)
    m.precision = precision
    x, frac, tg, tl = model_ref.synthetic_batch(c["T"], c["N"], c["F"], c["C"], c["S"], c["seed"])
    lo, hi = shard_range(c["N"], rank, world)
    m.grad_sync = GradSync(weight=(hi - lo) * world / float(c["N"]))
    m.train()
    dev = "cuda:%d" % rank
    for _ in range(2):      # twice: the second pass exercises buffer reuse / event reuse across steps
        m.zero_grad(set_to_none=True)
        out_ = m(x[lo:hi].to(dev))
        il = (frac[lo:hi].to(dev) * out_.shape[0]).long()
        loss = CTCLoss(reduction="sum")(out_, tg[lo:hi].to(dev), il, tl[lo:hi].to(dev)) / (hi - lo)
        loss.backward()
    torch.cuda.synchronize()
    grads = {k: p.grad.detach().cpu() for k, p in m.named_parameters()}
    torch.save(grads, "%s.rank%d" % (out, rank))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("precision", ["bf16", "x3"])
def test_two_rank_gradients_equal_mean_of_per_shard_oracle(tmp_path, precision):
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    import torch.multiprocessing as mp
    from ctc_pytorch_b200.dist import shard_range
    world = 2
    out = str(tmp_path / "grads")
    mp.spawn(_rank_main, args=(world, _free_port(), out, precision), nprocs=world, join=True)
    g0, g1 = torch.load(out + ".rank0"), torch.load(out + ".rank1")
    for k in g0:   # every rank holds the same reduced gradient
        assert torch.equal(g0[k], g1[k]), k
    # per-shard oracle (reference semantics: each call divides by its own batch size, BatchNorm over its own rows), weighted mean
    c = CASE
    torch.manual_seed(c["seed"])
    ref = model_ref.RefAcousticModel(c["F"], c["H"], c["L"], c["C"], batch_norm=True)
    x, frac, tg, tl = model_ref.synthetic_batch(c["T"], c["N"], c["F"], c["C"], c["S"], c["seed"])
    want = {k: torch.zeros_like(p) for k, p in ref.named_parameters()}
    ref.train()
    sd0 = {k: v.clone() for k, v in ref.state_dict().items()}
    for r in range(world):
        lo, hi = shard_range(c["N"], r, world)
        ref.load_state_dict(sd0)
        ref.zero_grad()
        o = ref(x[lo:hi])
        il = (frac[lo:hi] * o.shape[0]).long()
        (nn.CTCLoss(reduction="sum")(o, tg[lo:hi], il, tl[lo:hi]) / (hi - lo)).backward()
        for k, p in ref.named_parameters():
            want[k] += p.grad * ((hi - lo) / float(c["N"]))
    worst = 0.0
    for k in want:
        e = float((g0[k].double() - want[k].double()).norm() / (want[k].double().norm() + 1e-30))
        worst = max(worst, e)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    os.makedirs(os.path.join(root, "gpurun_out"), exist_ok=True)
    with open(os.path.join(root, "gpurun_out", "parity_report.jsonl"), "a") as fh:
        fh.write(json.dumps(dict(test="two_rank_mean_of_shard_gradients", precision=precision, world=world,
                                 grad_rel_l2_worst=worst)) + "\n")
    assert worst < (3e-2 if precision == "bf16" else 1e-3), worst
