"""Training-step time against the recurrent hidden size at cfg2's shape (T = 800, N = 32, 4 bidirectional LSTM layers with
BatchNorm): python tools/hidden_size_bench.py [--hidden 200,256,...] [--steps K] [--warmup W] [--out FILE.json]

Hidden sizes that are not a multiple of 128 run zero-padded at the next multiple; above 640 the recurrent kernels exchange
h_t / dG_t through global memory (DESIGN.md §3.2, §9). Per hidden size: --warmup untimed steps, then --steps timed steps
(forward + CTC loss + greedy decode + backward, CUDA events, a 192 MiB L2 flush before each), then one more pass of --steps
steps with every C-ABI call timed on its own (side-stream overlap off) for the per-launch recurrent kernel times. The GPU name
and its power limit (nvidia-smi query) are recorded beside the numbers."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from ctc_pytorch_b200 import _lib, ops, synth  # noqa: E402
from ctc_pytorch_b200.loss import CTCLoss  # noqa: E402
from ctc_pytorch_b200.model import CTC_Model, device_hidden  # noqa: E402


def power_limit_w():
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout
        return float(out.strip().splitlines()[0])
    except Exception:
        return None


def median(v):
    v = sorted(v)
    return v[len(v) // 2]


def run(H, steps, warmup, flush, dev):
    cfg = dict(synth.CONFIGS["cfg2"], H=H)
    torch.manual_seed(0)
    kw = synth.model_kwargs(cfg)
    m = CTC_Model(**kw).to(dev)
    m.train()
    x, frac, tg, tl = (t.to(dev) for t in synth.synthetic_batch(cfg["T"], cfg["N"], cfg["F"], cfg["C"], cfg["S"], 1))
    lossf = CTCLoss(reduction="sum")

    def step():
        out = m(x)
        il = (frac * out.shape[0]).long()
        loss = lossf(out, tg, il, tl) / x.shape[0]
        ops.greedy_decode(out, il)
        m.zero_grad(set_to_none=True)
        loss.backward()
        return loss

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    ts = []
    for _ in range(steps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        loss = step()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    # per-launch pass: every C-ABI call between its own pair of events, on one stream
    L = _lib.lib()
    per_call = {}
    orig = L.call

    def timed_call(nm, *a):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        r = orig(nm, *a)
        e.record()
        per_call.setdefault(nm, []).append((s, e))
        return r
    m.overlap_wgrad = m.overlap_gx = m.overlap_dg = False
    L.call = timed_call
    try:
        for _ in range(steps):
            flush.zero_()
            step()
        torch.cuda.synchronize()
    finally:
        L.call = orig
    launch_ms = {}
    for nm in ("ctcb200_lstm_fwd", "ctcb200_lstm_bwd"):
        v = [s.elapsed_time(e) for s, e in per_call.get(nm, [])]
        launch_ms[nm] = {"median_ms": median(v) if v else None, "launches_per_step": len(v) // steps}
    res = {"H": H, "device_hidden": device_hidden(H), "step_ms_median": median(ts), "step_ms_min": min(ts),
           "step_ms_max": max(ts), "steps": steps, "loss_last": float(loss.detach()), "recurrent_launch": launch_ms}
    del m
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--hidden", default="200,256,320,512,640,768,1024")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.steps < 1:
        raise SystemExit("--steps must be >= 1")
    dev = torch.device("cuda", torch.cuda.current_device())
    flush = torch.empty(192 << 20, dtype=torch.uint8, device=dev)
    rows = []
    for H in [int(v) for v in args.hidden.split(",")]:
        r = run(H, args.steps, args.warmup, flush, dev)
        print(json.dumps(r), flush=True)
        rows.append(r)
    cfg = synth.CONFIGS["cfg2"]
    doc = {"gpu": torch.cuda.get_device_name(dev), "power_limit_w": power_limit_w(),
           "shape": {k: cfg[k] for k in ("T", "N", "F", "C", "L")}, "precision": "bf16",
           "timing": "CUDA events per training step (fwd + CTC loss + greedy decode + bwd), 192 MiB L2 flush before each, "
                     "warm-up on every shape; recurrent launches timed one by one in a separate pass",
           "results": rows}
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(doc, fh, indent=1)
    print(json.dumps({k: v for k, v in doc.items() if k != "results"}))


if __name__ == "__main__":
    main()
