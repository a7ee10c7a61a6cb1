#!/usr/bin/env python
"""Benchmark of the CTC acoustic hot path (BASELINE.json: utterances/sec at T=800, N=32, feat=40, C=62).

    python bench.py --gpus 1 --steps K --warmup W            # our arm (sm_100a kernels through the C ABI)
    python bench.py --impl reference --steps K --warmup W    # the UNMODIFIED reference's own CPU path on the host cores

One "step" = one pass of the training hot loop of timit/steps/train_ctc.py:44-65 over one synthetic batch of the named
shape (default cfg2: 4 x BiLSTM-512 + BatchNorm, T=800, N=32 per GPU): forward, CTC loss / batch, frame arg-max + collapse +
edit distance (compute_wer), backward, (N>1: gradient all-reduce, bucketed per layer and overlapped with the backward pass),
Adam step.
  value  utterances/s with the batch already resident in HBM;
  e2e    the same step driven through the public classes with HOST buffers: pinned H2D of features / labels / lengths and
         D2H of the loss and the (errors, tokens) pair inside the timed region.
Default: weak scaling of cfg2 (every rank its own N=32 shard). Every run also measures SURVEY.md §8(e)'s partitioning
(cfg4, N=64 sharded N/G per rank: strong scaling) as the secondary `strong_cfg4` object; `--scaling strong` makes that the
headline instead. `--precision x3` selects the split-bf16 (3-product) operand mode whose gradients meet the fp32 1e-3 bar.
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.nn as nn  # noqa: E402

from ctc_pytorch_b200 import synth  # noqa: E402

CFG = synth.CONFIGS


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback")


def ncu_traffic(config, kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` summary."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(path):
        return None, None
    d = json.load(open(path))
    ent = d.get(config, {}).get(kernel)
    if not ent:
        return None, None
    return ent["dram_bytes"], ent.get("source")


class ClockSampler(object):
    """nvidia-smi clock / throttle sampling during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.rows = []          # (host time of arrival, csv line)
        self.windows = []       # [t0, t1] host-time intervals of the timed regions
        self.proc = None
        self.index = index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "25"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.monotonic(), line.strip()))

    def open_window(self):
        self.windows.append([time.monotonic(), None])

    def close_window(self):
        self.windows[-1][1] = time.monotonic()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, r in self.rows:
            # the process is started before the warm-up (nvidia-smi needs a few hundred ms to come up); only samples taken
            # inside a timed region count
            if self.windows and not any(w0 <= ts <= (w1 if w1 is not None else ts) for w0, w1 in self.windows):
                continue
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons),
                "window": "samples every 25 ms inside the timed regions (device-resident loop + e2e loop)"}


def make_batch(cfg, seed, lo=0, hi=None):
    """Seeded synthetic batch of the config's global shape; [lo, hi) selects a rank's shard of the padded batch."""
    x, frac, tg, tl = synth.synthetic_batch(cfg["T"], cfg["N"], cfg["F"], cfg["C"], cfg["S"], seed)
    hi = cfg["N"] if hi is None else hi
    return tuple(t[lo:hi].contiguous() for t in (x, frac, tg, tl))


def rnn_param(cfg):
    """rnn_param dict of a CONFIGS entry (helper for the scripts under tools/)."""
    return synth.model_kwargs(cfg)["rnn_param"]


def workload_name(name, cfg, per_gpu):
    return "%s: T=%d N=%d/GPU feat=%d C=%d %s%dxBiLSTM-%d+BN" % (
        name, cfg["T"], per_gpu, cfg["F"], cfg["C"], "2xConv2d+" if cfg.get("cnn") else "", cfg["L"], cfg["H"])


# --------------------------------------------------------------------------------------------------- reference arm
def cpu_threads():
    """Threads for the CPU arm. Measured on the GPU box's host (128 logical CPUs, profiles/cpu_thread_scaling_r1.txt):
    the reference's nn.LSTM step peaks at 16 intra-op threads (3.3 utt/s) and gets slower beyond (1.6 at 32, 0.6 at
    64), so 16 is "all the threads it can use"; CTCB200_CPU_THREADS overrides."""
    env = os.environ.get("CTCB200_CPU_THREADS")
    if env:
        return max(1, int(env))
    return max(1, min(16, os.cpu_count() or 1))


def reference_step_rate(cfg, steps, warmup, threads, budget_s):
    """The reference's own CPU path, unmodified: models/model_ctc.py CTC_Model + nn.CTCLoss(reduction='sum') + torch.optim.Adam
    driven by steps/train_ctc.py's run_epoch (forward, loss / batch, .item(), arg-max, compute_wer, zero_grad, backward,
    optimizer step), imported through oracle/ref_shim.py from /root/reference or its byte-for-byte staged copy oracle/_ref/
    (oracle/build_ref.py). One run_epoch call over a one-batch iterator = one step of the loop. Returns
    (utt/s, s/step, steps actually timed, source)."""
    from oracle import ref_shim
    ref = ref_shim.load()
    run_epoch = ref_shim.load_train_loop()
    torch.set_num_threads(threads)
    torch.manual_seed(0)
    model = ref.CTC_Model(**synth.model_kwargs(cfg))
    opt = torch.optim.Adam(model.parameters(), lr=1e-3, weight_decay=0.005)   # train_ctc.py:145 with conf/ctc_config.yaml
    loss_fn = nn.CTCLoss(reduction="sum")                                     # train_ctc.py:144
    batches = []
    for b in range(2):
        x, frac, tg, tl = make_batch(cfg, 1 + b)
        batches.append((x, frac, tg, tl, ["utt%d" % i for i in range(x.shape[0])]))
    cpu = torch.device("cpu")
    t_begin = time.perf_counter()
    for w in range(warmup):
        run_epoch(0, model, [batches[w % 2]], loss_fn, cpu, optimizer=opt, print_every=10 ** 9, is_training=True)
        if time.perf_counter() - t_begin > 0.4 * budget_s:
            break
    done = 0
    t0 = time.perf_counter()
    for k in range(steps):
        run_epoch(1, model, [batches[k % 2]], loss_fn, cpu, optimizer=opt, print_every=10 ** 9, is_training=True)
        done += 1
        if time.perf_counter() - t_begin > budget_s and done >= 3:
            break
    dt = time.perf_counter() - t0
    src = "oracle/_ref (staged copy of the unmodified reference)" if ref_shim.is_staged_copy() else "/root/reference"
    return cfg["N"] * done / dt, dt / done, done, src


def run_reference(args, name, cfg, rank, world):
    if rank != 0:
        return
    from oracle import ref_shim
    if not ref_shim.available():
        emit({"impl": "reference", "unavailable": "reference modules not staged: run __graft_entry__.build() where "
                                                  "/root/reference is mounted (oracle/build_ref.py)"})
        return
    cores = cpu_threads()
    budget = float(os.environ.get("CTCB200_REF_BUDGET_S", "420"))
    rate, sec, done, src = reference_step_rate(cfg, max(1, args.steps), args.warmup, cores, budget)
    sample = "full %s batches (N=%d utterances per step), %d timed steps, %d threads; unmodified run_epoch + CTC_Model from %s" % (
        name, cfg["N"], done, cores, src)
    line = {
        "impl": "reference", "metric": "utterances/sec (training step)", "value": rate, "unit": "utt/s",
        "n_gpus": args.gpus, "steps": done, "warmup": args.warmup, "ms_per_step": sec * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(name, cfg, cfg["N"]) + "; fwd + CTC loss + arg-max/collapse/edit distance + bwd + Adam",
                   "global_batch": cfg["N"], "host_threads": cores, "steps_requested": args.steps},
        "cpu_baseline": {"value": rate, "unit": "utt/s", "cores": cores, "kind": "reference", "sample": sample},
        "e2e": {"value": rate, "unit": "utt/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# -------------------------------------------------------------------------------------------------------- our arm
class Job(object):
    """Model + optimizer + batches of one (config, shard) on this rank's GPU, and the step function."""

    def __init__(self, name, cfg, rank, world, dev, precision, strong, n_batches=4):
        from ctc_pytorch_b200.model import CTC_Model
        from ctc_pytorch_b200.loss import CTCLoss
        from ctc_pytorch_b200.dist import GradSync, shard_range
        self.name, self.cfg, self.dev, self.world = name, cfg, dev, world
        if strong:
            self.lo, self.hi = shard_range(cfg["N"], rank, world)
        else:
            self.lo, self.hi = 0, cfg["N"]
        self.n_local = self.hi - self.lo
        self.n_global = cfg["N"] if strong else cfg["N"] * world
        torch.manual_seed(0)
        self.model = CTC_Model(**synth.model_kwargs(cfg)).to(dev)
        self.model.precision = precision
        # the reference's optimizer (train_ctc.py:145: Adam + L2 weight decay), torch's single-launch (fused) implementation
        self.opt = torch.optim.Adam(self.model.parameters(), lr=1e-3, weight_decay=0.005, fused=True)
        self.loss_fn = CTCLoss(reduction="sum")
        # strong scaling: every rank's loss is divided by ITS shard size (train_ctc.py:48), so the full-batch gradient is the
        # shard-size-weighted mean of the rank gradients
        weight = (self.n_local * world / float(self.n_global)) if strong else 1.0
        self.sync = GradSync(weight=weight) if world > 1 else None
        self.model.grad_sync = self.sync
        self.model.train()
        self.host = []
        for b in range(n_batches):
            seed = (100 * rank + b) if not strong else (1000 + b)
            hb = make_batch(cfg, seed, self.lo, self.hi)
            self.host.append(tuple(t.pin_memory() for t in hb))
        self.devb = [tuple(t.to(dev) for t in hb) for hb in self.host]
        self.h2d_bytes = sum(t.numel() * t.element_size() for t in self.host[0])
        self.wer_acc = torch.zeros(2, dtype=torch.int64, device=dev)
        # pinned landing slots of the per-step results of the end-to-end loop: (loss f32[1], (errors, tokens) int64[2]) = 20 bytes
        self.fetched = [(torch.full((1,), float("nan")).pin_memory(), torch.full((2,), -1, dtype=torch.int64).pin_memory())
                        for _ in range(64)]
        self.fetch_i = 0
        self.keep_last = False  # --dump-outputs: hold on to what this step hands back to its caller
        self.last = None

    def step(self, b, fetch=False, comm=True):
        from ctc_pytorch_b200 import ops
        x, frac, tg, tl = b
        model = self.model
        model.grad_sync = self.sync if comm else None
        out = model(x)
        out_len, bsz, _ = out.size()
        il = (frac * out_len).long()
        loss = self.loss_fn(out, tg, il, tl) / bsz
        # train_ctc.py:51-52: arg-max + compute_wer (collapse + edit distance), here on the device
        _, labels, lens = ops.greedy_decode(out, il, blank=0)
        dist_ = ops.edit_distance(labels, lens, tg, tl)
        self.wer_acc[0] += dist_.sum()
        self.wer_acc[1] += tl.sum()
        self.opt.zero_grad(set_to_none=True)
        loss.backward()        # with grad_sync set, the per-layer all-reduces are launched and joined inside the backward pass
        self.opt.step()
        if self.keep_last:
            self.last = {"loss": loss, "log_probs": out, "greedy_labels": labels, "greedy_lengths": lens, "edit_distance": dist_}
        if fetch:
            # device -> host read of this step's result into pinned memory, every step, without stalling the launch queue — the
            # policy of the product's epoch loop (ctc_pytorch_b200/train.py run_epoch: device-side accumulation, no per-step
            # host synchronisation); timed_loop synchronises before it stops the clock and checks that every slot arrived
            slot = self.fetched[self.fetch_i % len(self.fetched)]
            self.fetch_i += 1
            slot[0].copy_(loss.detach().reshape(1), non_blocking=True)
            slot[1].copy_(self.wer_acc, non_blocking=True)
            return slot
        return loss


PER_STEP = None   # list of per-step event times of every timed loop when --per-step is given


def timed_loop(job, steps, flush, world, e2e, keep_last=False):
    import torch.distributed as dist

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    marks = [torch.cuda.Event(enable_timing=True) for _ in range(steps)] if PER_STEP is not None else None
    barrier()
    e0.record()
    for k in range(steps):
        if e2e:
            hb = job.host[k % len(job.host)]
            b = tuple(t.to(job.dev, non_blocking=True) for t in hb)
            job.step(b, fetch=True)
        else:
            flush.zero_()  # L2 flush between steps (counted inside the timed region: ~0.03 ms)
            job.keep_last = keep_last and k == steps - 1   # only the final step's results are held (--dump-outputs)
            job.step(job.devb[k % len(job.devb)])
        if marks is not None:
            marks[k].record()
    e1.record()
    barrier()
    if e2e:   # every step's result reached the host inside the timed region
        for k in range(min(steps, len(job.fetched))):
            lo, we = job.fetched[(job.fetch_i - 1 - k) % len(job.fetched)]
            if not (math.isfinite(float(lo[0])) and int(we[1]) > 0):
                raise RuntimeError("end-to-end loop: the result of a step did not arrive on the host")
    if marks is not None:   # diagnostic (--per-step): where inside the timed region the time went
        PER_STEP.append({"e2e": bool(e2e), "ms": [round((e0 if k == 0 else marks[k - 1]).elapsed_time(marks[k]), 3) for k in range(steps)]})
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=job.dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item())


DUMP_SAMPLE = 1 << 16          # entries kept of each parameter-sized tensor
DUMP_LIMIT = 64 * 1024 * 1024  # bytes written in all


def dump_outputs(job, path):
    """Writes what the last step of `job` handed back to its caller as <path>/<name>.npy (float32, or float64 for the loss
    and the integer results): the loss, the log-probs, the greedy decode and its edit distances, and the state the step left
    behind, i.e. every parameter's gradient, every parameter after the optimizer step and the BatchNorm running statistics.
    Tensors with more than DUMP_SAMPLE entries are reduced to a fixed sample whose positions are seeded by the tensor's name,
    so that two builds of the project can be compared array for array."""
    import zlib
    import numpy as np

    def sample(name, t):
        flat = t.detach().reshape(-1)
        if flat.numel() <= DUMP_SAMPLE:
            return flat
        rng = np.random.default_rng(zlib.crc32(name.encode()))
        idx = np.sort(rng.choice(flat.numel(), DUMP_SAMPLE, replace=False))
        return flat[torch.from_numpy(idx).to(flat.device)]

    last = job.last
    arrays = {"loss": last["loss"].detach().double().reshape(1), "log_probs": last["log_probs"].detach().float()}
    for k in ("greedy_labels", "greedy_lengths", "edit_distance"):
        arrays[k] = last[k].double()
    for k, p in job.model.named_parameters():
        arrays["grad." + k] = sample("grad." + k, p.grad).float()
        arrays["param." + k] = sample("param." + k, p).float()
    for k, b in job.model.named_buffers():
        if b.is_floating_point():
            arrays["buffer." + k] = sample("buffer." + k, b).float()
    arrays = {k: v.cpu().numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise RuntimeError("--dump-outputs: %d bytes exceed the %d byte limit" % (total, DUMP_LIMIT))
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a)


def run_ours(args, name, cfg, rank, world):
    from ctc_pytorch_b200 import _lib
    import torch.distributed as dist

    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    L = _lib.lib()
    strong = args.scaling == "strong"
    job = Job(name, cfg, rank, world, dev, args.precision, strong)
    T, F, C, H, Lyr = cfg["T"], cfg["F"], cfg["C"], cfg["H"], cfg["L"]
    N = job.n_local
    flush = torch.empty(192 * 1024 * 1024, dtype=torch.uint8, device=dev)   # larger than the 126 MB L2
    warm = max(args.warmup, 3)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for w in range(warm):
        job.step(job.devb[w % len(job.devb)])

    # ---- timed region 1: inputs resident in HBM ----
    sampler.open_window()
    launches0 = L.launches
    ms_dev = timed_loop(job, args.steps, flush, world, e2e=False, keep_last=bool(args.dump_outputs))
    launches = L.launches - launches0
    sampler.close_window()
    if args.dump_outputs:
        job.keep_last = False
        if rank == 0:
            dump_outputs(job, args.dump_outputs)
        job.last = None
    # ---- timed region 2: end to end from host buffers ----
    sampler.open_window()
    ms_e2e = timed_loop(job, args.steps, flush, world, e2e=True)
    sampler.close_window()
    clocks = sampler.stop() if rank == 0 else None
    d2h_bytes = 4 + 16

    # ---- secondary measurements (all ranks take part in the collectives) ----
    other_precision = None
    if args.both_precisions:
        alt = "x3" if args.precision == "bf16" else "bf16"
        job.model.precision = alt
        for w in range(3):
            job.step(job.devb[w % len(job.devb)])
        k_alt = args.steps
        ms_alt = timed_loop(job, k_alt, flush, world, e2e=False)
        job.model.precision = args.precision
        other_precision = {"precision": alt, "ms_per_step": ms_alt / k_alt, "value": job.n_global * k_alt / (ms_alt * 1e-3),
                           "unit": "utt/s", "steps": k_alt}
    strong_line = None
    if args.strong_cfg4 and not strong and not (name == "cfg4"):
        c4 = CFG["cfg4"]
        job4 = Job("cfg4", c4, rank, world, dev, args.precision, True, n_batches=2)
        for w in range(3):
            job4.step(job4.devb[w % 2])
        k4 = args.steps
        ms4 = timed_loop(job4, k4, flush, world, e2e=False)
        strong_line = {"config": workload_name("cfg4", c4, job4.n_local), "scaling": "strong", "global_batch": c4["N"],
                       "per_gpu_batch": job4.n_local, "n_gpus": world, "steps": k4, "ms_per_step": ms4 / k4,
                       "value": c4["N"] * k4 / (ms4 * 1e-3), "unit": "utt/s",
                       "limiter": "the recurrence is latency-bound: T*L dependent time steps per pass cost the same for 8 as for "
                                  "64 utterances per GPU, so sharding the batch only shrinks the GEMM / streaming part of the step"}
        del job4
        torch.cuda.empty_cache()

    if rank != 0:
        return
    # ---- per-kernel pass (rank 0, N=1 semantics): device time of every C-ABI call, CUDA events on the launch stream ----
    per_call = {}
    orig_call = L.call

    def timed_call(nm, *a):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        r = orig_call(nm, *a)
        e.record()
        per_call.setdefault(nm, []).append((s, e))
        return r
    L.call = timed_call
    prof_steps = args.steps
    overlap_was, gx_was, dg_was = job.model.overlap_wgrad, job.model.overlap_gx, job.model.overlap_dg
    # kernels timed one at a time on one stream (the timed steps above overlap the wgrad GEMMs with BPTT and stream the input
    # projection under the forward recurrence)
    job.model.overlap_wgrad = job.model.overlap_gx = job.model.overlap_dg = False
    for k in range(prof_steps):
        flush.zero_()
        job.step(job.devb[k % len(job.devb)], comm=False)  # rank 0 only: no collective in this diagnostic pass
    torch.cuda.synchronize()
    L.call = orig_call
    job.model.overlap_wgrad, job.model.overlap_gx, job.model.overlap_dg = overlap_was, gx_was, dg_was
    kern_ms = {nm: sum(s.elapsed_time(e) for s, e in v) / prof_steps for nm, v in per_call.items()}
    kern_cnt = {nm: len(v) // prof_steps for nm, v in per_call.items()}
    step_ms_prof = sum(kern_ms.values())

    pk = peaks()
    Tr = T // 2 if cfg.get("cnn") else T     # frames the recurrence runs over (the CNN front halves the time axis)
    # dominant kernels: the persistent recurrent kernels (tensor-core work, latency bound by the per-step hand-off)
    prods = 3.0 if args.precision == "x3" else 1.0
    rec_flops_launch = 2.0 * Tr * 2 * 4 * H * H * N           # algorithmic: one layer, both directions (x3 mode issues 3x this)
    fwd_ms = kern_ms.get("ctcb200_lstm_fwd", 0.0) / max(1, kern_cnt.get("ctcb200_lstm_fwd", 1))
    bwd_ms = kern_ms.get("ctcb200_lstm_bwd", 0.0) / max(1, kern_cnt.get("ctcb200_lstm_bwd", 1))
    dom_name, dom_ms = ("lstm_bwd_kernel", bwd_ms) if bwd_ms >= fwd_ms else ("lstm_fwd_kernel", fwd_ms)
    ach = rec_flops_launch / (dom_ms * 1e-3) / 1e12 if dom_ms > 0 else 0.0
    traffic, traffic_src = ncu_traffic(name, dom_name)
    dsmem = None
    p_dsmem = os.path.join(ROOT, "profiles", "dsmem_microbench.json")
    if os.path.exists(p_dsmem):
        dsmem = json.load(open(p_dsmem))
    roofline = {"kernel": dom_name, "bound": "tensor", "achieved": ach, "peak": pk["tf_sust"], "unit": "TFLOP/s",
                "frac": ach / pk["tf_sust"], "traffic": traffic,
                "traffic_unit": "bytes per launch (%s)" % (traffic_src or "no ncu capture for this config"),
                "peak_source": pk["src"] + " (sustained bf16)", "avg_launch_ms": dom_ms, "us_per_timestep": dom_ms * 1e3 / Tr,
                "tensor_products_per_algorithmic_flop": prods,
                "note": "recurrence: T dependent steps per launch; each step is a cluster-wide hand-off of h_t / dG_t "
                        "(DSMEM bulk copies + mbarriers) around a [4H x H] x [H x 16] product, so the kernel is latency-bound, "
                        "not tensor-bound (DESIGN.md 3.2); the dense GEMMs' fraction is under rooflines_other"}
    if dsmem:
        roofline["dsmem_microbench"] = dsmem
    # secondary rooflines: all dense GEMM launches together, and the CTC alpha/beta sweep
    rows = Tr * N
    gemm_flops = 0.0
    I0 = (32 * 10) if cfg.get("cnn") else F
    for l in range(Lyr):
        I = I0 if l == 0 else 2 * H
        gemm_flops += 2.0 * rows * 8 * H * I * (3 if (l > 0 or cfg.get("cnn")) else 2)   # Gx, dWih (+ dX)
        gemm_flops += 2.0 * rows * 8 * H * H                          # dWhh (both directions)
    gemm_flops += 3 * 2.0 * rows * 2 * H * C
    gemm_ms = kern_ms.get("ctcb200_gemm_tn_bf16", 0.0) + kern_ms.get("ctcb200_gemm_atb_bf16", 0.0)   # K-major + MN-major launches
    ctc_bytes = 2.0 * Tr * N * C * 4
    ctc_ms = kern_ms.get("ctcb200_ctc_loss_fwd", 0.0) + kern_ms.get("ctcb200_ctc_loss_bwd", 0.0)
    extra = {
        "gemm_all": {"bound": "tensor", "achieved": gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms else None,
                     "peak": pk["tf_sust"], "unit": "TFLOP/s", "ms_per_step": gemm_ms,
                     "note": "algorithmic flops of the RNN-stack contractions; x3 mode issues 3 tensor products per flop"},
        "ctc_alpha_beta": {"bound": "hbm", "achieved": ctc_bytes / (ctc_ms * 1e-3) / 1e9 if ctc_ms else None,
                           "peak": pk["hbm"], "unit": "GB/s", "ms_per_step": ctc_ms,
                           "note": "N=32 is latency-bound (T dependent steps per warp); saturating-batch sweep: profiles/ctc_sweep_r2.json"},
        "kernel_ms_per_step": {k: round(v, 4) for k, v in sorted(kern_ms.items(), key=lambda kv: -kv[1])},
        "kernel_share_of_step": {k: round(v / step_ms_prof, 4) for k, v in sorted(kern_ms.items(), key=lambda kv: -kv[1])},
    }
    for k in ("gemm_all", "ctc_alpha_beta"):
        if extra[k]["achieved"]:
            extra[k]["frac"] = extra[k]["achieved"] / extra[k]["peak"]

    # ---- CPU baseline on the host cores: the unmodified reference on a bounded sample (2 full-size steps after 1 warm-up) ----
    cores = cpu_threads()
    cpu_base = None
    if not args.no_cpu_baseline:
        from oracle import ref_shim
        if ref_shim.available():
            rate, sec, done, src = reference_step_rate(cfg, 2, 1, cores, 90.0)
            cpu_base = {"value": rate, "unit": "utt/s", "cores": cores, "kind": "reference",
                        "sample": "%d timed steps of full %s batches (N=%d) after 1 warm-up step; unmodified run_epoch + CTC_Model "
                                  "from %s" % (done, name, cfg["N"], src)}
        else:
            cpu_base = {"value": None, "unit": "utt/s", "cores": cores, "kind": "reference",
                        "sample": "unavailable: reference modules not staged (oracle/build_ref.py)"}

    total_utts = job.n_global * args.steps
    line = {
        "metric": "utterances/sec (training step)", "value": total_utts / (ms_dev * 1e-3), "unit": "utt/s",
        "n_gpus": world, "steps": args.steps, "warmup": warm, "ms_per_step": ms_dev / args.steps,
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "bf16" if args.precision == "bf16" else "bf16x3", "data": "synthetic",
        "config": {"workload": workload_name(name, cfg, N) + "; fwd + CTC loss + arg-max/collapse/edit distance + bwd"
                               "%s + Adam" % (" + per-layer gradient all-reduce" if world > 1 else ""),
                   "global_batch": job.n_global, "parallelism": "dp%d" % world,
                   "timing": "CUDA events, max over ranks, 192 MiB L2 flush write between timed steps",
                   "numerics": ("bf16 tensor-core operands, fp32 accumulate/state/loss" if args.precision == "bf16" else
                                "split-bf16 operands (hi+lo, 3 tensor-core products per contraction), fp32 accumulate/state/loss")},
        "e2e": {"value": total_utts / (ms_e2e * 1e-3), "unit": "utt/s", "h2d_bytes_per_step": job.h2d_bytes,
                "d2h_bytes_per_step": d2h_bytes, "ms_per_step": ms_e2e / args.steps,
                "note": "every step: pinned H2D of x/frac/targets/lengths, D2H of the loss and the (errors, tokens) pair into pinned "
                        "memory (asynchronous, like the product's run_epoch: no per-step host synchronisation; all results "
                        "verified on the host before the clock stops)"},
        "gpu_launches": launches,
        "clocks": clocks,
        "roofline": roofline,
        "rooflines_other": extra,
    }
    if cpu_base is not None:
        line["cpu_baseline"] = cpu_base
    if other_precision is not None:
        line["other_precision"] = other_precision
    if strong_line is not None:
        line["strong_cfg4"] = strong_line
    if PER_STEP is not None:
        line["per_step_ms"] = PER_STEP
    emit(line)


_REAL_STDOUT = None


def quiet_stdout():
    """Route fd 1 to stderr while the run is in progress (NCCL, the reference's run_epoch and friends print on stdout);
    the one JSON line goes to the real stdout through emit()."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    sys.stdout.flush()
    if _REAL_STDOUT is None:
        os.write(1, data)
    else:
        os.write(_REAL_STDOUT, data)


def main():
    quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default=None, choices=sorted(CFG))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--precision", default="bf16", choices=["bf16", "x3"])
    ap.add_argument("--both-precisions", dest="both_precisions", type=int, default=1,
                    help="also time a few steps in the other operand mode (other_precision object)")
    ap.add_argument("--strong-cfg4", dest="strong_cfg4", type=int, default=1,
                    help="also measure cfg4 sharded N/G per rank (strong_cfg4 object)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--per-step", dest="per_step", action="store_true",
                    help="diagnostic: also record the device time of every step of the timed loops (key per_step_ms)")
    ap.add_argument("--dump-outputs", dest="dump_outputs", default=None, metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.per_step:
        global PER_STEP
        PER_STEP = []
    name = args.config or ("cfg4" if args.scaling == "strong" else "cfg2")
    cfg = CFG[name]
    wd = int(os.environ.get("BENCH_WATCHDOG", "0"))
    if wd > 0:  # debugging aid: dump every thread's stack if the run is still alive after `wd` seconds
        import faulthandler
        faulthandler.dump_traceback_later(wd, repeat=True, file=sys.stderr)
    from ctc_pytorch_b200.dist import init_from_env
    if args.impl == "reference":
        rank = int(os.environ.get("RANK", "0"))
        run_reference(args, name, cfg, rank, int(os.environ.get("WORLD_SIZE", "1")))
        return
    rank, world = init_from_env()
    run_ours(args, name, cfg, rank, world)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
