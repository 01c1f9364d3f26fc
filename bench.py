#!/usr/bin/env python
"""bench.py -- the driver's measurement contract for the ReChorus training hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c1|c2|c3|c4|c5]
                    [--headline_only] [--no_cpu_baseline] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic input: forward (gather + interaction), BPR loss,
backward and the optimizer update -- the body of helpers/BaseRunner.py:193-206.  metric = training samples/s counted as
user x (1+neg) = B*C per step (BASELINE.json).

Workloads = BASELINE.json configs, in order:
  c1  BPRMF d=64 K=1 B=256 on an ML-1M-shaped synthetic corpus; a step = BaseRunner.fit's loop, value over one epoch
  c2  BPRMF d=64, 1 M users x 1 M items, K=99, B=4096                       <- the headline (metric is quoted on it)
  c3  NeuMF d=64, MLP [64,32,16], K=4, B=4096, 1 M x 1 M
  c4  SASRec L=50 d=64, 2 blocks, 4 heads, K=99, B=4096, 1 M items
  c5  BPRMF d=128, 100 M items (1 M users) row-range sharded over the ranks, K=255, B=4096 per GPU
Default: N=1 -> the c2 line, with compact lines of c1/c3/c4/c5 (c5 on one GPU, the anchor of its scaling curve) under
"workloads".  N>1 -> the sharded c5 over N ranks (configs 1-4 do not shard: replicas of them measure nothing); rank 0
then repeats c5 alone on its GPU ("n1_same_code") so that every N>1 line carries its own 1-GPU anchor.

Prints ONE JSON line (rank 0).  `value`: inputs already resident in HBM.  `e2e`: the same step through the public plugin
call with the batch coming from pinned host memory every step and the loss read back every step.  `roofline`: dominant
kernel, algorithmic bytes / CUDA-event time / measured peak.  `cpu_baseline`: the reference's own classes through its
own BaseRunner.fit on this box's host cores (kind "reference", from oracle/_ref/src), else the oracle port.

`--dump-outputs DIR` (c2): after the timed steps, the last timed step's results go to DIR/*.npy in float32 (see
dump_c2_outputs).  Inputs and initial tables are seeded, so two builds run with the same arguments can be compared
file by file.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
import types

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

WORKLOADS = {
    "c1": dict(model="BPRMF", n_users=6033, n_items=3126, d=64, B=256, K=1, rows=568_761,
               desc="BPRMF emb_dim=64, ML-1M-shaped synthetic corpus (6,032 users, 3,125 items, 568,761 rows), num_neg=1, batch=256"),
    "c2": dict(model="BPRMF", n_users=1_000_000, n_items=1_000_000, d=64, B=4096, K=99,
               desc="BPRMF emb_dim=64, 1M synthetic items (1M users), num_neg=99, batch=4096"),
    "c3": dict(model="NeuMF", n_users=1_000_000, n_items=1_000_000, d=64, B=4096, K=4, layers="[64, 32, 16]",
               desc="NeuMF (GMF + MLP [64,32,16]) emb_dim=64, 1M users x 1M items, num_neg=4, batch=4096"),
    "c4": dict(model="SASRec", n_users=1_000_000, n_items=1_000_000, d=64, B=4096, K=99, L=50, blocks=2, heads=4,
               desc="SASRec history_max=50 emb_dim=64, 2 blocks, 4 heads, 1M items, num_neg=99, batch=4096"),
    "c5": dict(model="BPRMF", n_users=1_000_000, n_items=100_000_000, d=128, B=4096, K=255,
               desc="BPRMF emb_dim=128, 100M synthetic items (1M users) row-range sharded, num_neg=255, batch=4096 per GPU"),
}
METRIC = "training samples/sec (user x (1+neg))"
UNIT = "user*item/s"
POOL = 8          # distinct pre-generated batches cycled through (fresh ids every step)
DATA = "synthetic (seeded uniform ids, N(0,0.01) tables)"


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), float(p.get("bf16_tflops", 1729.8)), "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1730.0, "fallback (B200_PROFILING.md: 6.65 TB/s copy, 1.73 PFLOP/s bf16)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines, self.windows = index, None, [], []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def window(self, t0, t1):
        """mark [t0, t1] (time.time()) as 'GPU under the benchmark load'"""
        self.windows.append((t0, t1))

    def n_in_windows(self):
        return len([1 for ts, _ in self.lines if any(a <= ts <= b for a, b in self.windows)])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()          # exact PID we started
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, ln in self.lines:
            if self.windows and not any(a <= ts <= b + 0.02 for a, b in self.windows):
                continue
            parts = [x.strip() for x in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------------
# synthetic data (seeded; ids uniform in [1, n) -- id 0 is the reference's padding id, data/README.md:13)
# ------------------------------------------------------------------------------------------------------

def make_batches(w, seed, pool=POOL):
    """host feed dicts shaped like the reference's collate output (models/BaseModel.py:135-152)"""
    g = torch.Generator().manual_seed(seed)
    B, C = w["B"], w["K"] + 1
    out = []
    for _ in range(pool):
        f = {"user_id": torch.randint(1, w["n_users"], (B,), generator=g, dtype=torch.int64),
             "item_id": torch.randint(1, w["n_items"], (B, C), generator=g, dtype=torch.int64)}
        if w["model"] == "SASRec":
            L = w["L"]
            lengths = torch.randint(1, L + 1, (B,), generator=g)
            lengths[0] = L                                   # one full-length row: the batch max length is L
            hist = torch.randint(1, w["n_items"], (B, L), generator=g) * (torch.arange(L).view(1, L) < lengths.view(B, 1))
            f["history_items"], f["lengths"] = hist, lengths
        out.append(f)
    return out


def to_feed(host, device, B, pin=False):
    f = {k: (v.pin_memory() if pin else v.to(device)) for k, v in host.items()}
    f["batch_size"], f["phase"] = B, "train"
    return f


def model_flags(w):
    fl = ["--emb_size", str(w["d"]), "--num_neg", str(w["K"])]
    if w["model"] == "NeuMF":
        fl += ["--layers", w["layers"]]
    if w["model"] == "SASRec":
        fl += ["--history_max", str(w["L"]), "--num_layers", str(w["blocks"]), "--num_heads", str(w["heads"])]
    return fl


def build_model(w, device, extra=()):
    from rechorus_b200 import plugin
    from rechorus_b200.optim import RowSparseOptimizer
    from rechorus_b200.runner import BaseRunner
    cls = getattr(plugin, w["model"])
    p = argparse.ArgumentParser()
    p = BaseRunner.parse_runner_args(p)
    p = cls.parse_model_args(p)
    a = p.parse_args(model_flags(w) + ["--table_mode", "fused", *extra])
    a.device, a.model_path, a.log_file = device, "/tmp/_b2r_bench.pt", ""
    torch.manual_seed(0)
    n_users = w["n_users"] if w["model"] != "SASRec" else 10          # SASRec has no user table
    model = cls(a, types.SimpleNamespace(n_users=n_users, n_items=w["n_items"])).to(device)
    model.optimizer = RowSparseOptimizer(model, "Adam", lr=1e-3, l2=0.0,     # reference defaults (BaseRunner.py:28-38)
                                         device_clock=(w["model"] != "BPRMF"))
    model.train()
    return model, a


class Dist:
    """barrier + max-over-ranks plumbing (NCCL is used for nothing else on configs 1-4)"""

    def __init__(self, world, device):
        self.world, self.device = world, device

    def barrier(self):
        if self.world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def max_ms(self, ms):
        if self.world > 1:
            t = torch.tensor([ms], device=self.device)
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
            ms = float(t.item())
        return ms


def timed_loop(dist, fn, steps, warmup, k0=0):
    """W untimed + exactly K timed steps bracketed by barrier + synchronize; CUDA events; max over ranks"""
    for k in range(warmup):
        fn(k0 + k)
    dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.time()
    e0.record()
    out = None
    for k in range(steps):
        out = fn(k0 + warmup + k)
    e1.record()
    dist.barrier()
    return dist.max_ms(e0.elapsed_time(e1)) / steps, out, (w0, time.time())


# ------------------------------------------------------------------------------------------------------
# c2: the headline -- BPRMF through model.train_step (one C call per step)
# ------------------------------------------------------------------------------------------------------

def run_c2(args, rank, world, local_rank, sampler):
    from rechorus_b200 import lib as L, ops
    device = torch.device("cuda", local_rank)
    w = WORKLOADS["c2"]
    B, C, d = w["B"], w["K"] + 1, w["d"]
    model, margs = build_model(w, device)
    lib = L.load()
    dist = Dist(world, device)
    host = make_batches(w, seed=1000 + rank)
    pinned = [(f["user_id"].pin_memory(), f["item_id"].pin_memory()) for f in host]
    feeds = [to_feed(f, device, B) for f in host]
    n_uniq = [int(torch.unique(f["item_id"]).numel()) for f in host]
    n_uniq_u = [int(torch.unique(f["user_id"]).numel()) for f in host]

    def step_resident(k):
        # the next batch is handed over too (as a prefetching data loader would): its index plan is built on
        # the library's side stream while this step's kernels run
        return model.train_step(feeds[k % POOL], feeds[(k + 1) % POOL])

    # ---- value: ids resident in HBM ------------------------------------------------------------------
    for k in range(args.warmup):
        step_resident(k)
    dist.barrier()
    ops.check_ids(device)
    tags = {"score_fwd": L.PROF_SCORE_FWD, "score_bwd_query": L.PROF_SCORE_BWDQ, "segment_adam_items": L.PROF_SEGMENT_I,
            "segment_adam_users": L.PROF_SEGMENT_U, "plan_items": L.PROF_PLAN_I, "loss": L.PROF_LOSS}
    # bracket the tagged kernels on every prof_every-th step: >= 10 samples whatever --steps is (the driver's 20-step
    # run gets a bracket on every other step), sparse on long runs so the brackets' events do not weigh on them
    prof_every = max(2, args.steps // 64)
    prof_steps = list(range(0, args.steps, prof_every))
    evs = {name: {k: (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
                  for k in prof_steps} for name in tags}
    for name in tags:                      # events must exist (be created) before cudaEventRecord from C
        for a, b in evs[name].values():
            a.record(); b.record()
    torch.cuda.synchronize()
    # host cost of enqueuing one step with an empty launch queue (no back-pressure): 40 steps right after a sync
    h0 = time.perf_counter()
    for k in range(40):
        step_resident(k)
    host_cost_ms = (time.perf_counter() - h0) * 1e3 / 40
    torch.cuda.synchronize()
    launches0 = lib.b2r_launch_count()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    dist.barrier()
    w0 = time.time()
    t0.record()
    for k in range(args.steps):
        if k % prof_every == 0:
            for name, tag in tags.items():
                a, b = evs[name][k]
                lib.b2r_profile_arm(tag, a.cuda_event, b.cuda_event)
        loss = step_resident(args.warmup + k)
    t1.record()
    host_ms_step = (time.time() - w0) * 1e3 / args.steps       # host time to enqueue a step (no sync inside the loop)
    dist.barrier()
    sampler.window(w0, time.time())
    if args.dump_outputs and rank == 0:
        dump_c2_outputs(args.dump_outputs, model, feeds[(args.warmup + args.steps - 1) % POOL], loss)
    launches = lib.b2r_launch_count() - launches0
    ms_step = dist.max_ms(t0.elapsed_time(t1)) / args.steps
    value = world * B * C / (ms_step * 1e-3)
    for tag in tags.values():
        lib.b2r_profile_arm(tag, None, None)
    kern_ms = {name: statistics.mean(a.elapsed_time(b) for a, b in evs[name].values()) for name in tags}
    kern_n = len(prof_steps)
    fused = kern_ms["score_bwd_query"] < 0.012       # the fused kernel replaces fwd + loss + bwd_query
    if fused:
        kern_ms["fused_score_loss_bwd"] = kern_ms.pop("score_fwd")
        kern_ms.pop("score_bwd_query")
        kern_ms.pop("loss")
    merged_apply = kern_ms.get("segment_adam_users", 1.0) < 0.009   # both tables updated by ONE launch (b2r_bucket_apply_pair)
    if merged_apply:
        kern_ms.pop("segment_adam_users")
    final_loss = float(loss.item())

    # ---- self-check of the measured route on one more step (device-side torch fp32/fp64 formulas; the oracle-based
    # version of this check is tests/test_gpu_c2_step.py): every touched row's new weight vs lazy Adam on the exact
    # gradient, untouched rows unchanged ---------------------------------------------------------------------------
    check = c2_self_check(model, feeds[3], device)

    # ---- e2e: pinned host batch -> H2D -> step -> loss D2H, every step, through model.train_step -----
    # Triple-buffered device id buffers filled by a copy stream (the DataLoader's pin_memory/prefetch role);
    # the host reads every step's loss from pinned memory, a few steps behind the enqueue front (helpers/BaseRunner.py:207
    # reads it every step too).  All copies are enqueued inside the timed region.
    NB = 3
    copy_s = torch.cuda.Stream(device=device)
    main_s = torch.cuda.current_stream(device)
    bufs = [{"user_id": torch.empty(B, dtype=torch.int64, device=device),
             "item_id": torch.empty((B, C), dtype=torch.int64, device=device), "batch_size": B, "phase": "train"}
            for _ in range(NB)]
    ready = [torch.cuda.Event() for _ in range(NB)]
    done = [torch.cuda.Event() for _ in range(NB)]
    LAG, RING = 3, 4                      # the host reads every step's loss, LAG steps behind the enqueue front
    loss_h = [torch.empty((), dtype=torch.float32).pin_memory() for _ in range(RING)]
    loss_ev = [torch.cuda.Event() for _ in range(RING)]
    keep = [None] * RING                  # keeps each step's loss tensor alive until the host has read it
    d2h_s = torch.cuda.Stream(device=device)

    def stage(k):
        j = k % NB
        u, i = pinned[k % POOL]
        with torch.cuda.stream(copy_s):
            copy_s.wait_event(done[j])
            bufs[j]["user_id"].copy_(u, non_blocking=True)
            bufs[j]["item_id"].copy_(i, non_blocking=True)
            ready[j].record(copy_s)

    def run_e2e(n_steps, k0):
        for j in range(NB):
            done[j].record(main_s)
        stage(k0)
        stage(k0 + 1)
        seen = []
        for k in range(k0, k0 + n_steps):
            stage(k + 2)
            main_s.wait_event(ready[k % NB])
            main_s.wait_event(ready[(k + 1) % NB])
            ls = model.train_step(bufs[k % NB], bufs[(k + 1) % NB])
            done[k % NB].record(main_s)
            # the 4-byte loss read-back rides on its own stream: a D2H copy enqueued on the main stream would sit
            # between this step's last kernel and the next step's first one
            keep[k % RING] = ls
            with torch.cuda.stream(d2h_s):
                d2h_s.wait_event(done[k % NB])
                loss_h[k % RING].copy_(ls, non_blocking=True)
                loss_ev[k % RING].record(d2h_s)
            if k - LAG >= k0:
                loss_ev[(k - LAG) % RING].synchronize()
                seen.append(float(loss_h[(k - LAG) % RING]))
        for k in range(max(k0, k0 + n_steps - LAG), k0 + n_steps):
            loss_ev[k % RING].synchronize()
            seen.append(float(loss_h[k % RING]))
        copy_s.synchronize()
        return seen

    ops.bprmf_step_reset()
    run_e2e(args.warmup, 0)
    dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.time()
    e0.record()
    run_e2e(args.steps, args.warmup)
    e1.record()
    dist.barrier()
    sampler.window(w0, time.time())
    ms_e2e = dist.max_ms(e0.elapsed_time(e1)) / args.steps
    e2e_value = world * B * C / (ms_e2e * 1e-3)
    ops.check_ids(device)
    ops.bprmf_step_reset()

    # ---- the reference CONTRACT route on the same batches: forward -> (runner's un-shuffle) -> loss -> backward ->
    # optimizer.step(), i.e. what the reference's unchanged BaseRunner.fit drives (BaseRunner.py:185-207) ------------
    n_c = max(3, min(args.steps, 200))
    rows_ix = torch.arange(B).unsqueeze(-1)

    def contract_step(k, runner_shuffle):
        f = dict(feeds[k % POOL])
        if runner_shuffle:                  # BaseRunner.py:187-191,196-202: CPU rand + argsort, gather, index_put back
            indices = torch.argsort(torch.rand(B, C), dim=-1)
            f["item_id"] = f["item_id"][rows_ix, indices]
        model.optimizer.zero_grad()
        out = model(f)
        if runner_shuffle:
            pred = out["prediction"]
            restored = torch.zeros(*pred.shape).to(pred.device)
            restored[rows_ix, indices] = pred
            out["prediction"] = restored
        ls = model.loss(out)
        ls.backward()
        model.optimizer.step()
        return ls

    ms_nodes, _, _ = timed_loop(dist, lambda k: contract_step(k, False), n_c, 3)
    n_s = max(3, min(n_c, 30))             # the CPU argsort of a [4096, 100] tensor costs milliseconds per step
    ms_runner, _, _ = timed_loop(dist, lambda k: contract_step(k, True), n_s, 2)
    ops.check_ids(device)
    contract = {"what": "forward -> loss -> backward -> RowSparseOptimizer.step() through the autograd nodes (the route the "
                        "reference's unchanged BaseRunner.fit drives), batches resident",
                "ms_per_step": round(ms_nodes, 5), "value": round(world * B * C / (ms_nodes * 1e-3), 1), "steps": n_c,
                "with_runner_shuffle": {"ms_per_step": round(ms_runner, 5), "value": round(world * B * C / (ms_runner * 1e-3), 1),
                                        "steps": n_s, "note": "plus BaseRunner.py:187-202: CPU rand+argsort of [B,C], "
                                        "index gather and index_put un-shuffle every step"}}

    # ---- price of exact dense-Adam RESULTS from the row-sparse kernels (--exact_adam 1): same contract route, rows are
    # advanced through the optimizer steps they skipped before every read -------------------------------------------------
    try:
        from rechorus_b200.optim import RowSparseOptimizer
        lazy_opt = model.optimizer
        model.optimizer = RowSparseOptimizer(model, "Adam", lr=1e-3, l2=0.0, exact_dense=True)
        ms_exact, _, _ = timed_loop(dist, lambda k: contract_step(k, False), max(3, min(n_c, 60)), 3)
        contract["exact_adam"] = {"ms_per_step": round(ms_exact, 5), "value": round(world * B * C / (ms_exact * 1e-3), 1),
                                  "note": "RowSparseOptimizer(exact_dense=True): dense torch.optim.Adam results (rows advanced "
                                          "through their skipped steps, b2r_adam_exact_advance) on the same contract route; "
                                          "compare with contract_route.ms_per_step (lazy / SparseAdam semantics)"}
        model.optimizer = lazy_opt
        ops.check_ids(device)
    except Exception as e:                                    # never let the extra leg take the headline down
        contract["exact_adam"] = {"error": repr(e)[:200]}

    # ---- roofline of the dominant kernel -------------------------------------------------------------
    peak, _, peak_src = measured_peaks()
    nu = statistics.mean(n_uniq[(args.warmup + k) % POOL] for k in range(args.steps))
    nuu = statistics.mean(n_uniq_u[(args.warmup + k) % POOL] for k in range(args.steps))
    n = B * C
    alg = {   # algorithmic bytes per launch (DESIGN.md section "kernels")
        "fused_score_loss_bwd": n * (4 * d + 8 + 4) + 2 * B * 4 * d + 12 * B,
        "score_fwd": n * (4 * d + 8 + 4) + B * 4 * d,
        "score_bwd_query": n * (4 * d + 8 + 4) + B * 4 * d,
        "segment_adam_items": nu * 6 * 4 * d + n * 16,
        "segment_adam_users": nuu * 6 * 4 * d + B * 4 * d + B * 12,
    }
    if merged_apply:
        alg["segment_adam_items"] += alg["segment_adam_users"]
    alg = {k_: v for k_, v in alg.items() if k_ in kern_ms}
    dom = max(alg, key=lambda k_: kern_ms[k_])
    achieved = alg[dom] / (kern_ms[dom] * 1e-3) / 1e9
    traffic = None                              # DRAM bytes per launch of that kernel from the committed ncu capture
    for name in ("r2_traffic.json", "r1_traffic.json"):
        tpath = os.path.join(ROOT, "profiles", name)
        if os.path.exists(tpath):
            with open(tpath) as f:
                traffic = json.load(f).get(dom)
            break
    cuda_names = {"segment_adam_items": "k_apply_sorted<16,2> (item + user table in one launch: segment reduce + Adam)"
                  if merged_apply else "k_apply_sorted<16,2> (item table: segment reduce + Adam)",
                  "fused_score_loss_bwd": "k_bprmf_flash<16,4,3>", "segment_adam_users": "k_apply_sorted<16,2> (user table)",
                  "score_fwd": "k_rowdot_fwd", "score_bwd_query": "k_rowdot_bwd_query"}
    roofline = {"bound": "hbm", "kernel": dom, "cuda_kernel": cuda_names.get(dom, dom), "achieved": round(achieved, 1),
                "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4), "traffic": traffic,
                "peak_source": peak_src, "alg_bytes_per_launch": int(alg[dom]), "kernel_ms": round(kern_ms[dom], 5),
                "kernel_samples": kern_n}
    kernels = {k_: {"ms": round(v, 5), "GBps": round(alg[k_] / (v * 1e-3) / 1e9, 1) if k_ in alg else None}
               for k_, v in kern_ms.items()}
    # whole step against SURVEY 8(d)'s per-sample figure (fwd+bwd rows once, no optimizer) + the Adam rows
    survey_bytes = B * (2 * (C + 1) * 4 * d + 8 * (C + 1) + 4 * C)
    step_alg = survey_bytes - (nu + nuu) * 4 * d + (nu + nuu) * 6 * 4 * d   # grad-row write replaced by w,m,v rmw
    return {
        "metric": METRIC, "value": round(value, 1), "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(ms_step, 5), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": DATA,
        "config": {"workload": "c2: " + w["desc"], "optimizer": "Adam lr=1e-3 (row-sparse/lazy, fused)",
                   "parallelism": "replicas only" if world > 1 else "single GPU",
                   "l2_policy": "inputs larger than L2: 512 MB tables + 1 GB Adam state, fresh ids every step"},
        "e2e": {"value": round(e2e_value, 1), "unit": UNIT, "h2d_bytes_per_step": 8 * B + 8 * B * C,
                "d2h_bytes_per_step": 4, "ms_per_step": round(ms_e2e, 5),
                "api": "model.train_step(feed_dict, next_feed_dict) on pinned-host batches"},
        "gpu_launches": int(launches), "host_enqueue_ms_per_step": round(host_ms_step, 5),
        "host_cost_ms_per_step_empty_queue": round(host_cost_ms, 5), "roofline": roofline, "kernels": kernels,
        "step_roofline": {"alg_bytes_per_step": int(step_alg), "achieved": round(step_alg / (ms_step * 1e-3) / 1e9, 1),
                          "frac": round(step_alg / (ms_step * 1e-3) / 1e9 / peak, 4),
                          "survey_8d_bytes_no_optimizer": int(survey_bytes)},
        "contract_route": contract, "self_check": check, "final_loss": round(final_loss, 6),
    }


DUMP_ITEM_ROWS = 32768     # seeded sample of the last step's ~340k distinct item rows (8 MB)


def dump_c2_outputs(dirname, model, feed, loss):
    """What the last timed train_step returned and wrote: its loss, the user rows it updated (every distinct user of
    the batch) and a seeded sample of the item rows it updated, in sorted id order."""
    uu = torch.unique(feed["user_id"])
    ii = torch.unique(feed["item_id"])
    pick = torch.randperm(ii.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_ITEM_ROWS].sort().values
    ii = ii[pick.to(ii.device)]
    out = {"loss": loss.reshape(1), "user_rows": model.u_embeddings.weight.detach()[uu],
           "item_rows": model.i_embeddings.weight.detach()[ii]}
    os.makedirs(dirname, exist_ok=True)
    for name, t in out.items():
        np.save(os.path.join(dirname, name + ".npy"), t.float().cpu().numpy())


def c2_self_check(model, feed, device):
    """one extra train_step verified on the device with torch formulas (fp64 gradient of the BPR objective, lazy Adam):
    a benchmark whose last step is wrong is not a benchmark"""
    from rechorus_b200 import ops
    opt = model.optimizer
    U, I = model.u_embeddings.weight.data, model.i_embeddings.weight.data
    eu, ei = opt.entry(model.u_embeddings.weight), opt.entry(model.i_embeddings.weight)
    uid, iid = feed["user_id"], feed["item_id"]
    uu, inv_u = torch.unique(uid, return_inverse=True)
    ui, inv_i = torch.unique(iid, return_inverse=True)
    w0 = {"U": U[uu].double(), "I": I[ui].double()}
    s0 = {"U": (eu["m"][uu].double(), eu["v"][uu].double()), "I": (ei["m"][ui].double(), ei["v"][ui].double())}
    probe_u = torch.randint(1, U.shape[0], (4096,), device=device)
    probe_u = probe_u[~torch.isin(probe_u, uu)]
    keep_u = U[probe_u].clone()
    ops.bprmf_step_reset()
    loss = model.train_step(feed)
    t = opt.t
    Uc, Ic = w0["U"].clone().requires_grad_(True), w0["I"].clone().requires_grad_(True)
    x = torch.einsum("bd,bcd->bc", Uc[inv_u], Ic[inv_i])
    pos, neg = x[:, :1], x[:, 1:]
    S = ((pos - neg).sigmoid() * torch.softmax(neg - neg.max(), dim=1)).sum(1)
    ref_loss = -torch.log(S.clamp(1e-8, 1 - 1e-8)).mean()
    gU, gI = torch.autograd.grad(ref_loss, [Uc, Ic])
    b1, b2 = opt.betas
    worst = 0.0
    for name, g, W, idx in (("U", gU, U, uu), ("I", gI, I, ui)):
        m, v = s0[name]
        m = b1 * m + (1 - b1) * g
        v = b2 * v + (1 - b2) * g * g
        w1 = w0[name] - (opt.lr / (1 - b1 ** t)) * m / (v.sqrt() / (1 - b2 ** t) ** 0.5 + opt.eps)
        err = (W[idx].double() - w1).abs()
        ok = g.abs() > 1e-6                              # entries where Adam's division is well-conditioned
        worst = max(worst, float(err[ok].max()))
    untouched_same = bool(torch.equal(U[probe_u], keep_u))
    loss_err = abs(float(loss) - float(ref_loss))
    ok = worst <= 1e-6 and untouched_same and loss_err <= 1e-5
    if not ok:
        raise RuntimeError(f"bench self-check failed: weight err {worst:.3e}, loss err {loss_err:.3e}, untouched {untouched_same}")
    return {"ok": True, "max_weight_err_well_conditioned": worst, "loss_err": loss_err, "untouched_rows_unchanged": untouched_same,
            "what": "one extra train_step vs fp64 torch gradient + lazy Adam on the device, all touched rows of both tables"}


# ------------------------------------------------------------------------------------------------------
# c3 / c4: NeuMF and SASRec through the plugin contract (forward -> loss -> backward -> optimizer.step)
# ------------------------------------------------------------------------------------------------------

def alg_bytes_per_sample(w):
    """SURVEY.md 8(d): fwd+bwd, fp32, int64 ids, each needed row read once, each gradient row written once, no optimizer"""
    d, C = w["d"], w["K"] + 1
    if w["model"] == "BPRMF":
        return 2 * (C + 1) * 4 * d + 8 * (C + 1) + 4 * C
    if w["model"] == "NeuMF":
        rows = 2 + 2 * C
        return 2 * rows * 4 * d + 8 * (C + 1) + 4 * C
    rows = w["L"] + C
    return 2 * rows * 4 * d + 8 * (rows + 1) + 4 * C


def train_flops_per_sample(w):
    """SURVEY.md 8(d): forward flops x 3 (forward + two backward contractions)"""
    d, C = w["d"], w["K"] + 1
    if w["model"] == "NeuMF":
        import ast
        widths = [2 * d] + list(ast.literal_eval(w["layers"]))
        mlp = sum(2 * a * b for a, b in zip(widths[:-1], widths[1:]))
        return 3 * C * (mlp + 2 * (widths[-1] + d) + d)
    if w["model"] == "SASRec":
        L = w["L"]
        block = 3 * 2 * L * d * d + 2 * (2 * L * L * d) + 2 * 2 * L * d * d
        return 3 * (w["blocks"] * block + 2 * C * d)
    return 3 * 2 * C * d


def run_model_steps(wname, args, rank, world, local_rank, sampler, steps_cap):
    from rechorus_b200 import lib as L, ops
    device = torch.device("cuda", local_rank)
    w = WORKLOADS[wname]
    B, C = w["B"], w["K"] + 1
    model, _ = build_model(w, device)
    lib = L.load()
    dist = Dist(world, device)
    host = make_batches(w, seed=2000 + rank, pool=4)
    feeds = [to_feed(f, device, B) for f in host]
    pinned = [to_feed(f, device, B, pin=True) for f in host]
    steps, warmup = min(args.steps, steps_cap), max(3, min(args.warmup, 5))

    def step(k):
        f = feeds[k % len(feeds)]
        model.optimizer.zero_grad()
        loss = model.loss(model(f))
        loss.backward()
        model.optimizer.step()
        return loss.detach()        # (a kept non-detached loss would pin this step's autograd graph: see GraphedStep)

    launches0 = lib.b2r_launch_count()
    ms_eager, loss, win = timed_loop(dist, step, steps, warmup)
    launches = (lib.b2r_launch_count() - launches0) * steps // (steps + warmup)
    sampler.window(*win)
    # the same step captured once in a CUDA graph and replayed (rechorus_b200.graph.GraphedStep): one host launch per step
    from rechorus_b200.graph import GraphedStep
    graph_error = None
    try:
        gstep = GraphedStep(model, feeds[0], warmup=2)
        ms, loss, win = timed_loop(dist, lambda k: gstep(feeds[k % len(feeds)]), steps, warmup)
        loss = loss.clone()
        sampler.window(*win)
    except Exception as e:                             # report the eagerly launched step rather than no line at all
        graph_error = repr(e)[:200]
        import traceback
        traceback.print_exc(file=sys.stderr)
        gstep, ms = None, ms_eager

    def step_e2e(k):
        if gstep is None:                              # eager fallback: H2D of the pinned batch, then the same step
            pf = pinned[k % len(pinned)]
            f = {kk: (v.to(device, non_blocking=True) if isinstance(v, torch.Tensor) else v) for kk, v in pf.items()}
            model.optimizer.zero_grad()
            ls = model.loss(model(f))
            ls.backward()
            model.optimizer.step()
            return float(ls.detach())
        ls = gstep(pinned[k % len(pinned)])            # H2D of the batch into the graph's static buffers, replay
        return float(ls)                               # the runner reads every step's loss (BaseRunner.py:207)

    ms_e2e, _, win = timed_loop(dist, step_e2e, steps, warmup)
    sampler.window(*win)
    ops.check_ids(device)
    hbm, tf, src = measured_peaks()
    value = world * B * C / (ms * 1e-3)
    bytes_s = alg_bytes_per_sample(w) * B / (ms * 1e-3) / 1e9
    flops_s = train_flops_per_sample(w) * B / (ms * 1e-3) / 1e12
    h2d = sum(v.numel() * 8 for v in host[0].values())
    out = {"value": round(value, 1), "unit": UNIT, "ms_per_step": round(ms, 5), "steps": steps, "warmup": warmup,
           "config": {"workload": wname + ": " + w["desc"], "optimizer": "Adam lr=1e-3 (tables row-sparse/lazy, dense parameters exact)",
                      "route": ("forward -> loss -> backward -> optimizer.step() through the plugin contract, captured once in a "
                                "CUDA graph and replayed per batch (GraphedStep; device-side optimizer clock)") if graph_error is None
                               else "forward -> loss -> backward -> optimizer.step() through the plugin contract, launched eagerly"},
           "eager_ms_per_step": round(ms_eager, 5), "graph_error": graph_error,
           "e2e": {"value": round(world * B * C / (ms_e2e * 1e-3), 1), "unit": UNIT, "ms_per_step": round(ms_e2e, 5),
                   "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4},
           "gpu_launches_per_step": int(launches // max(steps, 1)), "final_loss": round(float(loss), 6),
           "gpu_launches": int(launches // max(steps, 1)) * steps,
           "roofline": {"bound": "hbm", "achieved": round(bytes_s, 1), "peak": hbm, "unit": "GB/s",
                        "frac": round(bytes_s / hbm, 4), "traffic": None, "peak_source": src,
                        "alg_bytes_per_step": int(alg_bytes_per_sample(w) * B), "scope": "whole step (SURVEY 8d bytes, no optimizer)"},
           "tensor_roofline": {"bound": "tensor", "achieved": round(flops_s, 2), "peak": tf, "unit": "TFLOP/s",
                               "frac": round(flops_s / tf, 5), "flops_per_step": int(train_flops_per_sample(w) * B),
                               "note": "dense contractions of the step against the measured bf16 tensor peak"}}
    del model
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------------------
# c1: a full BaseRunner.fit epoch on an ML-1M-shaped corpus
# ------------------------------------------------------------------------------------------------------

def run_c1(args, rank, world, local_rank, sampler):
    from rechorus_b200 import ops, plugin
    from rechorus_b200.optim import RowSparseOptimizer
    from rechorus_b200.runner import BaseRunner
    import ref_arm
    device = torch.device("cuda", local_rank)
    w = WORKLOADS["c1"]
    B, C = w["B"], w["K"] + 1
    dist = Dist(world, device)
    corpus = ref_arm.synthetic_corpus(w["n_users"], w["n_items"], w["rows"], seed=11 + rank)
    model, a = build_model(w, device, extra=["--batch_size", str(B), "--num_workers", "0", "--fused_optimizer", "1",
                                             "--fused_step", "1"])
    runner = BaseRunner(a)
    data = plugin.BPRMF.Dataset(model, corpus, "train")
    # (1) the reference's data path unchanged (Python sampler, per-sample feed dicts, collate, DataLoader) feeding the
    #     one-call step: host-bound by construction
    np.random.seed(0)
    torch.manual_seed(0)
    runner.fit(data, epoch=0)                                         # warm-up epoch (contexts, allocator)
    dist.barrier()
    t0 = time.time()
    loss = runner.fit(data, epoch=1)
    torch.cuda.synchronize()
    t_fit = time.time() - t0
    sampler.window(t0, time.time())
    # (2) batch production on the device (row f3): negatives by the sampler kernel, epoch permutation and collate on
    #     the GPU, every step one C call -- same epoch, no host in the loop
    t_dev, loss_dev, n_steps = None, None, None
    if hasattr(runner, "fit_on_device"):
        runner.fit_on_device(data, epoch=0)
        dist.barrier()
        t0 = time.time()
        loss_dev = runner.fit_on_device(data, epoch=1)
        torch.cuda.synchronize()
        t_dev = time.time() - t0
        sampler.window(t0, time.time())
        n_steps = (len(data) + B - 1) // B
    ops.check_ids(device)
    rows = len(data)
    hbm, _, src = measured_peaks()
    best = min(x for x in (t_fit, t_dev) if x)
    value = world * rows * C / best
    out = {"value": round(value, 1), "unit": UNIT, "ms_per_step": round(best * 1e3 / ((rows + B - 1) // B), 5),
           "config": {"workload": "c1: " + w["desc"], "optimizer": "Adam lr=1e-3 (row-sparse/lazy, fused)",
                      "step": "one epoch of BaseRunner.fit (2,222 steps of 256 rows), num_workers=0"},
           "epoch_s": {"host_batches (reference Dataset/DataLoader plumbing + train_step)": round(t_fit, 3),
                       "device_batches (sampler + collate kernels + train_step)": round(t_dev, 4) if t_dev else None},
           "e2e": {"value": round(world * rows * C / t_fit, 1), "unit": UNIT, "ms_per_step": round(t_fit * 1e3 / ((rows + B - 1) // B), 5),
                   "h2d_bytes_per_step": 8 * B + 8 * B * C, "d2h_bytes_per_step": 4,
                   "api": "runner.fit(dataset) with the reference's host data path (per-sample feed dicts, collate, DataLoader)"},
           "final_loss": round(float(loss), 6), "final_loss_device_batches": round(float(loss_dev), 6) if loss_dev is not None else None,
           "roofline": {"bound": "hbm", "achieved": round(alg_bytes_per_sample(w) * rows / best / 1e9, 2), "peak": hbm, "unit": "GB/s",
                        "frac": round(alg_bytes_per_sample(w) * rows / best / 1e9 / hbm, 5), "traffic": None, "peak_source": src,
                        "scope": "whole epoch (SURVEY 8d: 1,568 B per sample); B=256 steps are launch-latency bound, not HBM bound"}}
    del model
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------------------
# c5: 100 M-item table, row-range shards over the ranks, score routing
# ------------------------------------------------------------------------------------------------------

def run_c5(args, rank, world, local_rank, sampler, steps_cap, group=None, solo=False):
    from rechorus_b200 import lib as L, ops
    from rechorus_b200.shard import ShardedBPRMF
    device = torch.device("cuda", local_rank)
    w = WORKLOADS["c5"]
    B, C, d = w["B"], w["K"] + 1, w["d"]
    eff_world = 1 if solo else world
    dist = Dist(eff_world, device)
    lib = L.load()
    m = ShardedBPRMF(w["n_users"], w["n_items"], d, device, optimizer="Adam", lr=1e-3, world_override=1 if solo else None)
    g = torch.Generator().manual_seed(1234 + rank)
    host = [(torch.randint(1, w["n_users"], (B,), generator=g), torch.randint(1, w["n_items"], (B, C), generator=g))
            for _ in range(4)]
    pool = [(u.to(device), i.to(device)) for u, i in host]
    pinned = [(u.pin_memory(), i.pin_memory()) for u, i in host]
    steps, warmup = min(args.steps, steps_cap), max(3, min(args.warmup, 5))
    launches0 = lib.b2r_launch_count()
    ms, loss, win = timed_loop(dist, lambda k: m.train_step(*pool[k % 4]), steps, warmup)
    launches = lib.b2r_launch_count() - launches0
    sampler.window(*win)

    def step_e2e(k):
        u, i = pinned[k % 4]
        ls = m.train_step(u.to(device, non_blocking=True), i.to(device, non_blocking=True))
        return float(ls)                                  # loss read back every step

    ms_e2e, _, win = timed_loop(dist, step_e2e, steps, warmup)
    sampler.window(*win)
    ops.check_ids(device)
    hbm, _, src = measured_peaks()
    value = eff_world * B * C / (ms * 1e-3)
    # per-GPU HBM roofline on SURVEY 8(d)'s per-sample bytes (no optimizer): every rank serves B samples' worth of rows
    per_gpu = alg_bytes_per_sample(w) * B / (ms * 1e-3) / 1e9
    out = {"value": round(value, 1), "unit": UNIT, "ms_per_step": round(ms, 5), "steps": steps, "warmup": warmup,
           "n_gpus": eff_world,
           "config": {"workload": "c5: " + w["desc"], "optimizer": "Adam lr=1e-3 (row-sparse/lazy, fused)",
                      "parallelism": f"row-range shards x{eff_world}, score routing" if eff_world > 1 else
                                     "single GPU holds the whole table (51.2 GB) + Adam state (102 GB), no collectives",
                      "exchange": m.exchange_description() if hasattr(m, "exchange_description") else "NCCL all-to-all",
                      "l2_policy": "inputs larger than L2 (6.4+ GB of table per GPU), fresh ids every step"},
           "e2e": {"value": round(eff_world * B * C / (ms_e2e * 1e-3), 1), "unit": UNIT, "ms_per_step": round(ms_e2e, 5),
                   "h2d_bytes_per_step": 8 * B + 8 * B * C, "d2h_bytes_per_step": 4},
           "gpu_launches": int(launches), "final_loss": round(float(loss), 6),
           "mem_GB": round(torch.cuda.max_memory_allocated(device) / 1e9, 1),
           "roofline": {"bound": "hbm", "achieved": round(per_gpu, 1), "peak": hbm, "unit": "GB/s", "frac": round(per_gpu / hbm, 4),
                        "traffic": None, "peak_source": src, "alg_bytes_per_step_per_gpu": int(alg_bytes_per_sample(w) * B),
                        "scope": "whole step per GPU (SURVEY 8d: 266,248 B per sample, no optimizer)"}}
    if hasattr(m, "nvlink_bytes_per_step"):
        out["nvlink_bytes_per_step_per_gpu"] = m.nvlink_bytes_per_step(B, C)
    del m, pool
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------------------
# CPU legs: the reference's own classes through its own BaseRunner.fit (tools/ref_arm.py), else the oracle port
# ------------------------------------------------------------------------------------------------------

CPU_SAMPLE = {   # bounded samples: (steps, n_items override, note)
    "c1": dict(rows=None, note="one full epoch (568,761 rows, 2,222 steps of 256)"),
    "c2": dict(steps=6, note="full-size steps (B=4096, C=100) over the full 1M x 1M tables"),
    "c3": dict(steps=4, note="full-size steps (B=4096, C=5) over four full 1M x 64 tables"),
    "c4": dict(steps=2, note="full-size steps (B=4096, C=100, L=50)"),
    "c5": dict(steps=3, n_items=2_000_000, n_users=1_000_000,
               note="steps of B=4096, C=256, d=128 with the item table cut to 2 M rows: the reference's dense gradient + "
                    "dense Adam over 100 M x 128 would need 205 GB of host memory and minutes per step (its cost grows with "
                    "the table; the cut favours the CPU)"),
}


def cpu_leg(wname, steps_override=None):
    import ref_arm
    cores = ref_arm.use_all_host_threads()
    w = dict(WORKLOADS[wname])
    s = CPU_SAMPLE[wname]
    w["n_items"] = s.get("n_items", w["n_items"])
    w["n_users"] = s.get("n_users", w["n_users"])
    B, C = w["B"], w["K"] + 1
    steps = steps_override or s.get("steps")
    rows = w["rows"] if wname == "c1" else steps * B
    src = ref_arm.reference_src()
    if src is not None:
        corpus = ref_arm.synthetic_corpus(w["n_users"], w["n_items"], rows, seed=7, with_history=w.get("L", 0))
        r = ref_arm.reference_fit(w["model"], model_flags(w), corpus, B, warm_epoch=(wname != "c1"))
        value = r["rows"] * C / r["loop_s"]
        n_st = max(1, (r["rows"] + B - 1) // B)
        return {"value": round(value, 1), "unit": UNIT, "cores": cores, "os_cpu_count": os.cpu_count(), "kind": "reference",
                "ms_per_step": round(r["loop_s"] * 1e3 / max(1, (r["rows"] + B - 1) // B), 2),
                "sample": (f"{n_st} " if wname != "c1" else "") + s["note"] + (" after one untimed warm-up epoch of the same "
                          "size" if wname != "c1" else "") + "; the UNMODIFIED reference classes (" + os.path.relpath(src, ROOT) + ") through their own "
                          "BaseRunner.fit on CPU, num_workers=0; the epoch's Python negative sampling ("
                          + f"{r['sample_s']:.1f} s) is timed separately and not counted",
                "fit_s": round(r["fit_s"], 2), "loss": round(float(r["loss"]), 6)}
    # fallback: the oracle's restatement of the same loop body
    from oracle import rechorus_oracle as O
    g = torch.Generator().manual_seed(0)
    if w["model"] == "BPRMF":
        params = O.bprmf_init(w["n_users"], w["n_items"], w["d"], g)
    elif w["model"] == "NeuMF":
        import ast
        params = O.neumf_init(w["n_users"], w["n_items"], w["d"], ast.literal_eval(w["layers"]), g)
    else:
        params = O.sasrec_init(w["n_items"], w["d"], w["L"], w["blocks"], g)
    n = (steps or 8) + 1
    batches = make_batches(w, seed=7, pool=n)
    r = ref_arm.port_steps(w["model"], params, batches)
    return {"value": round(B * C * r["steps"] / r["loop_s"], 1), "unit": UNIT, "cores": cores, "os_cpu_count": os.cpu_count(),
            "kind": "port", "ms_per_step": round(r["loop_s"] * 1e3 / r["steps"], 2),
            "sample": f"{r['steps']} " + s["note"] + "; oracle port of BaseRunner.py:184-207 (the reference tree is not on this box)"}


def run_reference_arm(args, rank):
    if rank != 0:
        return None
    wname = args.workload
    w = WORKLOADS[wname]
    want = None if wname == "c1" else max(2, min(args.steps, {"c2": 30, "c3": 30, "c4": 6, "c5": 10}[wname]))
    cb = cpu_leg(wname, steps_override=want)
    return {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": want or 2222, "warmup": 0, "ms_per_step": cb["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": DATA,
            "config": {"workload": wname + ": " + w["desc"], "optimizer": "torch.optim.Adam dense (reference)",
                       "steps_requested": args.steps, "parallelism": "CPU, rank 0 only"},
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


# ------------------------------------------------------------------------------------------------------

def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", type=str, default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", type=str, default="", choices=[""] + sorted(WORKLOADS))
    ap.add_argument("--no_cpu_baseline", action="store_true", help="skip the CPU legs (dev runs)")
    ap.add_argument("--headline_only", action="store_true", help="N=1: only the headline workload, no per-config block")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="c2: write the last timed step's loss and updated table rows to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    explicit = bool(args.workload)
    if not args.workload:
        args.workload = "c2" if max(world, args.gpus) == 1 else "c5"
    if args.dump_outputs and (args.impl != "ours" or args.workload != "c2"):
        ap.error("--dump-outputs covers the c2 workload of --impl ours")

    if args.impl == "reference":
        out = run_reference_arm(args, rank)
        if out is not None:
            print(json.dumps(out), flush=True)
        return

    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.distributed.init_process_group("nccl", device_id=device)
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.3)                      # let nvidia-smi come up before the timed regions

    wl = args.workload
    base = {"metric": METRIC, "unit": UNIT, "n_gpus": world, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": DATA}
    if wl == "c2":
        out = run_c2(args, rank, world, local_rank, sampler)
    else:
        if wl == "c1":
            r = run_c1(args, rank, world, local_rank, sampler)
        elif wl in ("c3", "c4"):
            r = run_model_steps(wl, args, rank, world, local_rank, sampler, steps_cap=args.steps)
        else:
            r = run_c5(args, rank, world, local_rank, sampler, steps_cap=args.steps)
        out = dict(base)
        out.update(r)
        out.setdefault("steps", args.steps)
        out.setdefault("warmup", args.warmup)
        out["gpu_launches"] = r.get("gpu_launches", r.get("gpu_launches_per_step", 0) * r.get("steps", 1))
        if wl == "c5" and world > 1:
            # the 1-GPU point of the same code on the same box: rank 0 alone, the other ranks wait at the barrier
            torch.distributed.barrier()
            if rank == 0:
                try:
                    a1 = run_c5(args, rank, world, local_rank, sampler, steps_cap=min(args.steps, 30), solo=True)
                    out["n1_same_code"] = {k: a1[k] for k in ("value", "ms_per_step", "steps", "mem_GB", "roofline")}
                except Exception as e:                                   # e.g. a GPU without 155 GB free
                    out["n1_same_code"] = {"unavailable": repr(e)[:200]}
            torch.distributed.barrier()
    if rank == 0 and world == 1 and wl == "c2" and not explicit and not args.headline_only:
        # compact lines of the other BASELINE configs (each the workload's own single-GPU measurement)
        out["workloads"] = {}
        for name, fn in (("c1", lambda: run_c1(args, rank, world, local_rank, sampler)),
                         ("c3", lambda: run_model_steps("c3", args, rank, world, local_rank, sampler, steps_cap=60)),
                         ("c4", lambda: run_model_steps("c4", args, rank, world, local_rank, sampler, steps_cap=20)),
                         ("c5", lambda: run_c5(args, rank, world, local_rank, sampler, steps_cap=30))):
            try:
                out["workloads"][name] = fn()
            except Exception as e:
                out["workloads"][name] = {"error": repr(e)[:300]}
            torch.cuda.empty_cache()
    # if the timed regions were too short for nvidia-smi to sample, keep the GPU busy ~0.5 s more (untimed) so the clock
    # record reflects a loaded GPU; flagged in the output
    probe = False
    if sampler.n_in_windows() < 3:
        probe = True
        x = torch.empty(256 << 20, dtype=torch.float32, device=device)
        w0 = time.time()
        while time.time() - w0 < 0.5:
            x.add_(1.0)
            torch.cuda.synchronize()
        sampler.window(w0, time.time())
        del x
    clocks = sampler.stop()
    clocks["includes_untimed_continuation"] = probe
    out["clocks"] = clocks
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_leg(wl)
            for name, r in out.get("workloads", {}).items():
                if "error" not in r:
                    try:
                        r["cpu_baseline"] = cpu_leg(name)
                    except Exception as e:
                        r["cpu_baseline"] = {"error": repr(e)[:300]}
        print(json.dumps(out), flush=True)
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
