"""CPU reference legs of bench.py: the reference's OWN classes driven by its OWN ``BaseRunner.fit`` on a bounded synthetic
corpus (kind "reference"), or -- where the unmodified reference is not on the box -- the oracle port (kind "port").

The reference tree is the ``src/`` directory the RECHORUS_SRC environment variable names, else the unmodified copy
build() places in oracle/_ref/src.  Nothing of rechorus_b200 is imported here: this is the arm the product
is compared against.  ``oracle/`` is touched only by the "port" fallback (bench.py's cpu_baseline contract)."""
from __future__ import annotations

import argparse
import os
import sys
import time
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def reference_src():
    p = os.environ.get("RECHORUS_SRC") or os.path.join(ROOT, "oracle", "_ref", "src")
    return p if os.path.isfile(os.path.join(p, "main.py")) else None


def use_all_host_threads() -> int:
    """torchrun exports OMP_NUM_THREADS=1 to every rank; the CPU legs use the box's physical cores (torch's default:
    half of os.cpu_count() on an SMT host) and only rank 0 runs them."""
    want = max(1, (os.cpu_count() or 2) // 2)
    if torch.get_num_threads() < want:
        torch.set_num_threads(want)
    return torch.get_num_threads()


class _Clicked(dict):
    """train_clicked_set of a synthetic corpus: users without recorded clicks have none"""

    def __missing__(self, key):
        return set()


def synthetic_corpus(n_users, n_items, rows, seed, with_history=0):
    """The attributes helpers/BaseReader.py:32-60 (and SeqReader.py:21-36 when with_history > 0) produce, for `rows`
    seeded uniform interactions.  History: every row gets a random prefix length in [1, with_history]."""
    import pandas as pd
    rng = np.random.RandomState(seed)
    df = pd.DataFrame({"user_id": rng.randint(1, n_users, rows), "item_id": rng.randint(1, n_items, rows),
                       "time": np.arange(rows)})
    corpus = types.SimpleNamespace(n_users=n_users, n_items=n_items, train_clicked_set=_Clicked(),
                                   residual_clicked_set=_Clicked())
    if with_history:
        # one long synthetic history per row's user: row r reads user_his[u][:position]
        L = with_history
        user_his, position = {}, np.zeros(rows, dtype=np.int64)
        uids = df.user_id.values
        for r in range(rows):
            u = int(uids[r])
            if u not in user_his:
                user_his[u] = [(int(x), t) for t, x in enumerate(rng.randint(1, n_items, L))]
            position[r] = rng.randint(1, L + 1)
        position[0] = L                                  # one full-length row so the batch max length is L
        df["position"] = position
        corpus.user_his = user_his
    corpus.data_df = {"train": df}
    return corpus


def _ref_modules(src):
    for alias, typ in (("object", object), ("int", int), ("float", float)):
        if not hasattr(np, alias):
            setattr(np, alias, typ)                      # NumPy >= 1.24 removed them; the reference still spells them
    if src not in sys.path:
        sys.path.insert(0, src)
    import helpers.BaseRunner as RR
    import models.general.BPRMF as MB
    import models.general.NeuMF as MN
    import models.sequential.SASRec as MS
    return RR.BaseRunner, {"BPRMF": MB.BPRMF, "NeuMF": MN.NeuMF, "SASRec": MS.SASRec}


def reference_fit(model_name, model_flags, corpus, batch_size, lr=1e-3, l2=0.0, warm_epoch=True):
    """One ``BaseRunner.fit`` epoch of the unmodified reference on CPU (num_workers 0).  Returns seconds spent in the
    training loop proper (fit minus its own negative-sampling pass, timed separately so the step metric compares with
    a GPU step that is fed pre-drawn negatives), the sampling seconds, rows, and the epoch loss."""
    src = reference_src()
    if src is None:
        return None
    Runner, classes = _ref_modules(src)
    cls = classes[model_name]
    p = argparse.ArgumentParser()
    p = Runner.parse_runner_args(p)
    p = cls.parse_model_args(p)
    a = p.parse_args(list(model_flags) + ["--batch_size", str(batch_size), "--num_workers", "0", "--lr", str(lr),
                                          "--l2", str(l2), "--optimizer", "Adam"])
    a.device, a.model_path, a.log_file, a.train = torch.device("cpu"), "/tmp/_b2r_ref_arm.pt", "/tmp/_b2r_ref_arm.log", 1
    torch.manual_seed(0)
    np.random.seed(0)
    model = cls(a, corpus)
    model.apply(model.init_weights)
    data = cls.Dataset(model, corpus, "train")
    runner = Runner(a)
    t0 = time.perf_counter()
    data.actions_before_epoch()                          # the reference's own sampler (BaseModel.py:206-214), timed alone
    t_sample = time.perf_counter() - t0
    t_warm = None
    if warm_epoch:
        # untimed first epoch: first-touch page faults of the dense gradient / Adam state (gigabytes at 1 M rows) and
        # thread-pool start-up would otherwise be billed to a sample of a handful of steps
        t0 = time.perf_counter()
        runner.fit(data, epoch=0)
        t_warm = time.perf_counter() - t0
    t0 = time.perf_counter()
    loss = runner.fit(data, epoch=1)                     # samples again, then the loop of BaseRunner.py:184-207
    t_fit = time.perf_counter() - t0
    return {"loop_s": max(t_fit - t_sample, 1e-9), "fit_s": t_fit, "sample_s": t_sample, "rows": len(data), "loss": loss,
            "warm_epoch_s": t_warm}


def port_steps(model_name, params, batches, lr=1e-3, l2=0.0, warmup=1):
    """fallback when the reference tree is absent: the oracle's restatement of the same loop body"""
    from oracle import rechorus_oracle as O
    tr = O.ReferenceStyleTrainer(model_name, params, lr=lr, l2=l2, optimizer="Adam")
    for b in batches[:warmup]:
        tr.step(b)
    t0 = time.perf_counter()
    loss = None
    for b in batches[warmup:]:
        loss = tr.step(b)
    return {"loop_s": time.perf_counter() - t0, "steps": len(batches) - warmup, "loss": loss}
