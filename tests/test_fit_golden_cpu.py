"""CPU: this repository's host side (plugin Dataset classes, negative sampling, collate, BaseRunner.fit with its
DataLoader / candidate shuffle / optimizer construction, BaseRunner.evaluate) reproduces two epochs of the REFERENCE's
own runner on the same corpus and seeds (tests/golden/fit_*.npz, made by tests/golden/make_fit_golden.py).  The model
arithmetic is the oracle's here (the kernels need a GPU; tests/test_gpu_zz_fit_golden.py repeats this with them), so
what is pinned is SURVEY.md §8 rows a1, a2, a3, a11, a12: same batches, same permutations, same parameter groups,
same optimizer steps, same metrics."""
import argparse
import os
import sys

import numpy as np
import pytest
import torch

from oracle import rechorus_oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
sys.path.insert(0, GOLDEN)
import fit_corpus  # noqa: E402


def _oracle_model_class(name):
    from rechorus_b200 import plugin
    base = getattr(plugin, name)

    class OracleArithmetic(base):
        """the stand-alone plugin class (parameters, state_dict keys, Dataset, flags) with the oracle's CPU forward"""

        def forward(self, feed_dict):
            p = dict(self.named_parameters())
            return {"prediction": O.scores(name, p, feed_dict, getattr(self, "num_heads", 4))}

        def loss(self, out_dict):
            return O.bpr_loss(out_dict["prediction"])

    OracleArithmetic.__name__ = name
    return OracleArithmetic


def run_case(case, model_cls, device, extra=()):
    """shared with the GPU test: build corpus/model/runner from the fixture's flags, train EPOCHS epochs, evaluate"""
    from rechorus_b200.runner import BaseRunner
    cls_name, flags = fit_corpus.CASES[case]
    p = argparse.ArgumentParser()
    p = BaseRunner.parse_runner_args(p)
    p = model_cls.parse_model_args(p)
    a = p.parse_args(flags + fit_corpus.COMMON + list(extra))
    a.device, a.model_path, a.log_file = device, "/tmp/_b2r_fit_golden.pt", ""
    corpus = fit_corpus.build()
    gold = np.load(os.path.join(GOLDEN, case + ".npz"))
    model = model_cls(a, corpus)
    model.load_state_dict({k[3:]: torch.from_numpy(gold[k]) for k in gold.files if k.startswith("w0:")})
    model = model.to(device)
    data = {ph: model_cls.Dataset(model, corpus, ph) for ph in ("train", "dev")}
    for d in data.values():
        d.prepare()
    runner = BaseRunner(a)
    np.random.seed(42)
    torch.manual_seed(42)
    losses = [runner.fit(data["train"], epoch=e + 1) for e in range(fit_corpus.EPOCHS)]
    metrics = runner.evaluate(data["dev"], [5, 10], ["NDCG", "HR"])
    final = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    return gold, losses, metrics, final


@pytest.mark.parametrize("case", sorted(fit_corpus.CASES))
def test_host_side_reproduces_reference_runner(case):
    cls = _oracle_model_class(fit_corpus.CASES[case][0])
    # one intra-op thread: CPU reductions are split by thread count, and Adam turns the rounding of softmax-invariant
    # entries (SASRec's key biases) into visible steps, so the result would otherwise depend on the host's core count
    threads = torch.get_num_threads()
    torch.set_num_threads(1)
    try:
        gold, losses, metrics, final = run_case(case, cls, torch.device("cpu"))
    finally:
        torch.set_num_threads(threads)
    assert np.allclose(losses, gold["losses"], rtol=0, atol=2e-6), (losses, gold["losses"])
    worst = max(float((final[k[3:]] - torch.from_numpy(gold[k])).abs().max()) for k in gold.files if k.startswith("w1:"))
    assert worst <= 2e-5, worst
    for k in gold.files:
        if k.startswith("m:"):
            assert abs(metrics[k[2:]] - float(gold[k])) <= 1e-12, (k, metrics[k[2:]], float(gold[k]))
