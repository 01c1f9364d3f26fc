"""The drop-in boundary, end to end on a B200: the reference's UNCHANGED ``src/main.py`` (the ReChorus checkout
``rechorus_b200.overlay.DEFAULT_REF`` names) drives the kernel-backed BPRMF / NeuMF / SASRec through
``rechorus_b200.overlay``, and is compared with the unmodified reference's own CPU run of the same command line
(tools/run_reference.py: NumPy alias shim + runpy, nothing else), stored in tests/golden/overlay_reference.npz by
tests/golden/make_overlay_golden.py.  Same csv files, same seeds, ``--num_workers 0``: the reader, negative sampling,
DataLoader order and candidate permutations are the reference's own code in both runs, so the two trainings see
identical batches and differ only in who does the arithmetic.

Compared: per-epoch losses (the reference's log lines), the dev/test metric lines, and the saved checkpoints
(``model.save_model`` files interchange, SURVEY.md A.5).  Skipped where build() found no checkout to place in
oracle/_ref."""
import os
import re
import subprocess
import sys

import numpy as np
import pandas as pd
import pytest
import torch

from rechorus_b200.overlay import DEFAULT_REF as REF

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(not os.path.isfile(os.path.join(REF, "main.py")),
                                 reason="no ReChorus sources: build() found no checkout to place in oracle/_ref")]

N_USERS, N_ITEMS, ROWS, N_EVAL, N_NEG = 60, 90, 1500, 120, 29


def _dataset(root):
    rng = np.random.RandomState(7)
    d = os.path.join(root, "data", "tiny")
    os.makedirs(d)
    df = pd.DataFrame({"user_id": rng.randint(1, N_USERS, ROWS), "item_id": rng.randint(1, N_ITEMS, ROWS),
                       "time": np.arange(ROWS)})
    tr = df.iloc[:ROWS - 2 * N_EVAL]
    tr.to_csv(os.path.join(d, "train.csv"), sep="\t", index=False)
    seen = set(tr.user_id)
    for name, part in (("dev", df.iloc[ROWS - 2 * N_EVAL:ROWS - N_EVAL]), ("test", df.iloc[ROWS - N_EVAL:])):
        part = part[part.user_id.isin(seen)].copy()
        part["neg_items"] = [str(list(rng.randint(1, N_ITEMS, N_NEG))) for _ in range(len(part))]
        part.to_csv(os.path.join(d, name + ".csv"), sep="\t", index=False)
    return os.path.join(root, "data") + "/"


def _run(tmp, tag, launcher, model, extra, gpu):
    cwd = os.path.join(tmp, tag, "src")           # main.py writes ../log and ../model relative to the cwd
    os.makedirs(cwd)
    mp, lf = os.path.join(tmp, tag, "model.pt"), os.path.join(tmp, tag, "log.txt")
    cmd = [sys.executable, *launcher, "--ref", REF, "--model_name", model, "--dataset", "tiny", "--path",
           os.path.join(tmp, "data") + "/", "--gpu", gpu, "--num_workers", "0", "--epoch", "2", "--early_stop", "0",
           "--batch_size", "128", "--eval_batch_size", "64", "--emb_size", "64", "--lr", "0.01", "--l2", "0",
           "--topk", "5,10", "--metric", "NDCG,HR", "--model_path", mp, "--log_file", lf, "--regenerate", "1",
           "--save_final_results", "0", *extra]
    env = dict(os.environ, PYTHONPATH=ROOT)
    res = subprocess.run(cmd, cwd=cwd, env=env, capture_output=True, text=True, timeout=900)
    out = res.stdout + res.stderr
    assert res.returncode == 0, out[-3000:]
    losses = [float(x) for x in re.findall(r"Epoch \d+\s+loss=([0-9.]+)", out)]
    test_line = re.findall(r"Test After Training: \(([^)]*)\)", out)
    metrics = dict((kv.split(":")[0], float(kv.split(":")[1])) for kv in test_line[-1].split(",")) if test_line else {}
    return losses, metrics, torch.load(mp, map_location="cpu"), out


OVERLAY = ["-m", "rechorus_b200.overlay"]
REFERENCE = [os.path.join(ROOT, "tools", "run_reference.py")]
SGD_FLAGS = ["--num_neg", "7", "--optimizer", "SGD", "--lr", "0.5"]
DEEP = [("NeuMF", ["--num_neg", "2", "--layers", "[32, 16]"]),
        ("SASRec", ["--num_neg", "2", "--num_layers", "2", "--num_heads", "2", "--history_max", "8"])]
# the reference side of every comparison: tag -> (model, flags) of the reference's CPU run stored in GOLDEN
REFERENCE_RUNS = {"bprmf_ref": ("BPRMF", ["--num_neg", "3"]), "sgd_ref": ("BPRMF", SGD_FLAGS),
                  **{m + "_ref": (m, f) for m, f in DEEP}}
GOLDEN = os.path.join(ROOT, "tests", "golden", "overlay_reference.npz")


def _reference(tag):
    """losses, test metrics, final checkpoint and its tensor shapes of the reference's own run REFERENCE_RUNS[tag].
    Checkpoint tensors stored as a sample hold the entries at the flat positions picks[name]."""
    z = np.load(GOLDEN)

    def group(prefix):
        return {k[len(prefix):]: z[k] for k in z.files if k.startswith(prefix)}
    metrics = {k: float(v) for k, v in group(tag + ":m:").items()}
    weights = {k: torch.from_numpy(v) for k, v in group(tag + ":w:").items()}
    shapes = {k: tuple(int(n) for n in v) for k, v in group(tag + ":shape:").items()}
    picks = {k: torch.from_numpy(v).long() for k, v in group(tag + ":pick:").items()}
    return [float(x) for x in z[tag + ":losses"]], metrics, weights, shapes, picks


@pytest.fixture(scope="module")
def workdir(tmp_path_factory):
    tmp = str(tmp_path_factory.mktemp("overlay"))
    _dataset(tmp)
    return tmp


def test_bprmf_dense_adam_through_unchanged_main_equals_reference_cpu_run(workdir):
    """exact reference semantics: dense gradients into the torch.optim.Adam the reference's runner builds"""
    l_ref, m_ref, w_ref, _, _ = _reference("bprmf_ref")
    l_gpu, m_gpu, w_gpu, out = _run(workdir, "bprmf_gpu", OVERLAY, "BPRMF", ["--num_neg", "3", "--table_mode", "dense"], "0")
    assert "Device: cuda" in out
    assert len(l_ref) == 2 and np.allclose(l_gpu, l_ref, rtol=0, atol=1e-4), (l_gpu, l_ref)      # logged with 4 decimals
    assert set(w_gpu) == set(w_ref)
    for k in w_ref:
        assert (w_gpu[k] - w_ref[k]).abs().max() <= 5e-5, k
    for k in m_ref:
        assert abs(m_gpu[k] - m_ref[k]) <= 2.0 / N_EVAL + 1e-4, (k, m_gpu[k], m_ref[k])


def test_bprmf_fused_whole_step_route_through_unchanged_main_equals_reference_sgd(workdir):
    """the benchmarked route -- model.train_step, one C call per batch, row-sparse optimizer -- reached from the
    unchanged main.py via helpers.B200Runner.  Under SGD without weight decay a row-sparse update IS the dense update,
    so the reference's CPU run is the exact expectation."""
    l_ref, m_ref, w_ref, _, _ = _reference("sgd_ref")
    l_gpu, m_gpu, w_gpu, out = _run(workdir, "sgd_gpu", OVERLAY, "BPRMF",
                                    SGD_FLAGS + ["--table_mode", "fused", "--fused_step", "1", "--device_metrics", "1"], "0")
    assert np.allclose(l_gpu, l_ref, rtol=0, atol=1e-4), (l_gpu, l_ref)
    for k in w_ref:
        assert (w_gpu[k] - w_ref[k]).abs().max() <= 1e-5, k
    for k in m_ref:
        assert abs(m_gpu[k] - m_ref[k]) <= 2.0 / N_EVAL + 1e-4, (k, m_gpu[k], m_ref[k])


@pytest.mark.parametrize("model,flags", DEEP)
def test_deep_models_through_unchanged_main_track_reference_cpu_run(workdir, model, flags):
    l_ref, m_ref, w_ref, shapes, picks = _reference(model + "_ref")
    l_gpu, m_gpu, w_gpu, _ = _run(workdir, model + "_gpu", OVERLAY, model, flags + ["--table_mode", "dense"], "0")
    assert np.allclose(l_gpu, l_ref, rtol=0, atol=2e-4), (l_gpu, l_ref)
    assert set(w_gpu) == set(shapes) and all(tuple(w_gpu[k].shape) == shapes[k] for k in shapes)
    w_gpu = {k: (v.reshape(-1)[picks[k]] if k in picks else v) for k, v in w_gpu.items()}
    # Adam amplifies rounding-level gradient entries to lr-sized steps (see test_gpu_zz_fit_golden.py): the bulk of the
    # parameters agrees closely, the tail is bounded by the step budget lr * steps
    dev = torch.cat([(w_gpu[k] - w_ref[k]).abs().reshape(-1) for k in w_ref])          # (sampled entries: see GOLDEN)
    # NeuMF starts on a flat loss surface (loss stays at ln 2): nearly every gradient entry is rounding-level, and the
    # reference's own fp32 run sits ~1e-2 (90th percentile) from its fp64 run (tests/golden/fit_neumf.npz "w1_64:")
    med_tol = 2e-4 if model == "SASRec" else 5e-3
    assert float(dev.median()) <= med_tol and float(dev.max()) <= 0.01 * 2 * 12, (float(dev.median()), float(dev.max()))
    for k in m_ref:
        assert abs(m_gpu[k] - m_ref[k]) <= 0.1, (k, m_gpu[k], m_ref[k])


def test_out_of_range_id_raises_like_the_reference():
    """ATen raises IndexError inside the reference's forward (BPRMF.py:39-40).  The reference's own reader cannot hand such
    an id to the model (BaseReader.py:55-59 sizes the tables from the data and asserts the negatives), so the check is
    made on the class the overlay builds: the kernels clamp + count, and the model raises the same exception type at the
    next phase switch every runner performs (model.eval() / model.train(), BaseRunner.py:179,231)."""
    import argparse
    import types
    from rechorus_b200 import overlay
    classes = overlay.install(REF)
    cls = classes["BPRMF"]
    p = argparse.ArgumentParser()
    p = cls.parse_model_args(p)
    a = p.parse_args(["--emb_size", "64"])
    a.device, a.model_path = torch.device("cuda", 0), "/tmp/_b2r_oob.pt"
    model = cls(a, types.SimpleNamespace(n_users=20, n_items=30)).to(a.device)
    model.apply(model.init_weights)
    model.train()
    feed = {"user_id": torch.tensor([1, 2]).cuda(), "item_id": torch.tensor([[3, 4], [5, 99]]).cuda(), "batch_size": 2,
            "phase": "train"}
    out = model(feed)                                    # the kernel does not read out of bounds ...
    assert torch.isfinite(out["prediction"]).all()
    with pytest.raises(IndexError):                      # ... and the bad id surfaces as the reference's exception type
        model.eval()
    model.eval()                                         # counter was reset by the raise
