"""CPU, where build() placed the unmodified reference in oracle/_ref (rechorus_b200.overlay.DEFAULT_REF): the overlay
drives the reference's unchanged main.py up to the first forward, where the kernel-backed class refuses to run without CUDA (no CPU fallback)."""
import os
import subprocess
import sys

import numpy as np
import pandas as pd
import pytest

from rechorus_b200.overlay import DEFAULT_REF as REF

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

pytestmark = pytest.mark.skipif(not os.path.isfile(os.path.join(REF, "main.py")),
                                reason="no ReChorus sources: build() found no checkout to place in oracle/_ref")


def _tiny_dataset(root):
    rng = np.random.RandomState(0)
    d = os.path.join(root, "data", "tiny")
    os.makedirs(d)
    rows = [(u, rng.randint(1, 30), t) for t, u in enumerate(rng.randint(1, 12, 300))]
    df = pd.DataFrame(rows, columns=["user_id", "item_id", "time"])
    df.iloc[:240].to_csv(os.path.join(d, "train.csv"), sep="\t", index=False)
    for name, part in (("dev", df.iloc[240:270]), ("test", df.iloc[270:])):
        part = part.copy()
        part["neg_items"] = [str(list(rng.randint(1, 30, 9))) for _ in range(len(part))]
        part.to_csv(os.path.join(d, name + ".csv"), sep="\t", index=False)
    return os.path.join(root, "data") + "/"


@pytest.mark.parametrize("model", ["BPRMF", "SASRec"])
def test_reference_main_runs_our_class_and_refuses_cpu(tmp_path, model):
    path = _tiny_dataset(str(tmp_path))
    src = tmp_path / "src"          # main.py writes ../log and ../model relative to the cwd
    src.mkdir()
    cmd = [sys.executable, "-m", "rechorus_b200.overlay", "--ref", REF, "--model_name", model, "--dataset", "tiny", "--path", path,
           "--gpu", "", "--num_workers", "0", "--epoch", "1", "--emb_size", "64", "--history_max", "5"]
    env = dict(os.environ, PYTHONPATH=ROOT)
    res = subprocess.run(cmd, cwd=str(src), env=env, capture_output=True, text=True, timeout=300)
    out = res.stdout + res.stderr
    assert res.returncode != 0
    assert "rechorus_b200 runs on a CUDA device only" in out, out[-2000:]
    assert "u_embeddings" in out or "i_embeddings" in out            # main.py logged OUR module (logging.info(model))
