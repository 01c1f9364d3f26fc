"""Generate tests/golden/overlay_reference.npz: the UNMODIFIED reference's own CPU runs that tests/test_gpu_overlay.py
compares the overlay against (REFERENCE_RUNS there), each through tools/run_reference.py on that test's dataset.
BPRMF checkpoints are stored whole (their tests bound every entry); the NeuMF / SASRec tensors over SAMPLE_OVER entries
keep a seeded sample of SAMPLE entries and their flat positions (their test bounds the median and the tail), which
keeps the file near 150 KB.

    python tests/golden/make_overlay_golden.py

Needs the reference where tools/run_reference.py finds it (RECHORUS_SRC, else oracle/_ref/src placed by build())."""
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from tests import test_gpu_overlay as T  # noqa: E402

SAMPLE_OVER, SAMPLE = 2048, 1024


def main():
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        T._dataset(tmp)
        for tag, (model, flags) in T.REFERENCE_RUNS.items():
            losses, metrics, weights, _ = T._run(tmp, tag, T.REFERENCE, model, flags, "")
            out[tag + ":losses"] = np.array(losses)
            out.update({f"{tag}:m:{k}": np.array(v) for k, v in metrics.items()})
            for k, v in weights.items():
                v = v.numpy()
                out[f"{tag}:shape:{k}"] = np.array(v.shape)
                if model != "BPRMF" and v.size > SAMPLE_OVER:
                    pick = np.sort(np.random.RandomState(0).choice(v.size, SAMPLE, replace=False))
                    out[f"{tag}:pick:{k}"], v = pick.astype(np.int32), v.reshape(-1)[pick]
                out[f"{tag}:w:{k}"] = v
    np.savez_compressed(T.GOLDEN, **out)
    print(T.GOLDEN, len(out), "arrays")


if __name__ == "__main__":
    main()
