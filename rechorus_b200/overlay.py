"""Run the reference's UNCHANGED ``src/main.py`` with the kernel-backed model classes substituted.

    python -m rechorus_b200.overlay --ref <ReChorus>/src --model_name BPRMF --emb_size 64 --lr 1e-3 \
        --l2 1e-6 --dataset Grocery_and_Gourmet_Food --path /tmp/data/ [--table_mode fused]

What it does (SURVEY.md section 8b1): puts the reference ``src/`` on ``sys.path``, restores the NumPy aliases the
reference still uses (np.object / np.int / np.float), imports the reference's model modules, builds classes
that graft this package's kernel mixins onto the reference's own ``GeneralModel`` / ``SequentialModel`` (so the
reference's Dataset, reader, runner, argument plumbing and checkpoint code are the ones that run), replaces
``models.general.BPRMF.BPRMF`` etc. with them, and ``runpy``s ``main.py``.  With ``--fused_step 1`` or
``--device_metrics 1`` on the command line it also registers ``helpers.B200Runner`` (a subclass of the reference's own
BaseRunner) through the same by-name discovery.  Needs a CUDA device for the first forward call; there is no CPU
fallback.  ``--ref`` (a ReChorus ``src/`` directory) defaults to the ``RECHORUS_SRC`` environment variable, else to the
unmodified copy build() places in oracle/_ref/src.
"""
from __future__ import annotations

import os
import runpy
import sys

DEFAULT_REF = os.environ.get("RECHORUS_SRC") or os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                                                           "oracle", "_ref", "src")


def _make_runner_module(ref_runner_cls):
    """``helpers.B200Runner``: the reference's own BaseRunner (train / evaluate / predict / print_res / logging
    untouched) with two seams re-pointed at the kernels, selected by flags the unchanged ``main.py`` parses for us
    (``main.py:164-176`` resolves the runner by the model's ``runner`` attribute and lets it add arguments):
      --fused_step 1      fit() = one C call per batch (model.train_step: forward, loss, backward, row-sparse optimizer;
                          next batch's index plan prefetched) instead of the loop body of BaseRunner.py:185-207;
      --device_metrics 1  evaluate() ranks on the GPU (model.eval_ranks) instead of shipping predictions to the host.
    Without those flags every method is the reference's."""
    import types

    from . import runner as ours
    from .optim import RowSparseOptimizer

    class B200Runner(ref_runner_cls):
        @staticmethod
        def parse_runner_args(parser):
            parser = ref_runner_cls.parse_runner_args(parser)
            parser.add_argument("--fused_step", type=int, default=0,
                                help="1 (with --table_mode fused): one C call per training step (model.train_step)")
            parser.add_argument("--device_metrics", type=int, default=0,
                                help="1: rank the ground truth on the GPU (model.eval_ranks)")
            return parser

        def __init__(self, args):
            super().__init__(args)
            self.fused_step = getattr(args, "fused_step", 0)
            self.device_metrics = getattr(args, "device_metrics", 0)

        def fit(self, dataset, epoch=-1):
            model = dataset.model
            if (self.fused_step and hasattr(model, "train_step")
                    and isinstance(model.optimizer, RowSparseOptimizer)):       # the lazily-built fused optimizer
                dataset.actions_before_epoch()                                  # BaseRunner.py:178: negatives
                model.train()
                return ours.BaseRunner._fit_whole_steps(self, dataset, epoch)
            return super().fit(dataset, epoch)

        def evaluate(self, dataset, topks, metrics):
            if self.device_metrics and hasattr(dataset.model, "eval_ranks"):
                return ours.BaseRunner.evaluate_on_device(self, dataset, topks, metrics)
            return super().evaluate(dataset, topks, metrics)

    mod = types.ModuleType("helpers.B200Runner")
    mod.B200Runner = B200Runner
    return mod


def install(ref_src: str = DEFAULT_REF, b200_runner: bool = False):
    import numpy as np
    for alias, typ in (("object", object), ("int", int), ("float", float)):
        if not hasattr(np, alias):
            setattr(np, alias, typ)          # removed in NumPy >= 1.24; BaseModel.py:141, SASRec.py:69, utils.py:65
    if ref_src not in sys.path:
        sys.path.insert(0, ref_src)
    import models.BaseModel as RB                       # the reference's own base classes
    import models.general.BPRMF as ref_bprmf
    import models.general.NeuMF as ref_neumf
    import models.sequential.SASRec as ref_sasrec
    from . import plugin

    class BPRMF(plugin.BPRMFKernels, RB.GeneralModel):
        reader, runner = "BaseReader", "BaseRunner"
        extra_log_args = ["emb_size", "batch_size"]

        @staticmethod
        def parse_model_args(parser):
            parser = plugin.BPRMFKernels.parse_model_args(parser)
            return RB.GeneralModel.parse_model_args(parser)

        def __init__(self, args, corpus):
            RB.GeneralModel.__init__(self, args, corpus)
            self._base_init(args, corpus)

    class NeuMF(plugin.NeuMFKernels, RB.GeneralModel):
        reader, runner = "BaseReader", "BaseRunner"
        extra_log_args = ["emb_size", "layers"]

        @staticmethod
        def parse_model_args(parser):
            parser = plugin.NeuMFKernels.parse_model_args(parser)
            return RB.GeneralModel.parse_model_args(parser)

        def __init__(self, args, corpus):
            RB.GeneralModel.__init__(self, args, corpus)
            self._neumf_init(args, corpus)

    class SASRec(plugin.SASRecKernels, RB.SequentialModel):
        reader, runner = "SeqReader", "BaseRunner"
        extra_log_args = ["emb_size", "num_layers", "num_heads"]

        @staticmethod
        def parse_model_args(parser):
            parser = plugin.SASRecKernels.parse_model_args(parser)
            return RB.SequentialModel.parse_model_args(parser)

        def __init__(self, args, corpus):
            RB.SequentialModel.__init__(self, args, corpus)
            self._base_init(args, corpus)

    ref_bprmf.BPRMF, ref_neumf.NeuMF, ref_sasrec.SASRec = BPRMF, NeuMF, SASRec
    # --model_mode Impression (main.py:164: '{0}.{0}{1}'): the reference's own ImpressionModel / ImpressionSeqModel hosts
    # (flags, reader, runner, Dataset) with the forward on the kernels and the list-wise loss as one kernel family
    import models.BaseImpressionModel as RI

    class _ImpLoss:
        def loss(self, out_dict, target=None):
            from . import ops
            return ops.listwise_loss(out_dict["prediction"], target, self.loss_n, self.train_max_pos_item)

    class BPRMFImpression(_ImpLoss, plugin.BPRMFKernels, RI.ImpressionModel):
        reader, runner = "ImpressionReader", "ImpressionRunner"
        extra_log_args = ["emb_size", "batch_size"]

        @staticmethod
        def parse_model_args(parser):
            parser = plugin.BPRMFKernels.parse_model_args(parser)
            return RI.ImpressionModel.parse_model_args(parser)

        def __init__(self, args, corpus):
            RI.ImpressionModel.__init__(self, args, corpus)
            self.__dict__["_b2r_vectors"] = True
            self._base_init(args, corpus)

    class SASRecImpression(_ImpLoss, plugin.SASRecKernels, RI.ImpressionSeqModel):
        reader, runner = "ImpressionSeqReader", "ImpressionRunner"
        extra_log_args = ["emb_size", "num_layers", "num_heads"]

        @staticmethod
        def parse_model_args(parser):
            parser = plugin.SASRecKernels.parse_model_args(parser)
            return RI.ImpressionSeqModel.parse_model_args(parser)

        def __init__(self, args, corpus):
            RI.ImpressionSeqModel.__init__(self, args, corpus)
            self.__dict__["_b2r_vectors"] = True
            self._base_init(args, corpus)

    ref_bprmf.BPRMFImpression, ref_sasrec.SASRecImpression = BPRMFImpression, SASRecImpression
    if b200_runner:
        # main.py:10 `from helpers import *` imports what helpers.__all__ names; add the runner module there and let
        # the model classes choose it (main.py:166: eval('{0}.{0}'.format(model_name.runner)))
        import helpers
        import helpers.BaseRunner as ref_runner
        mod = _make_runner_module(ref_runner.BaseRunner)
        sys.modules["helpers.B200Runner"] = mod
        helpers.B200Runner = mod
        if "B200Runner" not in helpers.__all__:
            helpers.__all__.append("B200Runner")
        for cls in (BPRMF, NeuMF, SASRec):
            cls.runner = "B200Runner"
    return {"BPRMF": BPRMF, "NeuMF": NeuMF, "SASRec": SASRec, "BPRMFImpression": BPRMFImpression,
            "SASRecImpression": SASRecImpression}


def main(argv=None):
    argv = list(sys.argv[1:] if argv is None else argv)
    ref = DEFAULT_REF
    if "--ref" in argv:
        i = argv.index("--ref")
        ref = argv[i + 1]
        del argv[i:i + 2]
    if not os.path.isfile(os.path.join(ref, "main.py")):
        sys.exit("rechorus_b200.overlay: no ReChorus main.py under %r (pass --ref <ReChorus>/src or set RECHORUS_SRC)" % ref)
    # the runner seams only matter when one of their flags is on the command line; otherwise the reference's own
    # BaseRunner class is the one main.py instantiates
    want_runner = any(a in ("--fused_step", "--device_metrics") or a.startswith(("--fused_step=", "--device_metrics="))
                      for a in argv)
    install(ref, b200_runner=want_runner)
    sys.argv = [os.path.join(ref, "main.py")] + argv
    runpy.run_path(os.path.join(ref, "main.py"), run_name="__main__")


if __name__ == "__main__":
    main()
