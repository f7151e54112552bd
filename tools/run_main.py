#!/usr/bin/env python
"""Run the reference's UNCHANGED `Main.py` on the B200 engine.

    python tools/run_main.py --reference-dir /path/to/MPGCN [--graph-rollout] [--gpu-dyn-graphs] -- -GPU cuda:0 -in ../data -mode train

What it does, and nothing more:
  * puts this repository ahead of the reference checkout on `sys.path`, so that `import GCN, MPGCN` in the reference's
    `Model_Trainer.py:5` resolves to the shims at the repository root (`MPGCN.py`, `GCN.py`) while `Main.py`,
    `Model_Trainer.py`, `Data_Container_OD.py`, `Metrics.py` stay the reference's own files;
  * `torch.cuda.set_device(<-GPU argument>)`, so that CPU tensors handed to `GCN.Adj_Processor.process` (the trainer moves
    them to `params['GPU']` only afterwards, Model_Trainer.py:41-42,84) are staged on the model's device;
  * `--gpu-dyn-graphs`: `mpgcn_b200.dyn_graph.install(Data_Container_OD.DataInput)` -- `construct_dyn_G` on the GPU
    (Data_Container_OD.py:39-59: 2*7*N^2 scipy calls otherwise);
  * `--graph-rollout`: `mpgcn_b200.rollout.install(model)` on the trainer's model -- the `pred_len` forward passes of
    `ModelTrainer.test` (Model_Trainer.py:157-165) replay one captured CUDA graph per batch.
Everything after `--` is Main.py's own command line (Main.py:11-37).
"""
import argparse
import os
import runpy
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference-dir", default=os.path.join(ROOT, "oracle", "_ref"))
    ap.add_argument("--graph-rollout", action="store_true")
    ap.add_argument("--gpu-dyn-graphs", action="store_true")
    ap.add_argument("--seed", type=int, default=None, help="torch.manual_seed / numpy seed before Main.py runs (the reference sets none)")
    ap.add_argument("--stock", action="store_true", help="do NOT shadow MPGCN / GCN: run the reference as it is (CPU plumbing check)")
    ap.add_argument("main_args", nargs=argparse.REMAINDER)
    a = ap.parse_args()
    ref = os.path.abspath(a.reference_dir)
    main_py = os.path.join(ref, "Main.py")
    if not os.path.isfile(main_py):
        sys.exit(f"no Main.py under {ref}")
    margs = a.main_args[1:] if a.main_args[:1] == ["--"] else a.main_args
    sys.path[:0] = [ref] if a.stock else [ROOT, ref]
    for m in ("MPGCN", "GCN", "Model_Trainer", "Data_Container_OD", "Metrics"):
        sys.modules.pop(m, None)
    if not a.stock:
        import torch
        gpu = next((margs[i + 1] for i, t in enumerate(margs[:-1]) if t in ("-GPU", "--GPU")), "cuda:2")     # Main.py:11 default
        if gpu.startswith("cuda"):
            torch.cuda.set_device(torch.device(gpu))
        if a.gpu_dyn_graphs:
            import Data_Container_OD
            from mpgcn_b200 import dyn_graph
            dyn_graph.install(Data_Container_OD.DataInput)
        if a.graph_rollout:
            import Model_Trainer
            from mpgcn_b200 import rollout
            get_model = Model_Trainer.ModelTrainer.get_model
            Model_Trainer.ModelTrainer.get_model = lambda self: rollout.install(get_model(self))
    if a.seed is not None:
        import numpy as np
        import torch
        torch.manual_seed(a.seed)
        np.random.seed(a.seed)
    sys.argv = [main_py] + margs
    os.chdir(ref)           # Main.py's defaults are relative paths (../data, ./output)
    runpy.run_path(main_py, run_name="__main__")


if __name__ == "__main__":
    main()
