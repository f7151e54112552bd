"""The reference's UNCHANGED Main.py / Model_Trainer.py / Data_Container_OD.py on top of the engine (SURVEY.md section 8(b),
8(c) "Main.py plumbing", BASELINE.json configs[0]).

The reference ships no data (Data_Container_OD.py:15,34 read `od_day20180101_20210228.npz` and `adjacency_matrix.npy`), so
the tests write a synthetic pair of the right format (route (i) of SURVEY.md section 8(c)): a scipy sparse matrix whose
dense form reshapes to (-1, 47, 47) with >= 425 day rows, and a [47, 47] adjacency.  The reference itself is imported from
`oracle/_ref` (oracle/install_ref.py; untracked); without it the two trainer tests skip.  The rollout test compares with the
reference's prediction stored in tests/golden/ and needs no reference.

  * CPU (`-m "not gpu"`): the stock reference runs one epoch on that data (`tools/run_main.py --stock -GPU cpu`) -- the data
    shim is what Main.py expects;
  * GPU (`-m gpu`): the same command lines with this repository shadowing `MPGCN` / `GCN`: train 2 epochs, validation loss
    finite and decreasing, the checkpoint loads into the REFERENCE's own MPGCN class; then `-mode test` (autoregressive
    rollout + metrics) eagerly and with `--graph-rollout` -- identical scores.
"""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "oracle", "_ref")
RUN_MAIN = os.path.join(ROOT, "tools", "run_main.py")

needs_ref = pytest.mark.skipif(not os.path.isfile(os.path.join(REF, "Main.py")), reason="oracle/_ref (the unmodified reference) is not installed")


def write_synthetic_data(dirname, days=430, N=47, seed=0):
    """OD counts with weekly structure + a random sparse adjacency, in the two files DataInput.load_data reads."""
    import scipy.sparse as ss
    rng = np.random.default_rng(seed)
    base = rng.gamma(2.0, 20.0, size=(N, N))
    week = 1.0 + 0.3 * np.sin(2 * np.pi * np.arange(days) / 7.0)[:, None, None]
    od = rng.poisson(base[None] * week).astype(np.float64)
    ss.save_npz(os.path.join(dirname, "od_day20180101_20210228.npz"), ss.csr_matrix(od.reshape(days, N * N)))
    adj = (rng.random((N, N)) < 0.15).astype(np.float64)
    adj = np.maximum(adj, adj.T)
    np.fill_diagonal(adj, 1.0)
    np.save(os.path.join(dirname, "adjacency_matrix.npy"), adj)


def run_main(extra, main_args, timeout=1500):
    r = subprocess.run([sys.executable, RUN_MAIN] + extra + ["--"] + main_args, capture_output=True, text=True, timeout=timeout)
    assert r.returncode == 0, f"Main.py failed:\n{r.stdout[-3000:]}\n{r.stderr[-3000:]}"
    return r.stdout


def val_losses(stdout):
    """validation loss per epoch from the trainer's own prints (Model_Trainer.py:125-132)"""
    out = []
    for line in stdout.splitlines():
        m = re.match(r"Epoch (\d+), validation loss drops from \S+ to ([0-9.eE+-]+)\.", line)
        if m:
            out.append(float(m.group(2)))
    return out


@needs_ref
def test_stock_reference_runs_on_the_synthetic_data_cpu(tmp_path):
    """Plumbing of BASELINE.json configs[0] (localpool K=1, T=4, batch 2 on CPU), N = 47 as Data_Container_OD.py:16 hard-codes."""
    data, out = tmp_path / "data", tmp_path / "out"
    data.mkdir()
    write_synthetic_data(str(data))
    stdout = run_main(["--stock"], ["-GPU", "cpu", "-in", str(data), "-out", str(out), "-mode", "train", "-epoch", "1", "-kernel", "localpool",
                                   "-K", "1", "-obs", "4", "-batch", "2"])
    losses = val_losses(stdout)
    assert len(losses) == 1 and np.isfinite(losses[0])
    assert (out / "MPGCN_od.pkl").is_file()


@needs_ref
@pytest.mark.gpu
def test_unchanged_trainer_trains_and_tests_on_the_engine(tmp_path):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    data, out = tmp_path / "data", tmp_path / "out"
    data.mkdir()
    write_synthetic_data(str(data))
    common = ["-GPU", "cuda:0", "-in", str(data), "-out", str(out), "-batch", "4", "-lr", "1e-3"]
    stdout = run_main(["--seed", "0"], common + ["-mode", "train", "-epoch", "2"])      # the reference seeds nothing: fix the init for a stable assertion
    losses = val_losses(stdout)
    assert len(losses) >= 1 and all(np.isfinite(losses)), stdout[-2000:]
    assert len(losses) == 2 and losses[1] < losses[0], f"validation loss did not decrease over two epochs: {losses}"
    ckpt = torch.load(out / "MPGCN_od.pkl", map_location="cpu")
    # the checkpoint our modules wrote loads into the reference's own class, strictly
    sys.path.insert(0, REF)
    try:
        import importlib.util
        spec = importlib.util.spec_from_file_location("_ref_MPGCN_for_ckpt", os.path.join(REF, "MPGCN.py"))
        ref = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(ref)
    finally:
        sys.path.remove(REF)
    ref_model = ref.MPGCN(M=2, K=3, input_dim=1, lstm_hidden_dim=32, lstm_num_layers=1, gcn_hidden_dim=32, gcn_num_layers=3,
                          num_nodes=47, user_bias=True, activation=torch.nn.ReLU)
    ref_model.load_state_dict(ckpt["state_dict"], strict=True)
    # test mode: autoregressive rollout (pred_len = 3) + the reference's metrics, eagerly and through the captured graph
    scores = out / "MPGCN_prediction_scores.txt"
    run_main([], common + ["-mode", "test", "-pred", "3"])
    eager = scores.read_text().strip().splitlines()
    scores.unlink()
    run_main(["--graph-rollout", "--gpu-dyn-graphs"], common + ["-mode", "test", "-pred", "3"])
    graphed = scores.read_text().strip().splitlines()
    assert len(eager) == 2 and eager[0].startswith("train, MSE") and eager[1].startswith("test, MSE")
    vals = [float(v) for v in eager[1].split(",")[5:]]
    assert all(np.isfinite(vals)) and vals[0] > 0
    # same kernels on the same data: the graph replay reproduces the eager loop (the GPU dyn-graph builder differs from scipy
    # by ~1e-6, hence not bitwise)
    for le, lg in zip(eager, graphed):
        ve, vg = [float(v) for v in le.split(",")[5:]], [float(v) for v in lg.split(",")[5:]]
        assert np.allclose(ve, vg, rtol=1e-3), (le, lg)


@pytest.mark.gpu
def test_graph_rollout_install_matches_eager_and_reference(tmp_path):
    """rollout.install(model): the trainer-style horizon loop (Model_Trainer.py:157-165) through the captured graph is
    bit-identical to the eager loop, and both match the REFERENCE model's own loop (fp32 engine: <= 1e-4; fp16: <= 2e-3).
    The reference's prediction is the golden fixture rollout_n47_k3_p5 (oracle/gen_golden.py); its inputs and weights are
    regenerated here from the fixture's seeds and checked against the stored checksums."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    sys.path.insert(0, ROOT)
    import MPGCN as shim
    from conftest import load_golden
    from mpgcn_b200 import rollout
    from oracle import mpgcn_oracle as orc
    from oracle.gen_golden import ROLLOUT, horizon_loop, rollout_case_inputs, rollout_model_kwargs
    dev = torch.device("cuda:0")
    g = load_golden("rollout_n47_k3_p5")
    kw = rollout_model_kwargs()
    torch.manual_seed(ROLLOUT["seed"])
    init = shim.MPGCN(**kw).state_dict()          # the reference class draws the same default init under this seed
    np.testing.assert_allclose([float(v.double().sum()) for v in init.values()], g["param_sums"], rtol=1e-12,
                               err_msg="the default init no longer matches the weights the fixture was made with")
    x, G, go, gd = (torch.from_numpy(a) for a in rollout_case_inputs())
    np.testing.assert_allclose(float(x.double().sum()), float(g["x_checksum"]), rtol=1e-12)
    pred = ROLLOUT["pred"]
    want = g["y"]
    for prec, tol in (("fp32", 1e-4), ("fp16", 2e-3)):
        model = shim.MPGCN(**kw)
        model.load_state_dict(init)
        model = model.to(dev).eval()
        model.lstm_precision = prec
        for mod in model.modules():
            if isinstance(mod, shim.BDGCN):
                mod.precision = prec
        G_list = [G.to(dev), (go.to(dev), gd.to(dev))]
        eager = horizon_loop(model, x.to(dev), G_list, pred)
        rollout.install(model)
        graphed = horizon_loop(model, x.to(dev), G_list, pred)
        assert model.forward.captures == 1 and model.forward.replays == pred
        assert torch.equal(eager, graphed)
        rollout.uninstall(model)
        linf, l2 = orc.rel_errors(graphed.cpu().numpy(), want)
        assert linf <= tol and l2 <= tol, f"{prec}: rollout vs reference rel_Linf={linf:.2e} rel_L2={l2:.2e}"
