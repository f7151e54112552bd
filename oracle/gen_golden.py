"""Generate the golden fixtures under tests/golden/ by running the UNMODIFIED reference.

TEST INFRASTRUCTURE ONLY (see oracle/mpgcn_oracle.py header).

Run in the build container, where /root/reference is mounted:

    python oracle/gen_golden.py            # writes tests/golden/*.npz

The script imports the reference modules `MPGCN` and `GCN` from /root/reference by bare
name (exactly how `Model_Trainer.py:5` imports them), instantiates the reference classes
on CPU in fp32 at fixed seeds, runs forward + autograd backward, and stores inputs,
parameters, outputs and gradients.  /root/reference does not exist on the GPU box, so
the fixtures -- not the reference -- travel.  Nothing here is copied from the reference;
it is only *called*.
"""
from __future__ import annotations

import importlib.util
import os
import sys

import numpy as np
import torch

REF = os.environ.get("MPGCN_REFERENCE_DIR", "/root/reference")
OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
ROOT = os.path.dirname(os.path.dirname(OUT))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def _load_ref(name):
    """Import a reference module under a private name so a repo-local `MPGCN.py` shim can
    never shadow it."""
    spec = importlib.util.spec_from_file_location(f"_ref_{name}", os.path.join(REF, f"{name}.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _np(t):
    return t.detach().cpu().numpy().copy()


def make_supports(ref_gcn, kind, K, N, batch, rng):
    """Support stacks.  kind: 'dense' -> N(0,1)/sqrt(N) (no identity shortcut);
    'rw' -> reference Adj_Processor('random_walk_diffusion', K-1) on a U[0,1) adjacency
    (K supports, T_0 = I; GCN.py:80-82,128-138); 'cheb' -> chebyshev (lambda_max=2 fallback,
    GCN.py:117-126); 'localpool' (K must be 1)."""
    shape = (batch, N, N) if batch else (1, N, N)
    if kind == "dense":
        g = (rng.standard_normal((shape[0], K, N, N)) / np.sqrt(N)).astype(np.float32)
    else:
        adj = torch.from_numpy(rng.random(shape).astype(np.float32))
        if kind == "rw":
            proc = ref_gcn.Adj_Processor("random_walk_diffusion", K - 1)
        elif kind == "cheb":
            proc = ref_gcn.Adj_Processor("chebyshev", K - 1)
        elif kind == "localpool":
            assert K == 1
            proc = ref_gcn.Adj_Processor("localpool", 1)
        else:
            raise ValueError(kind)
        g = _np(proc.process(adj))
        assert g.shape[1] == K, (g.shape, K)
    return g if batch else g[0]


BDGCN_CASES = [
    # name, dynamic, K, N, B, C, H, act, bias, support kind
    ("bdgcn_s_k1_n7", False, 1, 7, 2, 4, 5, "relu", True, "localpool"),
    ("bdgcn_s_k3_n12", False, 3, 12, 2, 8, 8, "relu", True, "rw"),
    ("bdgcn_s_k3_n12_linear_nobias", False, 3, 12, 2, 8, 8, None, False, "dense"),
    ("bdgcn_d_k3_n10", True, 3, 10, 3, 8, 8, "relu", True, "rw"),
    ("bdgcn_s_k6_n9", False, 6, 9, 1, 4, 6, "relu", True, "dense"),
    ("bdgcn_s_k2_n16_cheb", False, 2, 16, 2, 6, 3, "relu", True, "cheb"),
    ("bdgcn_s_k3_n47_c32", False, 3, 47, 1, 32, 32, "relu", True, "rw"),
    ("bdgcn_d_k3_n33_c32", True, 3, 33, 2, 32, 32, "relu", True, "dense"),
    ("bdgcn_s_k1_n50_c32", False, 1, 50, 2, 32, 32, "relu", True, "localpool"),
]


def gen_bdgcn(ref_mpgcn, ref_gcn):
    for idx, (name, dyn, K, N, B, C, H, act, bias, gk) in enumerate(BDGCN_CASES):
        rng = np.random.default_rng(1000 + idx)
        torch.manual_seed(1000 + idx)
        layer = ref_mpgcn.BDGCN(K=K, input_dim=C, hidden_dim=H, use_bias=bias,
                                activation=torch.nn.ReLU if act == "relu" else None)
        if bias:   # reference inits b to 0; use a non-trivial bias so the add is exercised
            with torch.no_grad():
                layer.b.copy_(torch.from_numpy(rng.standard_normal(H).astype(np.float32) * 0.1))
        X = np.tanh(rng.standard_normal((B, N, N, C))).astype(np.float32)
        d_out = rng.standard_normal((B, N, N, H)).astype(np.float32)
        Xt = torch.from_numpy(X).requires_grad_(True)
        if dyn:
            go = make_supports(ref_gcn, gk, K, N, B, rng)
            gd = make_supports(ref_gcn, gk, K, N, B, rng)
            G = (torch.from_numpy(go), torch.from_numpy(gd))
        else:
            g = make_supports(ref_gcn, gk, K, N, 0, rng)
            G = torch.from_numpy(g)
        out = layer(Xt, G)
        out.backward(torch.from_numpy(d_out))
        rec = dict(X=X, W=_np(layer.W), d_out=d_out, out=_np(out), dX=_np(Xt.grad), dW=_np(layer.W.grad),
                   K=K, act=act or "none", dynamic=int(dyn))
        if bias:
            rec.update(b=_np(layer.b), db=_np(layer.b.grad))
        if dyn:
            rec.update(G_o=go, G_d=gd)
        else:
            rec.update(G=g)
        np.savez_compressed(os.path.join(OUT, name + ".npz"), **rec)
        print("wrote", name, "out", out.shape)


# At-size layer cases (C = H = 32, B = 1; tile boundaries of the tcgen05 engine: N = 129 -> second 128-row tile / first 2-CTA
# pair tile, N = 200 = BASELINE.json configs[1]).  To keep the fixtures small the activations are NOT stored: X and d_out are
# regenerated from the seed by `big_case_inputs` (numpy PCG64 streams are stable across versions; a checksum is stored and
# asserted by the tests), and of the reference's outputs only `BIG_ROWS` origin rows of out / dX are kept (every element of
# out depends on all of X, so a row subset pins the whole contraction), plus dW and db in full.
BIG_CASES = [
    # name, dynamic, K, N, support kind
    ("bdgcn_s_k3_n129_c32", False, 3, 129, "rw"),
    ("bdgcn_d_k3_n129_c32", True, 3, 129, "dense"),
    ("bdgcn_s_k3_n200_c32", False, 3, 200, "dense"),
]


def big_rows(N):
    """Origin rows kept in an at-size fixture: tile edges (63/64, 127/128, last) and a spread in between."""
    rows = {0, 1, 31, 32, 63, 64, 65, 100, 126, 127, 128, N - 2, N - 1} | set(range(7, N, 17))
    return np.asarray(sorted(r for r in rows if 0 <= r < N)[:28], dtype=np.int64)


def big_case_inputs(seed, N, C=32, H=32):
    """(X [1,N,N,C], d_out [1,N,N,H]) of an at-size fixture, from the seed alone."""
    rng = np.random.default_rng(seed)
    X = np.tanh(rng.standard_normal((1, N, N, C))).astype(np.float32)
    d_out = rng.standard_normal((1, N, N, H)).astype(np.float32)
    return X, d_out


def gen_bdgcn_big(ref_mpgcn, ref_gcn):
    for idx, (name, dyn, K, N, gk) in enumerate(BIG_CASES):
        seed = 6000 + idx
        C = H = 32
        rng = np.random.default_rng(seed + 500)
        torch.manual_seed(seed)
        layer = ref_mpgcn.BDGCN(K=K, input_dim=C, hidden_dim=H, use_bias=True, activation=torch.nn.ReLU)
        with torch.no_grad():
            layer.b.copy_(torch.from_numpy(rng.standard_normal(H).astype(np.float32) * 0.1))
        X, d_out = big_case_inputs(seed, N, C, H)
        Xt = torch.from_numpy(X).requires_grad_(True)
        if dyn:
            go, gd = make_supports(ref_gcn, gk, K, N, 1, rng), make_supports(ref_gcn, gk, K, N, 1, rng)
            G = (torch.from_numpy(go), torch.from_numpy(gd))
        else:
            g = make_supports(ref_gcn, gk, K, N, 0, rng)
            G = torch.from_numpy(g)
        out = layer(Xt, G)
        out.backward(torch.from_numpy(d_out))
        rows = big_rows(N)
        rec = dict(seed=seed, N=N, K=K, dynamic=int(dyn), act="relu", rows=rows, W=_np(layer.W), b=_np(layer.b),
                   x_checksum=np.float64(X.astype(np.float64).sum()), d_out_checksum=np.float64(d_out.astype(np.float64).sum()),
                   x_probe=X[0, rows[:4], 5, :4].copy(),
                   out_rows=_np(out)[:, rows], dX_rows=_np(Xt.grad)[:, rows], dW=_np(layer.W.grad), db=_np(layer.b.grad),
                   out_absmax=np.float32(np.abs(_np(out)).max()), dX_absmax=np.float32(np.abs(_np(Xt.grad)).max()),
                   out_norm=np.float64(np.linalg.norm(_np(out).astype(np.float64))), dX_norm=np.float64(np.linalg.norm(_np(Xt.grad).astype(np.float64))))
        if dyn:
            rec.update(G_o=go, G_d=gd)
        else:
            rec.update(G=g)
        np.savez_compressed(os.path.join(OUT, name.replace("bdgcn_", "big_bdgcn_") + ".npz"), **rec)
        print("wrote", name, "rows", len(rows))


LSTM_CASES = [("lstm_s50_t5_c8", 50, 5, 8), ("lstm_s96_t4_c32", 96, 4, 32), ("lstm_s33_t12_c32", 33, 12, 32)]


def gen_lstm():
    for idx, (name, S, T, C) in enumerate(LSTM_CASES):
        rng = np.random.default_rng(2000 + idx)
        torch.manual_seed(2000 + idx)
        lstm = torch.nn.LSTM(input_size=1, hidden_size=C, num_layers=1, batch_first=True)   # MPGCN.py:69
        x = (rng.random((S, T, 1)) * 8).astype(np.float32)       # log1p(flow)-like range
        d_h = rng.standard_normal((S, C)).astype(np.float32)
        xt = torch.from_numpy(x).requires_grad_(True)
        h0 = torch.zeros(1, S, C)
        out, _ = lstm(xt, (h0, h0.clone()))                      # MPGCN.py:80-87,103
        hT = out[:, -1, :]                                       # MPGCN.py:104
        hT.backward(torch.from_numpy(d_h))
        np.savez_compressed(os.path.join(OUT, name + ".npz"), x=x, d_hT=d_h, hT=_np(hT), dx=_np(xt.grad),
                            w_ih=_np(lstm.weight_ih_l0), w_hh=_np(lstm.weight_hh_l0),
                            b_ih=_np(lstm.bias_ih_l0), b_hh=_np(lstm.bias_hh_l0),
                            dw_ih=_np(lstm.weight_ih_l0.grad), dw_hh=_np(lstm.weight_hh_l0.grad),
                            db_ih=_np(lstm.bias_ih_l0.grad), db_hh=_np(lstm.bias_hh_l0.grad))
        print("wrote", name)


MODEL_CASES = [
    # name, N, K_supports, kernel, T, B, hidden        (M=2: static + dynamic, as Model_Trainer.py:47,107)
    ("mpgcn_cfg1_n50_k1", 50, 1, "localpool", 4, 2, 32),        # BASELINE.json configs[0]
    ("mpgcn_n6_k3", 6, 3, "rw", 3, 2, 8),
    ("mpgcn_n20_k3_h32", 20, 3, "rw", 5, 2, 32),
]


def _gen_one_model(ref_mpgcn, ref_gcn, seed, N, K, gk, T, B, hid):
    rng = np.random.default_rng(seed)
    torch.manual_seed(seed)
    model = ref_mpgcn.MPGCN(M=2, K=K, input_dim=1, lstm_hidden_dim=hid, lstm_num_layers=1,
                            gcn_hidden_dim=hid, gcn_num_layers=3, num_nodes=N, user_bias=True,
                            activation=torch.nn.ReLU)        # Model_Trainer.py:47-56
    x_seq = (rng.random((B, T, N, N, 1)) * 8).astype(np.float32)
    g_static = make_supports(ref_gcn, gk, K, N, 0, rng)
    g_o = make_supports(ref_gcn, gk, K, N, B, rng)
    g_d = make_supports(ref_gcn, gk, K, N, B, rng)
    d_y = rng.standard_normal((B, 1, N, N, 1)).astype(np.float32)
    y = model(x_seq=torch.from_numpy(x_seq), G_list=[torch.from_numpy(g_static), (torch.from_numpy(g_o), torch.from_numpy(g_d))])
    y.backward(torch.from_numpy(d_y))
    if not all(float(p.grad.abs().max()) > 0 for p in model.parameters()):
        return None
    rec = dict(x_seq=x_seq, G_static=g_static, G_o=g_o, G_d=g_d, d_y=d_y, y=_np(y), K=K, hidden=hid, seed=seed)
    for k, v in model.state_dict().items():
        rec["param:" + k] = _np(v)
    for k, p in model.named_parameters():
        rec["grad:" + k] = _np(p.grad)
    return rec


def gen_model(ref_mpgcn, ref_gcn):
    """Default init can leave a branch's FC ReLU dead on every cell (all of that branch's gradients exactly zero: round 1's
    cfg1 fixture pinned only the static half of the model), so each case takes the first seed of 3000+idx, 3100+idx, ...
    for which every parameter of BOTH branches receives a non-zero gradient."""
    for idx, (name, N, K, gk, T, B, hid) in enumerate(MODEL_CASES):
        for seed in range(3000 + idx, 6000, 100):
            rec = _gen_one_model(ref_mpgcn, ref_gcn, seed, N, K, gk, T, B, hid)
            if rec is not None:
                break
            print("  ", name, "seed", seed, "leaves a dead branch, trying the next")
        else:
            raise RuntimeError(f"{name}: no seed with two live branches")
        np.savez_compressed(os.path.join(OUT, name + ".npz"), **rec)
        print("wrote", name, "y", rec["y"].shape, "seed", seed)


ADJ_CASES = [
    # name, kernel, K (order), N, B
    ("adj_localpool_n9", "localpool", 1, 9, 2),
    ("adj_cheb_k2_n16", "chebyshev", 2, 16, 2),
    ("adj_cheb_k3_n33", "chebyshev", 3, 33, 1),
    ("adj_rw_k1_n12", "random_walk_diffusion", 1, 12, 2),
    ("adj_rw_k2_n47", "random_walk_diffusion", 2, 47, 2),
    ("adj_rw_k4_n20", "random_walk_diffusion", 4, 20, 1),
    ("adj_dual_k2_n21", "dual_random_walk_diffusion", 2, 21, 2),
    ("adj_rw_k2_n10_zero_row", "random_walk_diffusion", 2, 10, 1),
]


def gen_adj(ref_gcn):
    for idx, (name, kind, K, N, B) in enumerate(ADJ_CASES):
        rng = np.random.default_rng(4000 + idx)
        flow = rng.random((B, N, N)).astype(np.float32) * 5
        if "zero_row" in name:
            flow[0, 3, :] = 0        # zero out-degree: random_walk_normalize maps 1/0 -> 0 (GCN.py:105)
        proc = ref_gcn.Adj_Processor(kind, K)
        sup = _np(proc.process(torch.from_numpy(flow)))
        np.savez_compressed(os.path.join(OUT, name + ".npz"), flow=flow, supports=sup, kernel_type=kind, K=K)
        print("wrote", name, sup.shape)


DYN_CASES = [
    # name, N, days, split_ratio, zero_row
    ("dyn_n12_d70", 12, 70, [6.4, 1.6, 2], False),
    ("dyn_n20_d45", 20, 45, [6.4, 1.6, 2], False),      # 45 days -> train_len 28 -> 4 periods
    ("dyn_n9_d30_zero", 9, 30, [7, 1, 2], True),        # an all-zero origin row: NaN entries, as scipy produces
]


def gen_dyn(ref_data):
    """DataInput.construct_dyn_G of the unmodified reference (Data_Container_OD.py:39-59; scipy distance.cosine per pair)."""
    import warnings
    for idx, (name, N, days, split, zero_row) in enumerate(DYN_CASES):
        rng = np.random.default_rng(5000 + idx)
        od = rng.poisson(6.0, size=(days, N, N, 1)).astype(np.float64)
        od[:, :, 2, :] *= 0.25                                     # make the graphs less uniform
        if zero_row:
            od[:, 4, :, :] = 0
        di = ref_data.DataInput({"split_ratio": split})
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            o_g, d_g = di.construct_dyn_G(od)
        np.savez_compressed(os.path.join(OUT, name + ".npz"), od=od.astype(np.float32), split_ratio=np.asarray(split, dtype=np.float64),
                            O_dyn_G=o_g, D_dyn_G=d_g)
        print("wrote", name, o_g.shape, "nan:", int(np.isnan(o_g).sum()), int(np.isnan(d_g).sum()))


# The trainer-style horizon loop of tests/test_trainer_dropin.py (Model_Trainer.py:157-165) on the reference model.  Inputs come
# from seeds alone (`rollout_case_inputs`) and the weights are the default init under torch.manual_seed(seed) -- the same for
# the reference class and the engine's drop-in; checksums of both are stored and asserted by the test -- so only the
# reference's prediction is kept.
ROLLOUT = dict(N=47, K=3, T=7, B=4, pred=5, seed=3)


def rollout_model_kwargs():
    return dict(M=2, K=ROLLOUT["K"], input_dim=1, lstm_hidden_dim=32, lstm_num_layers=1, gcn_hidden_dim=32, gcn_num_layers=3,
                num_nodes=ROLLOUT["N"], user_bias=True, activation=torch.nn.ReLU)


def rollout_case_inputs():
    """(x [B,T,N,N,1], G [K,N,N], G_o [B,K,N,N], G_d [B,K,N,N]) of the rollout fixture: random-walk supports of U[0,1)
    adjacencies through the oracle's adj_process (pinned to the reference by the adj_* fixtures)."""
    from oracle import mpgcn_oracle as orc
    N, K, T, B = (ROLLOUT[k] for k in "NKTB")
    rng = np.random.default_rng(1)
    x = (rng.random((B, T, N, N, 1)) * 6).astype(np.float32)
    sup = lambda b: orc.adj_process(rng.random((max(b, 1), N, N)).astype(np.float32), "random_walk_diffusion", K - 1).astype(np.float32)
    G, go, gd = sup(0)[0], sup(B), sup(B)
    return x, G, go, gd


def horizon_loop(model, x, G_list, pred):
    """The reference trainer's autoregressive test loop (Model_Trainer.py:157-165)."""
    y_pred, cur = [], x
    with torch.no_grad():
        for _ in range(pred):
            step = model(x_seq=cur, G_list=G_list)
            cur = torch.cat([cur[:, 1:, :, :, :], step], dim=1)
            y_pred.append(step)
    return torch.cat(y_pred, dim=1)


def gen_rollout(ref_mpgcn):
    torch.manual_seed(ROLLOUT["seed"])
    model = ref_mpgcn.MPGCN(**rollout_model_kwargs()).eval()
    x, G, go, gd = (torch.from_numpy(a) for a in rollout_case_inputs())
    y = horizon_loop(model, x, [G, (go, gd)], ROLLOUT["pred"])
    np.savez_compressed(os.path.join(OUT, "rollout_n47_k3_p5.npz"), y=_np(y), x_checksum=np.float64(x.double().sum()),
                        param_sums=np.array([float(v.double().sum()) for v in model.state_dict().values()]))
    print("wrote rollout_n47_k3_p5", tuple(y.shape))


def main():
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    if not os.path.isdir(REF):
        sys.exit(f"reference not found at {REF}; fixtures can only be regenerated in the build container")
    ref_mpgcn = _load_ref("MPGCN")
    ref_gcn = _load_ref("GCN")
    only = sys.argv[1:]                  # e.g. `gen_golden.py big model`: regenerate only those groups
    want = lambda k: not only or k in only
    if want("bdgcn"):
        gen_bdgcn(ref_mpgcn, ref_gcn)
    if want("big"):
        gen_bdgcn_big(ref_mpgcn, ref_gcn)
    if want("lstm"):
        gen_lstm()
    if want("model"):
        gen_model(ref_mpgcn, ref_gcn)
    if want("adj"):
        gen_adj(ref_gcn)
    if want("dyn"):
        gen_dyn(_load_ref("Data_Container_OD"))
    if want("rollout"):
        gen_rollout(ref_mpgcn)


if __name__ == "__main__":
    main()
