"""CPU timing arm: the reference's execution strategy, restated with torch CPU ops.

TEST / BENCH INFRASTRUCTURE ONLY (see oracle/mpgcn_oracle.py header).  Used by `bench.py` for the
`cpu_baseline` object and the `--impl reference` arm, because /root/reference does not exist on the
GPU box and a Python reference cannot travel.

It deliberately mirrors what the reference *executes* on a CPU -- not the factored algebra our
engine uses -- so that its timing stands in for the reference's own:
  * BDGCN (reference MPGCN.py:24-50): for every ordered support pair (o, d) an origin-mode einsum
    followed by a destination-mode einsum (the origin product is recomputed inside the d loop, as
    the reference does), channel concatenation of the K*K results, one einsum with W, bias, ReLU;
    gradients by torch autograd;
  * temporal encoder (MPGCN.py:69,100-104): torch.nn.functional-level LSTM over B*N*N sequences
    (oneDNN on CPU, like nn.LSTM in the reference), last step only.
Checked against the numpy oracle in tests/test_oracle_golden.py::test_torch_port_matches_oracle.
"""
from __future__ import annotations

import time

import torch


def bdgcn_layer(X, G, W, b=None, relu=True):
    """K*K-pair evaluation (the reference's executed order)."""
    K = G.shape[-3] if isinstance(G, torch.Tensor) else G[0].shape[-3]
    pieces = []
    for o in range(K):
        for d in range(K):
            if isinstance(G, torch.Tensor):
                t = torch.einsum("bncl,nm->bmcl", X, G[o])
                t = torch.einsum("bmcl,ce->bmel", t, G[d])
            else:
                t = torch.einsum("bncl,bnm->bmcl", X, G[0][:, o])
                t = torch.einsum("bmcl,bce->bmel", t, G[1][:, d])
            pieces.append(t)
    y = torch.einsum("bmek,kh->bmeh", torch.cat(pieces, dim=-1), W)
    if b is not None:
        y = y + b
    return torch.relu(y) if relu else y


def lstm_last(x_cells, lstm):
    """x_cells [S,T,1] -> h_T [S,C] with a zero initial state."""
    out, _ = lstm(x_cells)
    return out[:, -1, :]


def time_bdgcn_layer_fwd_bwd(N, K, B=1, C=32, H=32, repeats=1, seed=0):
    """Seconds for one BDGCN layer forward + backward (B samples) on the host CPU."""
    g = torch.Generator().manual_seed(seed)
    X = torch.tanh(torch.randn(B, N, N, C, generator=g)).requires_grad_(True)
    G = torch.randn(K, N, N, generator=g) / N ** 0.5
    W = (torch.randn(K * K * C, H, generator=g) * (2.0 / (K * K * C + H)) ** 0.5).requires_grad_(True)
    b = torch.zeros(H, requires_grad=True)
    best = float("inf")
    for _ in range(repeats):
        t0 = time.perf_counter()
        y = bdgcn_layer(X, G, W, b, relu=True)
        y.sum().backward()
        best = min(best, time.perf_counter() - t0)
        X.grad = W.grad = b.grad = None
    return best


def time_lstm_fwd_bwd(cells, T, C=32, repeats=1, seed=0):
    """Seconds for the temporal encoder forward + backward over `cells` sequences."""
    torch.manual_seed(seed)
    lstm = torch.nn.LSTM(input_size=1, hidden_size=C, num_layers=1, batch_first=True)
    x = torch.rand(cells, T, 1) * 8
    best = float("inf")
    for _ in range(repeats):
        t0 = time.perf_counter()
        h = lstm_last(x, lstm)
        h.sum().backward()
        best = min(best, time.perf_counter() - t0)
        lstm.zero_grad()
    return best


def estimate_model_step_seconds(N, K, T, M=2, L=3, C=32, lstm_sample_cells=None, seed=0):
    """Bounded-sample estimate of one full-model forward+backward for ONE sample (B=1):
        M * ( L * t(BDGCN layer fwd+bwd, B=1) + t(LSTM fwd+bwd over N*N cells) )
    The BDGCN layer is timed at full size for B=1; the LSTM on `lstm_sample_cells` cells and scaled
    linearly to N*N (cells are independent).  Returns (seconds, detail dict)."""
    t_layer = time_bdgcn_layer_fwd_bwd(N, K, B=1, C=C, H=C, seed=seed)
    cells = N * N
    sample = min(cells, lstm_sample_cells or 200_000)
    t_lstm_sample = time_lstm_fwd_bwd(sample, T, C=C, seed=seed)
    t_lstm = t_lstm_sample * cells / sample
    total = M * (L * t_layer + t_lstm)
    return total, dict(t_bdgcn_layer_s=t_layer, t_lstm_sample_s=t_lstm_sample, lstm_sample_cells=sample, t_lstm_scaled_s=t_lstm,
                       formula="M*(L*t_layer + t_lstm), B=1")


class PortBDGCN(torch.nn.Module):
    """The port's layer as a module with the reference's parameter names (W [K*K*C, H], b [H]); MPGCN.py:6-50."""

    def __init__(self, K, input_dim, hidden_dim, use_bias=True, activation=None):
        super().__init__()
        self.K = K
        self.W = torch.nn.Parameter(torch.empty(K * K * input_dim, hidden_dim))
        torch.nn.init.xavier_normal_(self.W)
        self.b = torch.nn.Parameter(torch.zeros(hidden_dim)) if use_bias else None
        self.relu = activation is not None

    def forward(self, X, G):
        return bdgcn_layer(X, G, self.W, self.b, relu=self.relu)


class PortMPGCN(torch.nn.Module):
    """The port's model: per branch nn.LSTM over B*N*N cells (zero state, last step) -> L x PortBDGCN -> Linear+ReLU, mean over
    branches (MPGCN.py:54-112), including the reference's materialisations (zero (h0, c0), the full lstm_out, stack + mean).
    Used only where the real reference (oracle/_ref) is not available."""

    def __init__(self, M, K, input_dim, lstm_hidden_dim, lstm_num_layers, gcn_hidden_dim, gcn_num_layers, num_nodes, user_bias,
                 activation=None):
        super().__init__()
        self.M, self.N, self.C, self.layers = M, num_nodes, lstm_hidden_dim, lstm_num_layers
        self.branch_models = torch.nn.ModuleList()
        for _ in range(M):
            br = torch.nn.ModuleDict()
            br["temporal"] = torch.nn.LSTM(input_size=input_dim, hidden_size=lstm_hidden_dim, num_layers=lstm_num_layers, batch_first=True)
            br["spatial"] = torch.nn.ModuleList(PortBDGCN(K, lstm_hidden_dim if n == 0 else gcn_hidden_dim, gcn_hidden_dim, user_bias, activation)
                                                for n in range(gcn_num_layers))
            br["fc"] = torch.nn.Sequential(torch.nn.Linear(gcn_hidden_dim, input_dim), torch.nn.ReLU())
            self.branch_models.append(br)

    def forward(self, x_seq, G_list):
        B, T, N, _, I = x_seq.shape
        lstm_in = x_seq.permute(0, 2, 3, 1, 4).reshape(B * N * N, T, I)
        outs = []
        for m in range(self.M):
            br = self.branch_models[m]
            h0 = x_seq.new_zeros(self.layers, B * N * N, self.C)
            out, _ = br["temporal"](lstm_in, (h0, h0.clone()))
            g = out[:, -1, :].reshape(B, N, N, self.C)
            for layer in br["spatial"]:
                g = layer(g, G_list[m])
            outs.append(br["fc"](g))
        return torch.mean(torch.stack(outs, dim=-1), dim=-1).unsqueeze(dim=1)
