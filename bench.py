#!/usr/bin/env python
"""bench.py -- OD-cells/s of the MPGCN hot path (per-cell LSTM -> 3 x BDGCN -> FC head, M=2 branches, forward +
backward) on synthetic OD tensors, on N GPUs of one node.

    python bench.py --gpus 1 --steps 10 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W [--shard batch|row|k]
    python bench.py --impl reference --steps K --warmup W        # CPU arm: the unmodified reference from oracle/_ref

Workload (BASELINE.json metric "OD-cells/sec (B*T*N^2) 2D-GCN fwd+bwd at N=1000,K=3"): `--workload headline` = N=1000
nodes, K=3 supports, T=12, hidden 32, M=2 branches (static + dynamic graph), 3 BDGCN layers per branch, batch 8 per GPU
(SURVEY.md section 8(d)); cfg2..cfg5 select BASELINE.json configs[1..4].  A step = one forward + backward of the whole
hot path over one batch (+ the exchange step of the chosen shard).

    --shard batch (default)  every rank runs its own samples; only the parameter gradients are all-reduced      "weak"
    --shard row              every sample's ORIGIN ROWS are split over the ranks (SURVEY.md 8(e) row 1): the forward
                             reduce-scatters the pre-activation of every layer, the backward all-gathers dPre           "strong"
    --shard k                the DESTINATION SUPPORTS are split (8(e) row 2, the partition north_star names): all-reduce
                             of the pre-activation forward, of dX backward                                               "strong"

One JSON line is printed by rank 0 (field meanings: README.md / DESIGN.md section 7).
"""
from __future__ import annotations

import argparse
import importlib.util
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "OD-cells/sec (B*T*N^2), MPGCN hot path fwd+bwd"
UNIT = "OD-cells/s"
REF_DIR = os.path.join(ROOT, "oracle", "_ref")

WORKLOADS = {          # name: (N, K, T, batch per GPU)   -- BASELINE.json configs / SURVEY.md section 8(d)
    "headline": (1000, 3, 12, 8),
    "cfg2": (200, 3, 8, 16),
    "cfg3": (500, 3, 12, 32),
    "cfg4": (1000, 6, 12, 8),
    "cfg5": (2000, 3, 8, 2),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference", "library"], default="ours",
                    help="ours: the engine; reference: the reference's CPU path (bounded sample); library: (internal) the reference model on the "
                         "GPU through cuBLAS / cuDNN, printed as gpu_library_baseline by the default arm")
    ap.add_argument("--workload", choices=sorted(WORKLOADS), default="headline")
    ap.add_argument("--nodes", type=int, default=None, help="N (OD zones); overrides --workload")
    ap.add_argument("--supports", type=int, default=None, help="K")
    ap.add_argument("--obs", type=int, default=None, help="T")
    ap.add_argument("--batch", type=int, default=None, help="samples per GPU (batch shard) / in total (row, k shards)")
    ap.add_argument("--hidden", type=int, default=32)
    ap.add_argument("--precision", default="fp16", choices=["fp16", "fp32", "auto"])
    ap.add_argument("--shard", default="batch", choices=["batch", "row", "k"])
    ap.add_argument("--row-ranks", type=int, default=0,
                    help="row shard: ranks per row group (default: all).  R < N GPUs = hybrid: N/R groups of R consecutive ranks, every group "
                         "takes batch/(N/R) of the samples and splits THEIR origin rows R ways -- the exchange stays inside a group")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--profile", action="store_true", help="under ncu: honour --warmup < 3, skip the e2e / CPU / library arms (numbers are not bench values)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (loss, prediction, parameter gradients; rank 0's) "
                         "as DIR/<name>.npy in float32, at most 64 MB in all")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    N, K, T, B = WORKLOADS[a.workload]
    a.nodes = a.nodes or N
    a.supports = a.supports or K
    a.obs = a.obs or T
    a.batch = a.batch or B
    return a


def workload_config(a, world):
    if a.shard == "batch":
        gb, par = a.batch * world, f"batch-shard x{world}"
    else:
        R = a.row_ranks if (a.shard == "row" and 0 < a.row_ranks < world) else world
        gb = a.batch
        par = (f"{'origin-row' if a.shard == 'row' else 'K (destination-support)'}-shard x{R}" + (f" x batch-shard x{world // R}" if R < world else ""))
    return {
        "workload": f"MPGCN hot path N={a.nodes} K={a.supports} T={a.obs} hidden={a.hidden} M=2 L=3, "
                    + (f"batch {a.batch}/GPU" if a.shard == "batch" else f"batch {a.batch} in total"),
        "N": a.nodes, "K": a.supports, "T": a.obs, "hidden": a.hidden, "M": 2, "gcn_layers": 3,
        "batch_per_gpu": a.batch if a.shard == "batch" else None, "global_batch": gb, "parallelism": par,
        "precision": a.precision, "l2": "inputs exceed L2 (activations >= 0.5 GB per layer); no explicit flush",
    }


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return dict(tflops=float(d["bf16_tflops_sustained"]), tflops_burst=float(d["bf16_tflops"]), hbm=float(d["hbm_gbs"]),
                        source="MEASURED_PEAKS.json (bf16 sustained; kernel timed inside a long step)")
        except Exception:
            pass
    return dict(tflops=1400.0, tflops_burst=1590.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows)]
        pw = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "power_w_max": max(pw) if pw else None, "samples": len(self.rows)}


# ------------------------------------------------------------------------------------------------
# the reference (unmodified, from oracle/_ref) or -- only where that is absent -- its torch port
# ------------------------------------------------------------------------------------------------
def load_reference_impl():
    """-> (module-like object with BDGCN and MPGCN classes, kind).  kind "reference": the unmodified classes of
    underdoc-wang/MPGCN imported from oracle/_ref (oracle/install_ref.py put them there; the directory is not tracked);
    "port": oracle/torch_port.py, a torch restatement of the reference's execution order."""
    f = os.path.join(REF_DIR, "MPGCN.py")
    if os.path.isfile(f):
        spec = importlib.util.spec_from_file_location("_reference_MPGCN", f)      # private name: the repo's MPGCN.py shim cannot shadow it
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        return mod, "reference"
    from oracle import torch_port

    class _Port:
        BDGCN, MPGCN = torch_port.PortBDGCN, torch_port.PortMPGCN
    return _Port, "port"


class CpuArm:
    """The reference's CPU path, timed on a BOUNDED sample that is exactly one sixth of one B=1 model step at the
    benchmarked size: ONE BDGCN layer forward + backward (the reference's own `BDGCN` class, static supports on even
    samples, a dynamic (G_o, G_d) tuple on odd ones) plus its `nn.LSTM` forward + backward over a third of the N*N
    cells (the model has 6 layers and 2 LSTM passes per sample).  No size extrapolation: the layer runs at the full
    N, K; the sample is credited with T*N*N/6 OD cells and the reported time is the time it really took."""

    def __init__(self, a):
        import torch
        self.torch = torch
        self.a = a
        self.impl, self.kind = load_reference_impl()
        self.cores = os.cpu_count() or 1
        torch.set_num_threads(self.cores)
        N, K, C = a.nodes, a.supports, a.hidden
        g = torch.Generator().manual_seed(99)
        self.layer = self.impl.BDGCN(K=K, input_dim=C, hidden_dim=C, use_bias=True, activation=torch.nn.ReLU)
        self.lstm = torch.nn.LSTM(input_size=1, hidden_size=C, num_layers=1, batch_first=True)       # MPGCN.py:69
        self.X = torch.tanh(torch.randn(1, N, N, C, generator=g))
        self.G = torch.randn(K, N, N, generator=g) / N ** 0.5
        self.Gdyn = (torch.randn(1, K, N, N, generator=g) / N ** 0.5, torch.randn(1, K, N, N, generator=g) / N ** 0.5)
        self.cells = (N * N + 2) // 3
        self.x_cells = torch.rand(self.cells, a.obs, 1, generator=g) * 8
        self.lstm_threads = self._pick_lstm_threads()
        self.count = 0

    def _lstm_pass(self, x):
        h0 = x.new_zeros(1, x.shape[0], self.a.hidden)
        out, _ = self.lstm(x, (h0, h0.clone()))                     # MPGCN.py:80-87,103
        out[:, -1, :].sum().backward()                              # MPGCN.py:104
        self.lstm.zero_grad(set_to_none=True)

    def _pick_lstm_threads(self):
        """oneDNN's LSTM on B*N*N short sequences of hidden 32 slows down when spread over too many threads (round 1: 6.3 s
        for 20 000 cells on 128 threads); probe a few thread counts once (untimed) and keep the fastest."""
        torch = self.torch
        x = self.x_cells[:20000]
        best, best_t = self.cores, float("inf")
        for nt in sorted({min(self.cores, n) for n in (8, 16, 32, 64, self.cores)}):
            torch.set_num_threads(nt)
            self._lstm_pass(x[:2000])
            t0 = time.perf_counter()
            self._lstm_pass(x)
            t = time.perf_counter() - t0
            if t < best_t:
                best, best_t = nt, t
        torch.set_num_threads(self.cores)
        return best

    def sample(self):
        """-> (seconds, OD cells credited)"""
        torch = self.torch
        a = self.a
        G = self.G if self.count % 2 == 0 else self.Gdyn
        self.count += 1
        X = self.X.clone().requires_grad_(True)
        t0 = time.perf_counter()
        torch.set_num_threads(self.cores)
        y = self.layer(X, G)                                        # MPGCN.py:24-50
        y.sum().backward()
        self.layer.zero_grad(set_to_none=True)
        torch.set_num_threads(self.lstm_threads)
        self._lstm_pass(self.x_cells)
        torch.set_num_threads(self.cores)
        return time.perf_counter() - t0, a.obs * a.nodes * a.nodes / 6.0

    def describe(self):
        a = self.a
        return (f"1/6 of one B=1 model step at full size: one BDGCN layer fwd+bwd (N={a.nodes}, K={a.supports}, C=H={a.hidden}; "
                f"{'unmodified reference class from oracle/_ref' if self.kind == 'reference' else 'torch port of the reference order'}; static / dynamic "
                f"supports alternate) on {self.cores} threads + nn.LSTM fwd+bwd over {self.cells} of {a.nodes ** 2} cells, T={a.obs}, on "
                f"{self.lstm_threads} threads (fastest of a probe); credited T*N*N/6 OD cells; no size extrapolation")


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return None
    world = int(os.environ.get("WORLD_SIZE", "1"))
    arm = CpuArm(a)
    for _ in range(a.warmup):
        arm.sample()
    ts, cells = [], 0.0
    for _ in range(a.steps):
        t, c = arm.sample()
        ts.append(t)
        cells = c
    t_step = sum(ts) / len(ts)
    value = cells / t_step
    return {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": 1e3 * t_step, "higher_is_better": True, "scaling": "weak" if a.shard == "batch" else "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": workload_config(a, world),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": arm.cores, "kind": arm.kind, "sample": arm.describe(),
                         "best_ms": 1e3 * min(ts), "worst_ms": 1e3 * max(ts), "lstm_threads": arm.lstm_threads},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }


def gpu_library_baseline(a, dev):
    """The existing GPU implementation to beat (SURVEY.md 2.1 / 8(d), BASELINE.md 3.4): the reference model moved
    `.to('cuda')` -- einsum -> cuBLAS, nn.LSTM -> cuDNN -- in fp32 and with TF32 matmuls allowed, batch 1 (its autograd state is
    ~2 K^2 N^2 C 4 B per layer and sample), same N / K / T, CUDA events, best of 3 after one warm-up."""
    import torch
    from torch import nn
    impl, kind = load_reference_impl()
    N, K, T, hid = a.nodes, a.supports, a.obs, a.hidden
    out = {"kind": kind, "batch": 1, "unit": UNIT, "what": "reference model .to('cuda'): cuBLAS einsum / cuDNN LSTM, whole model fwd+bwd"}
    model = x = y_true = G = dyn = None
    try:
        torch.manual_seed(1234)
        model = impl.MPGCN(M=2, K=K, input_dim=1, lstm_hidden_dim=hid, lstm_num_layers=1, gcn_hidden_dim=hid, gcn_num_layers=3,
                           num_nodes=N, user_bias=True, activation=nn.ReLU).to(dev)
        g = torch.Generator(device="cpu").manual_seed(5)
        x = (torch.rand(1, T, N, N, 1, generator=g) * 8).to(dev)
        y_true = (torch.rand(1, 1, N, N, 1, generator=g) * 8).to(dev)
        G = (torch.randn(K, N, N, generator=g) / N ** 0.5).to(dev)
        dyn = ((torch.randn(1, K, N, N, generator=g) / N ** 0.5).to(dev), (torch.randn(1, K, N, N, generator=g) / N ** 0.5).to(dev))
        crit = nn.MSELoss()
        old = torch.backends.cuda.matmul.allow_tf32
        for mode, tf32 in (("fp32", False), ("tf32", True)):
            torch.backends.cuda.matmul.allow_tf32 = tf32
            best = float("inf")
            for it in range(4):
                model.zero_grad(set_to_none=True)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                loss = crit(model(x_seq=x, G_list=[G, dyn]), y_true)
                loss.backward()
                e1.record()
                torch.cuda.synchronize()
                if it > 0:
                    best = min(best, e0.elapsed_time(e1))
            out[mode] = {"ms_per_step": best, "value": T * N * N / (best * 1e-3)}
        torch.backends.cuda.matmul.allow_tf32 = old
        out["peak_mem_gb"] = round(torch.cuda.max_memory_allocated(dev) / 2 ** 30, 2)
    except Exception as e:       # e.g. out of memory at cfg5: report, do not fail the bench
        out["error"] = f"{type(e).__name__}: {str(e)[:200]}"
    finally:
        model = x = y_true = G = dyn = None
        torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, model, loss, y_pred):
    """Write what a training step computed -- loss.npy, y_pred.npy and grad.<parameter>.npy -- in float32, so that two builds
    run with the same arguments (hence the same seeded inputs and weights) can be compared output for output.  A prediction
    that does not fit in what is left of DUMP_BYTES is written as y_pred_sample.npy: the elements at a fixed, seeded set of
    flat indices, the same for every run of the same shape."""
    import numpy as np
    import torch
    arrays = {"loss": loss}
    arrays.update(("grad." + n, p.grad) for n, p in model.named_parameters() if p.grad is not None)
    left = DUMP_BYTES - 4 * sum(t.numel() for t in arrays.values())
    flat = y_pred.reshape(-1)
    if 4 * flat.numel() <= left:
        arrays["y_pred"] = y_pred
    else:
        idx = np.unique(np.random.default_rng(0).integers(0, flat.numel(), left // 4))
        arrays["y_pred_sample"] = flat[torch.from_numpy(idx).to(flat.device)]
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


def run_ours(a):
    import torch
    import torch.distributed as dist
    from torch import nn

    import MPGCN as shim
    from mpgcn_b200 import _lib, dist as mdist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (the engine has no CPU path)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    mdist.init_from_env("nccl", device=dev)
    lib = _lib.load()

    N, K, T, B, hid = a.nodes, a.supports, a.obs, a.batch, a.hidden
    torch.manual_seed(1234)                                   # identical weights on every rank
    model = shim.MPGCN(M=2, K=K, input_dim=1, lstm_hidden_dim=hid, lstm_num_layers=1, gcn_hidden_dim=hid, gcn_num_layers=3,
                       num_nodes=N, user_bias=True, activation=nn.ReLU).to(dev)
    model.lstm_precision = a.precision
    for mod in model.modules():
        if isinstance(mod, shim.BDGCN):
            mod.precision = a.precision
    crit = nn.MSELoss()
    sharded = a.shard != "batch" and world > 1
    # batch shard: a different batch per rank (weak scaling); row / K shard: the SAME batch on every rank (strong scaling)
    g = torch.Generator().manual_seed(4321 + (rank if not sharded else 0))
    x_host = (torch.rand(B, T, N, N, 1, generator=g) * 8).pin_memory()
    y_host = (torch.rand(B, 1, N, N, 1, generator=g) * 8).pin_memory()
    G_static = (torch.randn(K, N, N, generator=torch.Generator().manual_seed(7)) / N ** 0.5).to(dev)
    go_host = (torch.randn(B, K, N, N, generator=g) / N ** 0.5).pin_memory()
    gd_host = (torch.randn(B, K, N, N, generator=g) / N ** 0.5).pin_memory()
    params = [p for p in model.parameters()]
    plan = None
    n_groups = 1
    if sharded:
        from mpgcn_b200 import shard as mshard
        R = a.row_ranks if (a.shard == "row" and 0 < a.row_ranks < world) else world
        assert world % R == 0 and B % (world // R) == 0, "--row-ranks must divide the number of GPUs, and the batch the number of groups"
        n_groups = world // R
        group = None
        if n_groups > 1:          # hybrid: batch over the groups, origin rows inside a group (every rank creates every group)
            groups = [dist.new_group(list(range(gi * R, (gi + 1) * R))) for gi in range(n_groups)]
            group = groups[rank // R]
            Bg, g0 = B // n_groups, (rank // R) * (B // n_groups)
            x_host, y_host, go_host, gd_host = (t[g0:g0 + Bg] for t in (x_host, y_host, go_host, gd_host))
        plan = mshard.ShardPlan(a.shard, rank % R, R, N, K, group=group)
        mshard.enable_peer_exchange(plan, dev)          # row shard: exchange inside our own kernels over NVLink peer memory, if available
        hosts = mshard.shard_host_inputs(plan, x_host, y_host, go_host, gd_host)       # this rank's slices (pinned)
        fwd = lambda x, go, gd: mshard.sharded_forward(model, plan, x, G_static, (go, gd))
    else:
        hosts = (x_host, y_host, go_host, gd_host)
        fwd = lambda x, go, gd: model(x_seq=x, G_list=[G_static, (go, gd)])

    def step(x, y, go, gd):
        """-> (loss, prediction), detached: holding them keeps no autograd graph alive"""
        for p in params:
            p.grad = None
        y_pred = fwd(x, go, gd)
        if sharded:
            loss = mshard.sharded_mse_loss(plan, y_pred, y)
            loss.backward()
            # every rank holds partial parameter gradients of its group's samples: sum inside a group, mean over the groups
            mshard.allreduce_sum_gradients(params, plan, model, over_world=n_groups > 1, scale=1.0 / n_groups)
        else:
            loss = crit(y_pred, y)
            loss.backward()
            mdist.allreduce_mean_gradients(params)      # the only exchange step of the batch shard (no-op for one rank)
        return loss.detach(), y_pred.detach()

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- resident-input arm -------------------------------------------------------------------
    x, y, go, gd = (t.to(dev) for t in hosts)
    n_warm = a.warmup if a.profile else max(3, a.warmup)
    for _ in range(n_warm):
        last = step(x, y, go, gd)         # kept like the timed steps' results, so the timed region allocates nothing new
    sync_all()
    lib.mpgcn_profile_reset()
    lib.mpgcn_profile_enable(1)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    e0.record()
    for _ in range(a.steps):
        last = step(x, y, go, gd)
    e1.record()
    sync_all()
    ms = max_over_ranks(e0.elapsed_time(e1))
    clocks = sampler.stop() if rank == 0 else None
    lib.mpgcn_profile_enable(0)
    prof = _lib.profile_read()
    ms_per_step = ms / a.steps
    samples_per_step = B if sharded else world * B
    cells_per_step = samples_per_step * T * N * N
    value = cells_per_step / (ms_per_step * 1e-3)
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, model, *last)
    del last

    # ---- end-to-end arm: host buffers in, loss out, every step -----------------------------------
    e2e = None
    if not (a.no_e2e or a.profile):
        del x, go, gd
        h2d = sum(t.numel() * t.element_size() for t in hosts)

        # Double-buffered input pipeline, as a prefetching data loader would do it: step k's inputs are copied from pinned
        # host memory on a side stream while step k-1 computes; every step still pays its own H2D copies and reads its loss
        # back (D2H) inside the timed region.
        copy_stream = torch.cuda.Stream(device=dev)

        def stage():
            with torch.cuda.stream(copy_stream):
                bufs = [t.to(dev, non_blocking=True) for t in hosts]
                ev = torch.cuda.Event()
                ev.record(copy_stream)
            return bufs, ev

        def e2e_loop(n):
            nxt = stage()
            losses = []
            for k in range(n):
                bufs, ev = nxt
                torch.cuda.current_stream().wait_event(ev)
                for b in bufs:
                    b.record_stream(torch.cuda.current_stream())
                if k + 1 < n:
                    nxt = stage()
                loss, _ = step(*bufs)
                losses.append(float(loss.item()))            # device -> host read of the loss, every step
            return losses

        e2e_loop(2)
        sync_all()
        t0 = time.perf_counter()
        e0.record()
        e2e_loop(a.steps)
        e1.record()
        sync_all()
        wall_ms = (time.perf_counter() - t0) * 1e3
        ms_e2e = max_over_ranks(max(e0.elapsed_time(e1), wall_ms)) / a.steps
        e2e = {"value": cells_per_step / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d * world, "d2h_bytes_per_step": 4 * world,
               "ms_per_step": ms_e2e}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return None

    # ---- rooflines: dominant kernel, whole layer, whole step --------------------------------------
    peaks = measured_peaks()
    big = ["FWD_A", "FWD_B", "BWD_V", "BWD_DX"]
    fl = sum(prof[t]["flops"] for t in big)
    tms = sum(prof[t]["ms"] for t in big)
    nl = sum(prof[t]["launches"] for t in big)
    achieved = fl / (tms * 1e-3) / 1e12 if tms > 0 else 0.0
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "ncu_dram_traffic.json")
    if os.path.exists(tp):
        try:
            tj = json.load(open(tp))
            traffic, traffic_src = tj.get("bytes_per_launch"), tj.get("source", "ncu --set full capture under profiles/ (not measured by this run)")
        except Exception:
            traffic = None
    roofline = {
        "bound": "tensor", "kernel": "mpgcn::tc::contract2_kernel (FWD_A/FWD_B/BWD_V/BWD_DX launches)", "achieved": achieved, "peak": peaks["tflops"],
        "unit": "TFLOP/s", "frac": achieved / peaks["tflops"], "traffic": traffic, "traffic_source": traffic_src, "peak_source": peaks["source"],
        "launches": nl, "avg_launch_ms": tms / nl if nl else None, "algorithmic_flops_per_launch": fl / nl if nl else None,
        "share_of_step": tms / ms if ms > 0 else None,
        "per_stage": {t: {"launches": v["launches"], "ms": round(v["ms"], 3),
                          "tflops": (v["flops"] / (v["ms"] * 1e-3) / 1e12 if v["ms"] > 0 and v["flops"] > 0 else None)} for t, v in prof.items()},
    }
    # whole BDGCN layer calls (every kernel + gaps, CUDA events around the C-ABI calls): algorithmic F_fb per layer and sample
    lfl = prof["LAYER_FWD"]["flops"] + prof["LAYER_BWD"]["flops"]
    lms = prof["LAYER_FWD"]["ms"] + prof["LAYER_BWD"]["ms"]
    lach = lfl / (lms * 1e-3) / 1e12 if lms > 0 else 0.0
    roofline_layer = {"bound": "tensor", "what": "whole mpgcn_bdgcn_forward + mpgcn_bdgcn_backward calls: N^3 contractions, channel mixes, dW, casts, ReLU prep",
                      "achieved": lach, "peak": peaks["tflops"], "unit": "TFLOP/s", "frac": lach / peaks["tflops"],
                      "calls": prof["LAYER_FWD"]["launches"] + prof["LAYER_BWD"]["launches"], "ms_per_step": lms / a.steps,
                      "fwd_ms_per_call": prof["LAYER_FWD"]["ms"] / max(1, prof["LAYER_FWD"]["launches"]),
                      "bwd_ms_per_call": prof["LAYER_BWD"]["ms"] / max(1, prof["LAYER_BWD"]["launches"]), "share_of_step": lms / ms if ms > 0 else None}
    f_fb = 4.0 * K * N ** 3 * (hid + hid) + 6.0 * K * K * N * N * hid * hid
    step_fl = B * 6 * f_fb / (world if sharded else 1)          # per GPU (row / K shard: the B samples are split over the ranks)
    lstm_fl = prof["LSTM_FWD"]["flops"] + prof["LSTM_BWD"]["flops"]
    sach = step_fl / (ms_per_step * 1e-3) / 1e12
    roofline_step = {"bound": "tensor", "what": "algorithmic BDGCN flops of the step (6 layers x batch x F_fwd+bwd) / step time, per GPU; the LSTM, head and "
                                                "exchange time count, their flops do not", "achieved": sach, "peak": peaks["tflops"], "unit": "TFLOP/s",
                     "frac": sach / peaks["tflops"], "with_lstm_flops": (step_fl + lstm_fl / a.steps) / (ms_per_step * 1e-3) / 1e12,
                     "lstm_ms_per_step": (prof["LSTM_FWD"]["ms"] + prof["LSTM_BWD"]["ms"]) / a.steps, "head_ms_per_step": prof["HEAD"]["ms"] / a.steps,
                     "exchange_kernels_ms_per_step": prof["EXCHANGE"]["ms"] / a.steps}
    gpu_launches = sum(v["launches"] for t, v in prof.items() if t not in _lib.REGION_TAGS)

    cpu_baseline = None
    if world == 1 and not (a.no_cpu_baseline or a.profile):
        arm = CpuArm(a)
        arm.sample()                                     # warm-up (allocator, oneDNN primitives)
        best, cells = float("inf"), 0.0
        for _ in range(2):
            t, cells = arm.sample()
            best = min(best, t)
        cpu_baseline = {"value": cells / best, "unit": UNIT, "cores": arm.cores, "kind": arm.kind, "sample": arm.describe() + "; best of 2",
                        "sample_ms": 1e3 * best, "lstm_threads": arm.lstm_threads}
    lib_baseline = None
    if world == 1 and not (a.no_gpu_baseline or a.profile):
        # in a child process: the reference's library path needs ~2 K^2 N^2 C 4 B of autograd state per layer (56 GB at the
        # headline size) and at cfg5 (N=2000: 4e6 LSTM sequences) it dies inside the libraries with an illegal memory access --
        # neither may take this process (or its GPU memory) with it
        del model
        torch.cuda.empty_cache()
        cmd = [sys.executable, os.path.abspath(__file__), "--impl", "library", "--nodes", str(N), "--supports", str(K), "--obs", str(T),
               "--hidden", str(hid), "--gpus", "1"]
        try:
            r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=dict(os.environ, CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", str(local))))
            lib_baseline = json.loads(r.stdout.strip().splitlines()[-1]) if r.returncode == 0 and r.stdout.strip() else \
                {"error": f"child exited with {r.returncode}: {r.stderr.strip().splitlines()[-1][:200] if r.stderr.strip() else ''}"}
        except Exception as e:
            lib_baseline = {"error": f"{type(e).__name__}: {str(e)[:200]}"}
        for mode in ("fp32", "tf32"):
            if isinstance(lib_baseline.get(mode), dict):
                lib_baseline[mode]["ours_over_library"] = value / world / lib_baseline[mode]["value"]

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": n_warm,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong" if a.shard != "batch" else "weak", "vs_baseline": None,
        "dtype": "f16" if a.precision != "fp32" else "f32", "data": "synthetic", "config": workload_config(a, world),
        "clocks": clocks, "e2e": e2e, "gpu_launches": gpu_launches, "roofline": roofline, "roofline_layer": roofline_layer,
        "roofline_step": roofline_step, "cpu_baseline": cpu_baseline, "gpu_library_baseline": lib_baseline,
    }
    if plan is not None:
        line["shard"] = plan.describe()
    if world > 1:
        dist.destroy_process_group()
    return line


def main():
    a = parse()
    # Libraries (NCCL's version banner, torchrun notices) may write to fd 1; the contract is ONE JSON line on stdout.
    # Route everything else to stderr and hand the real stdout only to the final print.
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = sys.stderr
    try:
        if a.impl == "library":
            import torch
            line = gpu_library_baseline(a, torch.device("cuda", 0))
        else:
            line = run_reference(a) if a.impl == "reference" else run_ours(a)
    finally:
        sys.stdout = real_stdout
    if line is not None:
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
