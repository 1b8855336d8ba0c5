#!/usr/bin/env python
"""Benchmark of the EGNN forward hot path (BASELINE.json metric: node-pairs/sec, dim=512 N=1024).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference|eager] [--dtype bf16|fp32]
                    [--dump-outputs DIR]

One "step" = one EGNN(dim=512) layer forward over one batch (B=4 graphs x N=1024 nodes, dense
all-pairs = 4,194,304 node pairs) of synthetic N(0,1) inputs with the reference's default init
(BASELINE.json configs[1], SURVEY.md section 8(d) "c2").  Multi-GPU: one process per GPU under torchrun,
every rank runs its own batch (graphs are independent units: weak scaling, no data-path collective);
with more than one rank the line also carries `row_sharded`: ONE graph (dense, N=8192) whose i-rows are
split over the ranks with one all-gather of [coors | feats] -- the strong-scaling case with a collective.

Prints ONE JSON line (rank 0).  `value` = whole-job pairs/s with inputs resident in HBM, timed
per step with CUDA events on the launch stream (L2 flushed between steps, flush not timed),
max over ranks.  `e2e` = the same through the public module API with pinned HOST tensors
(H2D + D2H inside the timed region).  `roofline` describes the fused edge kernel, timed live by
the library's own CUDA-event stage brackets (egnn_profile_*).  `cpu_baseline` = the UNMODIFIED
reference's own torch forward (baseline/_ref, installed by baseline/install_ref.py) on the host cores,
one graph of the batch at a time (BASELINE.md section 3).  `gpu_eager_baseline` = the same unmodified
reference in PyTorch eager on the same B200 (the ">= 10x" comparison of BASELINE.json's north_star).
`secondary` = the other four BASELINE configurations (c1, c3, c4 at 8 graphs per GPU, c5).

`--impl reference` times the reference's own torch CPU forward (kind "reference"; if baseline/_ref is
absent, oracle/egnn_torch_port.py -- a torch restatement with the same ATen call sequence -- and kind
"port"), all host threads, one graph of the same B=4 x N=1024 workload per step.

`--dump-outputs DIR` (with `--impl ours`) writes the (feats, coors) the module returned in the last timed step as
DIR/feats.npy and DIR/coors.npy, in float32 (exact for bf16 and fp32 outputs; 8 MiB for c2).  Module and inputs
come from fixed seeds, so two builds run with the same arguments can be compared output for output.  Under
torchrun each rank runs its own batch; rank r > 0 writes feats_rank<r>.npy and coors_rank<r>.npy.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True     # the benchmark writes nothing into the source tree, which may be read-only
REPO = os.path.dirname(os.path.abspath(__file__))
for p in (REPO, os.path.join(REPO, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

torch.set_grad_enabled(False)      # forward benchmark: no autograd state is kept

WORKLOADS = {
    # BASELINE.json configs[1]
    "c2": dict(kind="layer", cfg=dict(dim=512), B=4, N=1024, C=3, label="EGNN(dim=512) dense all-pairs B=4 N=1024"),
    # BASELINE.json configs[0] (latency-bound; for reference only)
    "c1": dict(kind="layer", cfg=dict(dim=512), B=1, N=16, C=3, label="EGNN(dim=512) dense all-pairs B=1 N=16"),
}


def peaks():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm_gbs=p["hbm_gbs"], bf16_tflops=p["bf16_tflops"], sm_max_mhz=p.get("sm_max_mhz", 1965.0),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, sm_max_mhz=1965.0, source="fallback (B200_PROFILING.md)")


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-i", str(index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1])); pw.append(float(r[2]))
            except Exception:
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return dict(sm_mhz=statistics.median(sm) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    power_w_max=max(pw) if pw else None, samples=len(sm), reasons=sorted(reasons))


# ----------------------------------------------------------------------------- workload
def build_workload(name, dtype, device, seed=0):
    """Module with the reference's default init (weights N(0,1e-3), PyTorch-default biases) and
    synthetic N(0,1) inputs (SURVEY.md section 8(d) 'Synthetic inputs')."""
    from egnn_pytorch_b200 import EGNN
    w = WORKLOADS[name]
    torch.manual_seed(seed)
    mod = EGNN(**w["cfg"]).to(dtype).to(device).eval()
    g = torch.Generator().manual_seed(seed + 1)
    feats = torch.randn(w["B"], w["N"], w["cfg"]["dim"], generator=g)
    coors = torch.randn(w["B"], w["N"], w["C"], generator=g)
    return mod, feats, coors


def work_per_pair(cfg):
    """Per-pair work of SURVEY.md section 8(d): reference-formulation FLOPs, and the split formulation's
    activation count and implemented tensor FLOPs."""
    d, e, F, m = cfg["dim"], cfg.get("edge_dim", 0), cfg.get("fourier_features", 0), cfg.get("m_dim", 16)
    E = 2 * d + 2 * F + 1 + e
    H = 2 * E
    return dict(E=E, H=H, m=m, f_ref=2 * E * H + 2 * H * m + 2 * m * 4 * m + 2 * 4 * m, act=H + m + 4 * m,
                tensor_flops=2 * ((H + 63) // 64 * 64) * 16)


def compulsory_bytes(w, es):
    """SURVEY.md section 8(d): 2*B*N*d*s (feats in+out) + 2*B*N*C*4 (coors) + weights*s."""
    d, B, N, C = w["cfg"]["dim"], w["B"], w["N"], w["C"]
    E = 2 * d + 1
    H = 2 * E
    weights = H * E + H + 16 * H + 16 + (2 * d) * (d + 16) + 2 * d + d * 2 * d + d + 64 * 16 + 64 + 64 + 1
    return 2 * B * N * d * es + 2 * B * N * C * 4 + weights * es


def equivariance_error(mod, feats, coors, dtype, device):
    """tests/test_equivariance.py:8-34 as a number: max|feats(Rx+t) - feats(x)|, max|coors(Rx+t) - (coors(x)R+t)|,
    reported absolute AND relative to the output magnitude (the c2 outputs are O(100): x_i + sum over 1024
    neighbours), plus the same figure for the unmodified reference in fp32 GPU-eager on the same inputs when
    baseline/_ref is installed."""
    g = torch.Generator().manual_seed(7)
    q, _ = torch.linalg.qr(torch.randn(3, 3, generator=g, dtype=torch.float64))
    t = torch.randn(1, 1, 3, generator=g, dtype=torch.float64)
    x = coors[:1].double()
    xr = (x @ q + t)

    def measure(fn, f):
        f2, c2 = fn(f, x.float().to(device))
        f1, c1 = fn(f, xr.float().to(device))
        ef = float((f1.double() - f2.double()).abs().max())
        ec = float((c1.double().cpu() - (c2.double().cpu() @ q + t)).abs().max())
        sf, sc = float(f2.double().abs().max()), float(c2.double().abs().max())
        return dict(feats=ef, coors=ec, feats_out_scale=sf, coors_out_scale=sc, feats_rel=ef / max(sf, 1e-30),
                    coors_rel=ec / max(sc, 1e-30))

    out = measure(mod, feats[:1].to(device, dtype))
    out["note"] = ("absolute max error; *_rel = error / max|output|.  fp32 ulp at the coordinate output scale = "
                   f"{float(np.spacing(np.float32(out['coors_out_scale']))):.2e}")
    ref = load_reference()
    if ref is not None:
        try:
            rmod = ref.EGNN(**WORKLOADS["c2"]["cfg"]).to(device).eval()
            rmod.load_state_dict({k: v.float() for k, v in mod.state_dict().items()})
            out["reference_gpu_eager_fp32"] = measure(lambda f, c: rmod(f, c), feats[:1].to(device, torch.float32))
            del rmod
            torch.cuda.empty_cache()
        except Exception as e:  # noqa: BLE001
            out["reference_gpu_eager_fp32"] = dict(error=f"{type(e).__name__}: {e}"[:160])
    return out


# ----------------------------------------------------------------------------- the reference (baseline/_ref)
def load_reference():
    """The UNMODIFIED reference package installed under baseline/_ref (baseline/install_ref.py), or None."""
    ref_dir = os.path.join(REPO, "baseline", "_ref")
    if not os.path.exists(os.path.join(ref_dir, "egnn_pytorch", "egnn_pytorch.py")):
        return None
    if ref_dir not in sys.path:
        sys.path.insert(0, ref_dir)
    try:
        import egnn_pytorch
        return egnn_pytorch
    except Exception:       # noqa: BLE001
        return None


def bench_config(world, w, path=None):
    """`config` of the JSON line -- identical in the GPU arm and in the reference arm (same workload)."""
    return dict(workload=w["label"], per_gpu_batch=w["B"], nodes=w["N"], pairs_per_step=w["B"] * w["N"] * w["N"] * world,
                init="reference default init (weights N(0, 1e-3), PyTorch-default biases), inputs N(0,1), seed 0",
                l2="GPU arm: L2 flushed between timed steps (256 MiB memset, not timed); CPU reference arm: "
                   "intermediates of one graph (21.6 GB) exceed every cache",
                parallelism=f"batch-sharded x{world} (independent graphs, no collective)")


class CpuReference:
    """The reference's own dense forward on the host cores: `EGNN(dim=512)` from baseline/_ref (kind 'reference'),
    else the torch restatement oracle/egnn_torch_port.py (kind 'port').  fp32, eval, no_grad, all host threads
    (BASELINE.md section 3); one graph of the B=4 batch per call -- B=4 at once needs > 62 GB of intermediates."""

    def __init__(self, name, seed=0):
        self.w = WORKLOADS[name]
        self.threads = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
        torch.set_num_threads(self.threads)
        torch.manual_seed(seed)
        ref = load_reference()
        if ref is not None:
            self.kind = "reference"
            self.mod = ref.EGNN(**self.w["cfg"]).eval()
            self.fn = lambda f, x: self.mod(f, x)
        else:
            from oracle.egnn_torch_port import egnn_dense_forward
            from egnn_pytorch_b200 import EGNN      # parameter container only (no forward): same init, same keys
            self.kind = "port"
            P = {k: v.detach().clone() for k, v in EGNN(**self.w["cfg"]).state_dict().items()}
            self.fn = lambda f, x: egnn_dense_forward(P, f, x)
        g = torch.Generator().manual_seed(seed + 1)
        self.feats = torch.randn(self.w["B"], self.w["N"], self.w["cfg"]["dim"], generator=g)
        self.coors = torch.randn(self.w["B"], self.w["N"], self.w["C"], generator=g)
        self.n = self.w["N"]

    def step(self, b):
        """One graph (index b mod B), the first self.n nodes of it.  Returns seconds."""
        b %= self.w["B"]
        f, x = self.feats[b:b + 1, :self.n], self.coors[b:b + 1, :self.n]
        t0 = time.perf_counter()
        with torch.no_grad():
            self.fn(f, x)
        return time.perf_counter() - t0

    def fit_budget(self, first_s, calls, budget_s):
        """If `calls` forwards at the measured pace would exceed the budget, shrink the sampled sub-graph
        (dense all-pairs cost is quadratic in the node count; pairs/s is what is reported)."""
        if first_s * calls > budget_s and self.n > 256:
            scale = (budget_s / (first_s * calls)) ** 0.5
            self.n = max(256, int(self.n * scale) // 64 * 64)

    def describe(self, calls, pairs, secs):
        full = self.n == self.w["N"]
        what = "one full graph" if full else f"the first {self.n} of {self.w['N']} nodes of one graph (dense all-pairs on the sub-graph)"
        return (f"{calls} forward(s), each {what} of the B={self.w['B']} batch ({pairs} pairs, {secs:.1f} s); "
                f"{'unmodified reference egnn_pytorch.EGNN (baseline/_ref)' if self.kind == 'reference' else 'torch restatement oracle/egnn_torch_port.py'}"
                f", torch {torch.__version__} CPU fp32, torch.set_num_threads({self.threads})")


def cpu_sample(name, budget_s=30.0):
    """cpu_baseline leg of the GPU arm: 1 warm-up + up to 3 timed forwards within ~budget_s of CPU work."""
    ref = CpuReference(name)
    first = ref.step(0)
    ref.fit_budget(first, 3, budget_s)
    if ref.n != ref.w["N"]:
        first = ref.step(0)
    reps = int(max(1, min(3, budget_s / max(first, 1e-3) - 1)))
    ts = [ref.step(i + 1) for i in range(reps)]
    t = min(ts)
    pairs = ref.n * ref.n
    return dict(value=pairs / t, unit="pairs/s", cores=ref.threads, kind=ref.kind, nproc=os.cpu_count(),
                seconds_per_graph=t, sample="min of " + ref.describe(reps, pairs * reps, sum(ts)))


def cpu_baseline_subprocess(name):
    """Run the sample in a fresh interpreter (no CUDA context, all host threads)."""
    try:
        res = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "cpu-sample", "--workload", name],
                             capture_output=True, text=True, timeout=600)
        for line in reversed(res.stdout.strip().splitlines()):
            if line.startswith("{"):
                return json.loads(line)
        err = res.stderr[-300:]
    except Exception as e:      # noqa: BLE001
        err = f"{type(e).__name__}: {e}"
    return dict(value=None, unit="pairs/s", cores=os.cpu_count(), kind="reference", sample="failed: " + err)


# ----------------------------------------------------------------------------- arms
def dist_setup(args):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local))
    return world, rank, local


def barrier_max(world, value, device):
    if world == 1:
        return value
    import torch.distributed as dist
    t = torch.tensor([value], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def time_ms(fn, iters, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def gpu_eager_baseline(name, dev, ours_ms):
    """The unmodified reference in PyTorch eager on this GPU (bf16 and fp32), same workload, same B=4 batch at once."""
    ref = load_reference()
    if ref is None:
        return dict(unavailable="baseline/_ref not installed (python baseline/install_ref.py)")
    w = WORKLOADS[name]
    pairs = w["B"] * w["N"] * w["N"]
    out = dict(kind="unmodified reference egnn_pytorch.EGNN (baseline/_ref), PyTorch eager, same GPU, inputs resident")
    for tag, dt, iters in (("bf16", torch.bfloat16, 5), ("fp32", torch.float32, 3)):
        try:
            torch.manual_seed(0)
            mod = ref.EGNN(**w["cfg"]).to(dt).to(dev).eval()
            g = torch.Generator().manual_seed(1)
            f = torch.randn(w["B"], w["N"], w["cfg"]["dim"], generator=g).to(dev, dt)
            x = torch.randn(w["B"], w["N"], w["C"], generator=g).to(dev, dt)
            torch.cuda.reset_peak_memory_stats(dev)
            ms = time_ms(lambda: mod(f, x), iters, warm=2)
            out[tag] = dict(ms_per_step=ms, pairs_per_s=pairs / ms * 1e3, peak_mem_gb=torch.cuda.max_memory_allocated(dev) / 2 ** 30,
                            speedup_of_this_repo=ms / ours_ms)
            del mod, f, x
        except Exception as e:      # noqa: BLE001
            out[tag] = dict(error=f"{type(e).__name__}: {e}"[:200])
        torch.cuda.empty_cache()
    return out


def secondary_configs(dev):
    """The other BASELINE.json configurations on one GPU: ms per forward, kernel family, all-pairs/s and edges/s
    (SURVEY.md section 8(d)), CUDA-graph replay for the launch-bound ones, and the unmodified reference in PyTorch
    eager on the same GPU when installed.  c4 = the 8 graphs one GPU holds when B=64 is sharded over 8 GPUs."""
    from egnn_pytorch_b200 import EGNN, EGNN_Network, GraphedForward
    ref = load_reference()
    g = torch.Generator().manual_seed(1)
    rows = []

    def run(name, cls, kwargs, dtype, args, kw, pairs, edges, iters, ref_iters):
        row = dict(config=name, dtype=str(dtype)[6:])
        try:
            torch.manual_seed(0)
            ours = getattr(sys.modules["egnn_pytorch_b200"], cls)(**kwargs).to(dtype).to(dev).eval()
            ms = time_ms(lambda: ours(*args, **kw), iters)
            layer = ours.layers[0][1] if hasattr(ours, "layers") else ours
            row.update(ms=ms, kernel_path=layer.last_path, all_pairs_per_s=pairs / ms * 1e3,
                       edges_per_s=None if not edges else edges / ms * 1e3)
            if ms < 2.0:
                gf = GraphedForward(ours, *args, **kw)
                row["graphed_ms"] = time_ms(lambda: gf(*args), iters)
                del gf
            if ref is not None:
                theirs = getattr(ref, cls)(**kwargs).to(dtype).to(dev).eval()
                theirs.load_state_dict(ours.state_dict())
                rms = time_ms(lambda: theirs(*args, **kw), ref_iters, warm=1)
                o, r = ours(*args, **kw), theirs(*args, **kw)
                row.update(ref_eager_ms=rms, speedup=rms / min(ms, row.get("graphed_ms", ms)),
                           max_diff_feats=float((o[0].float() - r[0].float()).abs().max()),
                           max_diff_coors=float((o[1].float() - r[1].float()).abs().max()))
                del theirs
        except Exception as e:      # noqa: BLE001
            row["error"] = f"{type(e).__name__}: {e}"[:200]
        torch.cuda.empty_cache()
        rows.append(row)

    f, x = torch.randn(1, 16, 512, generator=g).to(dev), torch.randn(1, 16, 3, generator=g).to(dev)
    run("c1 EGNN(512) B=1 N=16", "EGNN", dict(dim=512), torch.float32, (f, x), {}, 256, None, 200, 50)
    tok = torch.randint(0, 21, (1, 1024), generator=g).to(dev)
    x = torch.randn(1, 1024, 3, generator=g).to(dev)
    m = torch.ones(1, 1024, dtype=torch.bool, device=dev)
    c3 = dict(num_tokens=21, num_positions=1024, dim=32, depth=3, num_nearest_neighbors=8, coor_weights_clamp_value=2.0)
    for dt in (torch.float32, torch.bfloat16):
        run("c3 EGNN_Network depth=3 dim=32 N=1024 k=8 mask", "EGNN_Network", c3, dt, (tok, x.to(dt)), dict(mask=m),
            3 * 1024 * 1024, 3 * 1024 * 8, 100, 20)
    f = torch.randn(8, 4096, 256, generator=g).to(dev, torch.bfloat16)
    x = torch.randn(8, 4096, 3, generator=g).to(dev, torch.bfloat16)
    e = torch.randn(8, 4096, 4096, 4, generator=g, dtype=torch.bfloat16).to(dev)
    run("c4 EGNN(256, edge_dim=4) k=32 N=4096, 8 graphs (one GPU's share of B=64)", "EGNN",
        dict(dim=256, edge_dim=4, num_nearest_neighbors=32), torch.bfloat16, (f, x, e), {}, 8 * 4096 * 4096, 8 * 4096 * 32, 10, 2)
    del e, f
    n = 8192
    i = torch.arange(n, device=dev)
    adj = (i[:, None] - i[None, :]).abs() <= 1
    tok = torch.randint(0, 21, (1, n), generator=g).to(dev)
    x = torch.randn(1, n, 3, generator=g).to(dev)
    m = torch.ones(1, n, dtype=torch.bool, device=dev)
    c5 = dict(num_tokens=21, dim=32, depth=3, num_adj_degrees=3, adj_dim=8, only_sparse_neighbors=True)
    for dt in (torch.float32, torch.bfloat16):
        run("c5 EGNN_Network only_sparse num_adj_degrees=3 adj_dim=8 N=8192 chain", "EGNN_Network", c5, dt, (tok, x.to(dt)),
            dict(adj_mat=adj, mask=m), 3 * n * n, 3 * n * 9, 10, 2)
    return rows


def arm_ours(args):
    from egnn_pytorch_b200 import _native as nat
    world, rank, local = dist_setup(args)
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    lib = nat.load()
    w = WORKLOADS[args.workload]
    dtype = {"bf16": torch.bfloat16, "fp32": torch.float32}[args.dtype]
    mod, feats, coors = build_workload(args.workload, dtype, dev, seed=rank)
    f_dev, x_dev = feats.to(dev, dtype), coors.to(dev)
    pairs_rank = w["B"] * w["N"] * w["N"]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)        # > 126 MB L2

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
            torch.cuda.synchronize(dev)

    # ---- warm-up (also builds the packed-parameter cache)
    for _ in range(max(args.warmup, 3)):
        mod(f_dev, x_dev)
    path = mod.last_path
    sync_all()

    # ---- device-resident timing: K steps, CUDA events per step on the launch stream
    lib.egnn_profile_read(None, None, None, 1)
    lib.egnn_profile_enable(1)
    sampler = ClockSampler(local) if rank == 0 else None
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    sync_all()
    for a, b in evs:
        flush.zero_()                      # L2 flush between timed iterations (not timed)
        a.record()
        last = mod(f_dev, x_dev)
        b.record()
    sync_all()
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs:
        suffix = f"_rank{rank}" if rank else ""
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, t in zip(("feats", "coors"), last):
            np.save(os.path.join(args.dump_outputs, f"{name}{suffix}.npy"), t.float().cpu().numpy())
    ms_total = sum(a.elapsed_time(b) for a, b in evs)
    ms = (C.c_float * 4)(); spans = (C.c_int32 * 4)(); launches = C.c_int64()
    lib.egnn_profile_read(ms, spans, C.byref(launches), 1)
    lib.egnn_profile_enable(0)
    ms_total = barrier_max(world, ms_total, dev)
    ms_per_step = ms_total / args.steps
    value = pairs_rank * world / (ms_per_step * 1e-3)

    # ---- end-to-end: pinned host tensors through the public module API, H2D + D2H timed
    hf = feats.to(dtype).pin_memory()
    hx = coors.pin_memory()
    for _ in range(2):
        mod(hf, hx)
    sync_all()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        of, ox = mod(hf, hx)               # returns CPU tensors (synchronous D2H)
    torch.cuda.synchronize(dev)
    e2e_s = barrier_max(world, time.perf_counter() - t0, dev)
    e2e_value = pairs_rank * world / (e2e_s / args.steps)
    h2d = hf.numel() * hf.element_size() + hx.numel() * hx.element_size()
    d2h = of.numel() * of.element_size() + ox.numel() * ox.element_size()

    row_sharded = None
    if world > 1:
        row_sharded = row_sharded_probe(world, rank, dev)

    if rank != 0:
        return
    # ---- roofline of the fused edge kernel (stage 2), timed live by the library's event brackets
    pk = peaks()
    wp = work_per_pair(w["cfg"])
    pair_ms = ms[2] / max(1, spans[2])
    pair_s = pair_ms * 1e-3
    es = 2 if dtype == torch.bfloat16 else 4
    sfu_peak = 148 * 16 * pk["sm_max_mhz"] * 1e6 / 1e9                 # G activations / s  (16 MUFU/clk/SM)
    act_rate = pairs_rank * wp["act"] / pair_s / 1e9
    traffic = None
    tpath = os.path.join(REPO, "profiles", "traffic.json")
    if os.path.exists(tpath):
        traffic = json.load(open(tpath)).get(f"{args.workload}:{path}")
    tensor_tf = pairs_rank * wp["tensor_flops"] / pair_s / 1e12 if path == "bf16-tcgen05" else 0.0
    roofline = dict(
        bound="sfu", kernel="fused edge kernel (stage 2 of egnn_layer_forward)", path=path,
        achieved=act_rate, peak=sfu_peak, unit="Gsilu/s", frac=act_rate / sfu_peak, traffic=traffic,
        note="split formulation: the binding unit is the MUFU/SFU pipe (SURVEY.md section 8(d)); "
             f"peak = 148 SM x 16 MUFU/clk x {pk['sm_max_mhz']:.0f} MHz; the kernel's own instruction mix without any "
             "synchronisation tops out at 15.0 of 16 /clk/SM (profiles/r02_pipe_bench.txt)",
        launch_ms=pair_ms, stage_ms_per_step={k: ms[i] / args.steps for i, k in
                                              enumerate(["select", "node_pre", "edge", "node_post"])},
        tensor=dict(achieved=tensor_tf, peak=pk["bf16_tflops"], unit="TFLOP/s", frac=tensor_tf / pk["bf16_tflops"],
                    note="implemented bf16 MMA FLOPs only (2*Hpad*16 per pair)"),
        hbm=dict(achieved=compulsory_bytes(w, es) / pair_s / 1e9, peak=pk["hbm_gbs"], unit="GB/s",
                 frac=compulsory_bytes(w, es) / pair_s / 1e9 / pk["hbm_gbs"], algorithmic_bytes=compulsory_bytes(w, es)),
        effective_reference_tflops=pairs_rank * wp["f_ref"] / pair_s / 1e12,
        peaks=pk["source"])

    out = dict(
        metric="EGNN fwd node-pairs/sec (dim=512 N=1024)", value=value, unit="pairs/s", n_gpus=world,
        steps=args.steps, warmup=max(args.warmup, 3), ms_per_step=ms_per_step, higher_is_better=True, scaling="weak",
        vs_baseline=None, dtype="bf16" if path == "bf16-tcgen05" else "f32", data="synthetic",
        config=bench_config(world, w), kernel_path=path,
        e2e=dict(value=e2e_value, unit="pairs/s", h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h,
                 ms_per_step=e2e_s / args.steps * 1e3),
        gpu_launches=int(launches.value), clocks=clocks, roofline=roofline)
    if row_sharded is not None:
        out["row_sharded"] = row_sharded
    if not args.lean:
        out["equivariance_err"] = equivariance_error(mod, feats, coors, dtype, dev)
    if world == 1 and not args.lean:
        out["train_step"] = train_step_probe(args.workload, dev, pairs_rank)
        out["gpu_eager_baseline"] = gpu_eager_baseline(args.workload, dev, ms_per_step)
        out["secondary"] = secondary_configs(dev)
    if world == 1 and not args.no_cpu_baseline and not args.lean:
        out["cpu_baseline"] = cpu_baseline_subprocess(args.workload)
    print(json.dumps(out))


def row_sharded_probe(world, rank, dev):
    """Strong scaling WITH a collective (SURVEY.md section 8(e) row 2): one dense graph, EGNN(dim=512), N=8192, B=1,
    its i-rows split over the ranks.  Filled in by parallel.RowShardedLayer (see there); every rank takes part."""
    try:
        from egnn_pytorch_b200 import parallel
        return parallel.row_sharded_benchmark(world, rank, dev)
    except Exception as e:      # noqa: BLE001  (a probe must never break the benchmark line)
        return dict(error=f"{type(e).__name__}: {e}"[:300])


def train_step_probe(workload, dev, pairs):
    """Informational (not part of the metric): one forward + backward of the same workload through the autograd
    bridge (fp32 recompute-in-backward kernels, egnn_layer_backward), median of 3 after 2 warm-ups."""
    try:
        mod, feats, coors = build_workload(workload, torch.float32, dev, seed=0)
        mod.requires_grad_(True)
        f = feats.to(dev, torch.float32).requires_grad_(True)
        x = coors.to(dev).requires_grad_(True)
        ts = []
        with torch.enable_grad():
            for it in range(5):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                fo, xo = mod(f, x)
                (fo.sum() + xo.sum()).backward()
                b.record()
                torch.cuda.synchronize(dev)
                if it >= 2:
                    ts.append(a.elapsed_time(b))
                mod.zero_grad(set_to_none=True)
                f.grad = x.grad = None
        ms = sorted(ts)[1]
        return dict(ms_per_step=ms, pairs_per_s=pairs / ms * 1e3, dtype="f32", what="forward + backward, device-resident")
    except Exception as e:  # noqa: BLE001  (a probe must never break the benchmark line)
        return dict(error=f"{type(e).__name__}: {e}"[:200])


def arm_reference(args):
    """The reference's own torch forward on the host cores (baseline/_ref; torch restatement if absent), rank 0 only.
    Each step = one graph of the B=4 x N=1024 batch (graphs cycle through the batch), sized down to a sub-graph only
    if the whole --steps/--warmup run would not end within a few minutes on this host."""
    world, rank = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0"))
    if rank != 0:          # under torchrun the other ranks exit 0 without work (no process group needed)
        return
    w = WORKLOADS[args.workload]
    ref = CpuReference(args.workload)
    first = ref.step(0)                                  # untimed: page faults, thread pool, oneDNN/MKL init
    calls = args.warmup + args.steps
    ref.fit_budget(first, calls, budget_s=240.0)
    for i in range(args.warmup):
        ref.step(i)
    times = [ref.step(args.warmup + i) for i in range(args.steps)]
    pairs = ref.n * ref.n
    dt = sum(times)
    value = pairs * len(times) / dt
    base = dict(value=value, unit="pairs/s", cores=ref.threads, nproc=os.cpu_count(), kind=ref.kind,
                sample=ref.describe(len(times), pairs * len(times), dt))
    print(json.dumps(dict(
        impl="reference", metric="EGNN fwd node-pairs/sec (dim=512 N=1024)", value=value, unit="pairs/s",
        n_gpus=world, steps=args.steps, warmup=args.warmup, ms_per_step=dt / len(times) * 1e3, higher_is_better=True,
        scaling="weak", vs_baseline=None, dtype="f32", data="synthetic",
        config=bench_config(world, w), cpu_baseline=base,
        e2e=dict(value=value, unit="pairs/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))))


def arm_eager(args):
    """Optional stand-alone run of the `gpu_eager_baseline` leg."""
    dev = torch.device("cuda", 0)
    print(json.dumps(dict(impl="reference-gpu-eager", **gpu_eager_baseline(args.workload, dev, float("nan")))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "eager", "cpu-sample"])
    ap.add_argument("--workload", default="c2", choices=list(WORKLOADS))
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--lean", action="store_true", help="metric, e2e and roofline only (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the (feats, coors) of the last timed step as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.impl == "cpu-sample":
        print(json.dumps(cpu_sample(args.workload)))
        return
    {"ours": arm_ours, "reference": arm_reference, "eager": arm_eager}[args.impl](args)
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        import torch.distributed as dist
        if dist.is_initialized():
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
