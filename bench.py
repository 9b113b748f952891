#!/usr/bin/env python
"""bench.py -- region-timesteps/s of the ST-MGCN hot path (fwd + MSE + bwd [+ gradient all-reduce]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg3] [--impl ours|reference]

Contract (driver): prints ONE JSON line on rank 0.  ``value`` = whole-job region-timesteps/s with the inputs
resident in HBM; ``e2e`` = the same metric through the public module API with HOST (pinned) inputs, the
host->device copies and a device->host read of the loss inside the timed region; ``roofline`` = the
Chebyshev SpMM (the forward's 18 recurrence launches at cfg3) timed alone with CUDA events against the
measured HBM peak; ``cpu_baseline`` = the UNMODIFIED reference modules (``oracle/_ref``, staged by build() or
``oracle/stage_reference.py``; the oracle port if absent) on the host's cores on a bounded sample.  ``--impl reference``
times only that CPU path.  ``--dump-outputs DIR`` writes what the last timed step computed (see ``dump_outputs``).

Default workload: cfg3 = BASELINE.json configs[2] (4096 regions, 3 graphs, K=3, seq_len=12, batch 64 per
GPU, fp32) -- the configuration BASELINE.json's metric quotes the SpMM HBM figure on, and the largest fp32
single-GPU configuration; with N GPUs the per-GPU batch stays 64 (weak scaling; N=8 is cfg4's 512 windows).
A step's working set (tens of GB of LSTM tape) is far larger than the 126 MB L2, so no explicit L2 flush.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

REPO = os.path.dirname(os.path.abspath(__file__))
for _p in (REPO, os.path.join(REPO, "st-mgcn_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

METRIC = "region-timesteps/sec (fwd+bwd)"
UNIT = "region-timesteps/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="cfg3")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=None, help="override the per-GPU batch")
    ap.add_argument("--arith", default="auto", choices=["auto", "fp32", "bf16"],
                    help="tensor-core arithmetic of the shared LSTM: fp32 = 3-pass bf16 hi/lo planes (fp32-grade, 1e-4 parity), "
                         "bf16 = single pass on one bf16 plane; auto = what BASELINE.json quotes the workload in")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--cuda-graph", action="store_true",
                    help="replay the step from a captured CUDA graph (stmgcn_b200.graphs.GraphedStep); measured gain "
                         "at cfg3 is ~1 %% -- the step is GPU-bound, not launch-bound -- so eager is the default")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the output, loss and parameter gradients of the last timed step "
                         "as DIR/<name>.npy (written by rank 0: its own output and loss, the all-reduced gradients)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return args


# ---------------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------------
def peaks():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            return json.load(fh), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "sm_max_mhz": 1965.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int = 0):
        self.tmp = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.proc = None
        self.gpu_index = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu_index)], stdout=self.tmp,
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.tmp.flush()
        self.tmp.seek(0)
        sm, reasons, sm_max = [], set(), None
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.tmp.read().splitlines():
            f = [v.strip() for v in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                sm_max = float(f[2])
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        try:
            os.unlink(self.tmp.name)
        except OSError:
            pass
        if sm:
            sm.sort()
            out.update(sm_mhz=sm[len(sm) // 2], sm_max_mhz=sm_max, reasons=sorted(reasons), samples=len(sm))
        return out


DUMP_BUDGET_BYTES = 64 << 20


def dump_outputs(path, out, loss, model):
    """Write what a step hands back to its caller -- the model output, the MSE loss and every parameter gradient -- as
    float32 ``path/out.npy``, ``path/loss.npy`` and ``path/grad.<parameter name>.npy``.  The inputs are a pure function of
    the arguments, so two builds can be compared file by file.  An output too large for the 64 MB budget is written as
    the fixed sample ``out.reshape(-1)[::stride]``.  With several GPUs, rank 0 calls this: ``out`` and ``loss`` are its
    own shard of the batch, the gradients are the all-reduced means every rank holds."""
    import numpy as np
    arrays = {"loss": loss.detach().float().cpu().numpy()}
    arrays.update({"grad." + k: p.grad.detach().float().cpu().numpy() for k, p in model.named_parameters()})
    o = out.detach().float().cpu().numpy()
    room = DUMP_BUDGET_BYTES - sum(a.nbytes for a in arrays.values())
    if room <= 0:
        raise RuntimeError(f"--dump-outputs: the gradients alone exceed {DUMP_BUDGET_BYTES} bytes")
    if o.nbytes > room:
        o = o.reshape(-1)[::-(-o.nbytes // room)]
    arrays["out"] = o
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def spmm_algorithmic_bytes(n, nnz, f_total, k_order, elem=4):
    """SURVEY.md section 8(d): per GCN call K*CSR + N*F*e*(3K-1)."""
    csr = nnz * 8 + (n + 1) * 4
    return k_order * csr + n * f_total * elem * (3 * k_order - 1)


# ---------------------------------------------------------------------------------------------------
# reference arm: the oracle port (dense supports + nn.LSTM, the reference's algorithm) on host cores
# ---------------------------------------------------------------------------------------------------
REF_DIR = os.path.join(REPO, "oracle", "_ref")


def _reference_modules():
    """The UNMODIFIED reference's ``GCN`` / ``STMGCN`` modules from ``oracle/_ref`` (staged by
    ``oracle/stage_reference.py``), imported under private names so they can never shadow the repo's drop-in modules.
    Returns None when the directory was not staged (then the oracle port is timed instead)."""
    if not os.path.exists(os.path.join(REF_DIR, "STMGCN.py")):
        return None
    import importlib.util

    def load(name):
        spec = importlib.util.spec_from_file_location(f"_stmgcn_ref_{name}", os.path.join(REF_DIR, name + ".py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        return mod

    ref_gcn = load("GCN")
    saved = sys.modules.get("GCN")
    sys.modules["GCN"] = ref_gcn                 # STMGCN.py:4 does `from GCN import GCN`: must resolve to the reference's
    try:
        ref_stmgcn = load("STMGCN")
    finally:
        if saved is not None:
            sys.modules["GCN"] = saved
        else:
            sys.modules.pop("GCN", None)
    return ref_gcn, ref_stmgcn


def cpu_reference_run(w, steps, warmup, sample_batch=None, log=None, step_budget_s=6.0):
    """Time the reference's CPU implementation of the path on the host cores.

    kind "reference": the unmodified reference modules from ``oracle/_ref`` -- ``Adj_Preprocessor.process`` (dense
    supports, GCN.py:57-97), ``ST_MGCN.forward`` (STMGCN.py:100-119), ``nn.MSELoss``, ``backward`` -- exactly the step of
    ``Model_Trainer.py:35-41`` without the optimizer.  kind "port": the oracle's dense restatement (same algorithm, same
    torch ops) when ``oracle/_ref`` is absent.

    Thread count: "all the host threads it can use" is calibrated, not assumed -- on the GPU boxes os.cpu_count()
    reports 128 logical CPUs but running 128 intra-op threads is ~50x SLOWER than 16-32 (measured: 64 s vs 1.1 s for a
    2-window step), so candidates are tried smallest-first on a 1-window step and the fastest is used; `cores` in the
    result is the number of threads actually used.  The sample batch is then sized to ~step_budget_s per step."""
    import torch
    from torch import nn
    from stmgcn_b200 import synth
    ncpu = os.cpu_count() or 1
    torch.set_num_threads(min(ncpu, 16))
    ref = _reference_modules()
    t0 = time.time()
    adjs = synth.make_adjacency_list(w)
    if ref is not None:
        ref_gcn, ref_stmgcn = ref
        kind = "reference"
        pre = ref_gcn.Adj_Preprocessor("chebyshev", w.cheb_order)
        import contextlib
        import io
        with contextlib.redirect_stdout(io.StringIO()):        # GCN.py:119-121 prints its lambda_max fallback notice
            sups = [pre.process(a) for a in adjs]              # GCN.py:57-97 (dense polynomials, once)
        torch.manual_seed(0)
        model = ref_stmgcn.ST_MGCN(**synth.model_kwargs(w))
        crit = nn.MSELoss(reduction="mean")

        def one_step(x, y):
            t1 = time.time()
            model.zero_grad(set_to_none=True)
            loss = crit(model(obs_seq=x, sta_adj_list=sups), y)          # Model_Trainer.py:35,38
            loss.backward()                                               # Model_Trainer.py:41
            return time.time() - t1
    else:
        kind = "port"
        sys.path.insert(0, os.path.join(REPO, "oracle"))
        import stmgcn_oracle as O
        sups = [O.chebyshev_supports_dense(a, w.cheb_order) for a in adjs]
        params = O.init_params(w.n_graphs, w.seq_len, w.input_dim, w.lstm_hidden, w.lstm_layers, w.gcn_hidden,
                               w.n_supports, seed=0)

        def one_step(x, y):
            t1 = time.time()
            O.dense_loss_and_grads(params, x, y, sups, relu=True, lstm=O.lstm_library)
            return time.time() - t1
    prep_s = time.time() - t0

    x1, y1 = synth.make_inputs(w, seed=0, batch=1)
    one_step(x1, y1)                                           # warm the allocator / oneDNN primitives
    cands = sorted({c for c in (4, 8, 16, 32, 64, ncpu // 2, ncpu) if 1 <= c <= ncpu})
    best_t, best_c = None, cands[0]
    for c in cands:
        torch.set_num_threads(c)
        dt = min(one_step(x1, y1), one_step(x1, y1))
        if log:
            log(f"[cpu] calibrate threads={c}: {dt:.2f}s")
        if best_t is None or dt < best_t:
            best_t, best_c = dt, c
        elif dt > 1.5 * best_t:
            break                                              # oversubscribed from here on
    torch.set_num_threads(best_c)
    if sample_batch is None:
        sample_batch = max(1, min(w.batch, 16, int(step_budget_s / max(best_t, 1e-3))))
    x, y = synth.make_inputs(w, seed=0, batch=sample_batch)
    times = []
    for i in range(warmup + steps):
        dt = one_step(x, y)
        if i >= warmup:
            times.append(dt)
        if log:
            log(f"[cpu] step {i} {dt:.2f}s")
    mean = sum(times) / len(times)
    value = sample_batch * w.n_regions * w.seq_len / mean
    try:
        model_name = [l.split(":")[1].strip() for l in open("/proc/cpuinfo") if l.startswith("model name")][0]
    except Exception:
        model_name = "unknown"
    what = ("the UNMODIFIED reference modules (oracle/_ref: Adj_Preprocessor.process dense supports, ST_MGCN.forward, "
            "MSELoss, backward)" if kind == "reference" else
            "the oracle port (dense supports + nn.LSTM, as the reference executes; oracle/_ref not staged)")
    return dict(value=value, unit=UNIT, cores=best_c, kind=kind,
                sample=f"{w.name} shapes with batch {sample_batch} (of {w.batch}), {steps} timed step(s) after "
                       f"{warmup} warm-up, fwd+MSE+bwd through {what}, "
                       f"{best_c} intra-op threads (calibrated; {ncpu} logical CPUs visible); support preprocessing "
                       f"{prep_s:.1f}s excluded; cpu '{model_name}'"), mean


def run_reference(args, w):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    total = args.steps + args.warmup
    cb, mean = cpu_reference_run(w, args.steps, args.warmup, None, step_budget_s=max(1.5, min(8.0, 150.0 / total)))
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": mean * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(w, 1, w.batch), "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def workload_config(w, world, per_gpu_batch, arith="fp32"):
    return {"workload": f"{w.name}: {w.n_regions} regions, {w.n_graphs} graphs, Chebyshev K={w.cheb_order}, "
                        f"seq_len={w.seq_len}, batch={per_gpu_batch}/GPU x {world} GPU(s), {arith}, H={w.lstm_hidden} "
                        f"L={w.lstm_layers} G={w.gcn_hidden} C={w.input_dim}, graph density {w.density}",
            "global_batch": per_gpu_batch * world, "parallelism": f"dp{world}",
            "l2": "per-step working set (GBs of activations) exceeds the 126 MB L2; no explicit flush",
            "step": "forward + MSELoss + backward (+ one gradient all-reduce when world > 1); optimizer excluded",
            "cuda_graph": None}


# ---------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------
def run_ours(args, w):
    import torch
    import torch.distributed as dist
    from torch import nn
    import GCN
    import STMGCN
    from stmgcn_b200 import _lib, dp, graphs, ops, synth
    from stmgcn_b200.graph import supports_from_dense

    arith = args.arith if args.arith != "auto" else ("bf16" if w.dtype == "bf16" else "fp32")
    ops.set_lstm_planes(1 if arith == "bf16" else 2)
    rank, world, local_rank = dp.init_from_env()
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py --impl ours needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    b = args.batch or w.batch

    # supports: sparse-native construction (no dense N^3 preprocessing); replicated on every rank
    pre = GCN.Adj_Preprocessor("chebyshev", w.cheb_order)
    sups = [pre.process_sparse(a).to(dev) for a in synth.make_adjacency_list(w)]
    torch.manual_seed(0)
    model = STMGCN.ST_MGCN(**synth.model_kwargs(w)).to(dev)
    bucket = dp.GradBucket(model)
    crit = nn.MSELoss(reduction="mean")
    x_h, y_h = synth.make_inputs(w, seed=100 + rank, batch=b)          # each rank: its own shard of windows
    x_h, y_h = x_h.pin_memory(), y_h.pin_memory()
    x_d, y_d = x_h.to(dev), y_h.to(dev)

    use_graph = args.cuda_graph
    launches_per_step = None
    last = {}                              # output and loss of the latest step (--dump-outputs); detached, so the
                                           # step's autograd graph and LSTM tape are freed as before
    if use_graph:
        # one eager step to count this library's launches, then capture fwd + loss + bwd (+ all-reduce) once
        l0 = _lib.launch_count()
        bucket.zero_()
        crit(model(obs_seq=x_d, sta_adj_list=sups), y_d).backward()
        torch.cuda.synchronize()
        launches_per_step = _lib.launch_count() - l0
        gstep = graphs.GraphedStep(model, crit, x_d, y_d, sups, bucket=bucket, all_reduce=False)

        def step(x, y):
            loss = gstep(x, y)
            bucket.all_reduce_mean_()          # the one collective of the step stays outside the graph (NCCL, eager)
            last.update(out=gstep.out, loss=loss)
            return loss
    else:
        def step(x, y):
            bucket.zero_()
            out = model(obs_seq=x, sta_adj_list=sups)
            loss = crit(out, y)
            loss.backward()
            bucket.all_reduce_mean_()
            last.update(out=out.detach(), loss=loss.detach())
            return loss

    ms_step_local = [0.0]                  # this rank's own device time per step of the last timed() call

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        ms_step_local[0] = float(ms.item()) / steps
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # ---- device-resident inputs ---------------------------------------------------------------------
    for _ in range(max(args.warmup, 3)):
        step(x_d, y_d)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    l0 = _lib.launch_count()
    ms_total = timed(lambda: step(x_d, y_d), args.steps)
    launches = (_lib.launch_count() - l0) // args.steps if launches_per_step is None else launches_per_step
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last["out"], last["loss"], model)
    ms_step = ms_total / args.steps
    units = b * world * w.n_regions * w.seq_len
    value = units / (ms_step * 1e-3)

    # ---- correctness gate: the loss of the timed step against the fp64 oracle's value for these exact inputs ----------
    # (tests/golden/bench_loss.json, written by oracle/make_bench_loss.py in the build container: SparseOracle.forward
    # on the same seeded model and inputs).  A kernel that is fast but wrong at THIS size cannot print a number.
    loss_val = float(step(x_d, y_d).item())
    loss_check = {"loss": loss_val, "reference": None, "rel_err": None, "tolerance": 1e-4, "ok": None,
                  "source": "tests/golden/bench_loss.json (fp64 sparse oracle, oracle/make_bench_loss.py)"}
    table_path = os.path.join(REPO, "tests", "golden", "bench_loss.json")
    ok_flag = 1.0
    if os.path.exists(table_path):
        with open(table_path) as fh:
            table = json.load(fh)
        ref_loss = table.get(f"{w.name}/batch{b}/rank{rank}")
        if ref_loss is not None:
            rel = abs(loss_val - ref_loss) / max(abs(ref_loss), 1e-30)
            tol = 1e-4 if ops.lstm_planes() == 2 else 2e-2        # fp32-grade arithmetic / single-pass bf16 (SURVEY 8(d))
            loss_check.update(reference=ref_loss, rel_err=rel, tolerance=tol, ok=bool(rel <= tol))
            ok_flag = 1.0 if rel <= tol else 0.0
    okt = torch.tensor([ok_flag], device=dev)
    per_rank_ms = torch.zeros(world, device=dev)
    per_rank_ms[rank] = ms_step_local[0]
    if world > 1:
        dist.all_reduce(okt, op=dist.ReduceOp.MIN)
        dist.all_reduce(per_rank_ms, op=dist.ReduceOp.SUM)
    if float(okt.item()) < 1.0:
        raise RuntimeError(f"bench.py: loss check failed on some rank (rank {rank}: {loss_check}); refusing to report a number")
    # the collective alone (CUDA events around the all-reduce of the flat gradient bucket, mean of 20)
    allreduce_us = None
    if world > 1:
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        dist.barrier()
        e0.record()
        for _ in range(20):
            bucket.all_reduce_mean_()
        e1.record()
        torch.cuda.synchronize()
        allreduce_us = e0.elapsed_time(e1) / 20 * 1e3

    # ---- end to end: host (pinned) inputs through the public module API ------------------------------------
    e2e = None
    if not args.no_e2e:
        x_buf, y_buf = torch.empty_like(x_d), torch.empty_like(y_d)

        def e2e_step():
            if use_graph:                                       # pinned host -> the graph's static input buffers
                loss = step(x_h, y_h)
            else:
                x_buf.copy_(x_h, non_blocking=True)
                y_buf.copy_(y_h, non_blocking=True)
                loss = step(x_buf, y_buf)
            return loss.item()                                  # device -> host read of the step's result

        for _ in range(2):
            e2e_step()
        ms_e2e = timed(e2e_step, args.steps) / args.steps
        e2e = {"value": units / (ms_e2e * 1e-3), "unit": UNIT,
               "h2d_bytes_per_step": (x_h.numel() + y_h.numel()) * 4, "d2h_bytes_per_step": 4,
               "ms_per_step": ms_e2e}

    # ---- roofline of the dominant memory-bound kernel: the Chebyshev SpMM (forward's recurrence launches) ----
    roofline = None
    if rank == 0:
        pk, pk_kind = peaks()
        ssets = [supports_from_dense(s) for s in sups]
        n, k_ord = w.n_regions, w.cheb_order
        stacks = [(torch.randn(w.n_supports, n, b, w.seq_len, device=dev),
                   torch.randn(w.n_supports, n, b, w.lstm_hidden, device=dev)) for _ in ssets]

        def spmm_forward_all():
            for sset, (st, ss) in zip(ssets, stacks):
                ops.cheb_stack_(sset, st)
                ops.cheb_stack_(sset, ss)

        def spmm_dominant():                    # the dominant launch type: spatial recurrence step k >= 2, all graphs
            for sset, (st, ss) in zip(ssets, stacks):
                g = sset.graphs[0]
                for k in range(2, w.n_supports):
                    ops.spmm_step(g, False, 2.0, ss[k - 1], -1.0, ss[k - 2], 0.0, None, ss[k])

        def time_local(fn, reps):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / reps

        for _ in range(3):
            spmm_forward_all()
        reps = 5
        l1 = _lib.launch_count()
        ms_spmm = time_local(spmm_forward_all, reps)
        n_launch = (_lib.launch_count() - l1) // reps
        alg = sum(spmm_algorithmic_bytes(n, s.graphs[0].nnz if s.graphs else 0, b * f, k_ord)
                  for s in ssets for f in (w.seq_len, w.lstm_hidden))
        l2 = _lib.launch_count()
        ms_dom = time_local(spmm_dominant, reps) if k_ord >= 2 else None
        n_dom = (_lib.launch_count() - l2) // reps
        f_sp = b * w.lstm_hidden
        alg_dom = [s.graphs[0].nnz * 8 + (n + 1) * 4 + n * f_sp * 4 * 3 for s in ssets]       # r_k = 2 reads + 1 write
        if ms_dom:
            us_launch = ms_dom * 1e3 / max(n_dom, 1)
            achieved = (sum(alg_dom) * (k_ord - 1)) / (ms_dom * 1e-3) / 1e9
        else:
            us_launch, achieved = ms_spmm * 1e3 / max(n_launch, 1), alg / (ms_spmm * 1e-3) / 1e9
        # DRAM bytes per launch of this launch type: read from the committed summary of this round's `ncu --set full`
        # capture of exactly this launch (tools/ncu_spmm.sh -> tools/ncu_summary.py -> profiles/r2_spmm_ncu.json); only
        # valid for the shape it was captured on (cfg3, batch 64)
        traffic, traffic_src = None, None
        tpath = os.path.join(REPO, "profiles", "r2_spmm_ncu.json")
        if w.name == "cfg3" and b == 64 and os.path.exists(tpath):
            with open(tpath) as fh:
                tj = json.load(fh)
            try:
                mb = float(tj["dram__bytes_read.sum"]) + float(tj["dram__bytes_write.sum"])
                traffic = mb * 1e6
                traffic_src = ("profiles/r2_spmm_ncu.json: dram__bytes_read.sum + dram__bytes_write.sum of one launch "
                               f"({tj['dram__bytes_read.sum']} + {tj['dram__bytes_write.sum']} MB), ncu --set full")
            except (KeyError, ValueError):
                pass
        roofline = {"bound": "hbm", "kernel": "spmm_row_gather_kernel<4> (Chebyshev recurrence step, spatial, k>=2)",
                    "achieved": achieved, "peak": pk["hbm_gbs"], "peak_kind": f"{pk_kind} (MEASURED_PEAKS.json hbm_gbs)",
                    "unit": "GB/s", "frac": achieved / pk["hbm_gbs"], "traffic": traffic, "traffic_source": traffic_src,
                    "gather_ceiling": {"measured_gather_GBps": 17900, "source": "profiles/r2_gather_probe.log (tools/gather_probe.cu: "
                                       "512-byte row-segment gathers through L2/L1, same N / F / degree)",
                                       "note": "the launch gathers nnz*F*4 B = 2.87 GB against 0.2 GB of algorithmic HBM bytes; "
                                               "at the measured gather rate that alone is 160 us"},
                    "algorithmic_bytes_per_launch": sum(alg_dom) / len(alg_dom), "avg_us_per_launch": us_launch,
                    "launches_timed": n_dom,
                    "forward_all": {"algorithmic_bytes": alg, "launches": n_launch, "ms": ms_spmm,
                                    "achieved_gbs": alg / (ms_spmm * 1e-3) / 1e9,
                                    "frac": alg / (ms_spmm * 1e-3) / 1e9 / pk["hbm_gbs"]},
                    "scope": f"per launch: Y = 2 L X - Z on (N={n}, F={f_sp}) fp32, bytes = nnz*8 + (N+1)*4 + 3*N*F*4 "
                             f"(SURVEY.md 8(d)); timed alone with CUDA events over {n_dom} launches ({w.n_graphs} graphs x "
                             f"k=2..{k_ord}); forward_all = all {n_launch} recurrence launches of one forward "
                             f"(temporal F={b * w.seq_len} + spatial F={f_sp}). The kernel is bound by its L2 gather volume "
                             f"nnz*F*4 B per launch (see DESIGN.md section 3), not by HBM"}
        del stacks

    # ---- the kernels that dominate the step by time: the shared LSTM of one graph branch, timed alone --------------
    roofline_lstm = None
    if rank == 0 and w.lstm_hidden == 64 and w.input_dim == 1:
        rnn = model.rnn_list[0]
        lyr, hid, t_len = w.lstm_layers, w.lstm_hidden, w.seq_len
        rows = w.n_regions * b
        xo = torch.randn(w.n_regions, b, t_len, 1, device=dev)
        s_gate = torch.rand(b, t_len, device=dev)
        wts = [p_.detach().clone().requires_grad_(True) for p_ in rnn._lstm_weights()]
        d_top = torch.randn(w.n_regions, b, hid, device=dev)

        def lstm_once():
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            torch.cuda.synchronize()
            l_a = _lib.launch_count()
            ev[0].record()
            h_top, _, _ = ops.SharedLSTM.apply(xo, s_gate, None, None, lyr, hid, False, *wts)
            ev[1].record()
            l_b = _lib.launch_count()
            h_top.backward(d_top)
            ev[2].record()
            torch.cuda.synchronize()
            return ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]), l_b - l_a, _lib.launch_count() - l_b

        for _ in range(2):
            lstm_once()
        runs = [lstm_once() for _ in range(3)]
        ms_f = sum(r[0] for r in runs) / len(runs)
        ms_b = sum(r[1] for r in runs) / len(runs)
        u = rows * hid * 4                                    # one (rows, H) array at 4 bytes per value (fp32, or bf16 hi + lo)
        planes = ops.lstm_planes()
        hu = planes / 2.0                                     # a hidden-state array: 2 bf16 planes = 1 unit, 1 plane = 0.5
        fwd_u = bwd_u = 0
        for l in range(lyr):
            for t in range(t_len):
                # forward: h_below planes, h_{t-1} planes + c_{t-1} | h planes, c
                fwd_u += (hu if l > 0 else 0) + ((hu + 1) if t > 0 else 0) + hu + 1
                # fused backward: A planes (h_below, h_{t-1}), c_{t-1}, dh_in, dh_rec + dc in | dc, dh_rec, dx_below out
                dh_in = 1 if l < lyr - 1 else (1 if t == t_len - 1 else 0)
                bwd_u += (hu if l > 0 else 0) + ((hu + 1) if t > 0 else 0) + dh_in + (2 if t < t_len - 1 else 0)
                bwd_u += 1 + (1 if t > 0 else 0) + (1 if l > 0 else 0)
        fwd_b = fwd_u * u + rows * t_len * 4
        bwd_b = bwd_u * u + rows * t_len * 4
        roofline_lstm = {
            "scope": f"shared {lyr}-layer LSTM of ONE graph branch (rows = N*B = {rows}, H = {hid}, T = {t_len}), timed alone with "
                     "CUDA events, mean of 3 after 2 warm-ups; algorithmic bytes count every (rows, H) array a layer-step must "
                     f"read or write once at 4 B per value ({planes} bf16 plane(s) per hidden state): forward h_below, h/c_(t-1) in, "
                     "h, c out; fused backward (gate recompute + BPTT pointwise + data and weight gradients in one kernel): "
                     "h_below, h/c_(t-1), dh_in, dh_rec, dc in, dc, dh_rec, dx_below out; weights are resident / L2",
            "bound": "hbm", "peak": pk["hbm_gbs"], "unit": "GB/s", "planes": planes,
            "forward": {"kernel": "lstm16_fwd_kernel", "launches": runs[0][2], "ms": ms_f, "algorithmic_bytes": fwd_b,
                        "achieved": fwd_b / (ms_f * 1e-3) / 1e9, "frac": fwd_b / (ms_f * 1e-3) / 1e9 / pk["hbm_gbs"]},
            "backward": {"kernel": "lstm16_bwd_kernel (+ lstm16_wgrad_reduce_kernel)", "launches": runs[0][3], "ms": ms_b,
                         "algorithmic_bytes": bwd_b, "achieved": bwd_b / (ms_b * 1e-3) / 1e9,
                         "frac": bwd_b / (ms_b * 1e-3) / 1e9 / pk["hbm_gbs"]}}
        del xo, s_gate, wts, d_top

    # ---- CPU baseline beside it (rank 0, N=1 only; bounded sample) ------------------------------------------
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_baseline, _ = cpu_reference_run(w, 2, 1, None, step_budget_s=6.0)

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None,
                "dtype": "f32" if ops.lstm_planes() == 2 else "bf16", "data": "synthetic",
                "config": dict(workload_config(w, world, b, arith), cuda_graph=use_graph,
                               arithmetic=("fp32 state and accumulation; tensor-core products as 3-pass bf16 hi/lo planes "
                                           "(3xBF16, fp32-grade)" if ops.lstm_planes() == 2 else
                                           "fp32 state and accumulation; single-pass bf16 tensor-core products")),
                "clocks": clocks,
                "gpu_launches": int(launches), "loss_check": loss_check,
                "per_rank_ms_per_step": [float(v) for v in per_rank_ms.tolist()], "allreduce_us": allreduce_us,
                "e2e": e2e, "roofline": roofline, "roofline_lstm": roofline_lstm, "cpu_baseline": cpu_baseline}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse_args()
    from stmgcn_b200 import synth
    w = synth.WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, w)
    else:
        run_ours(args, w)


if __name__ == "__main__":
    main()
