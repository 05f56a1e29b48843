#!/usr/bin/env python
"""Benchmark of the DSTD-GCN training hot path on B200 (metric of BASELINE.json: train samples/s at the H3.6M shape).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--workload h36m|cmu|3dpw] [--impl reference]

One "step" = one iteration of the reference engine loop (engine/prediction.py:215-294) on one batch of synthetic
poses: forward on the batch, forward on the time-reversed batch (``inverse: True`` in every shipped config), MPJPE
losses, one backward, gradient all-reduce (N > 1), Adam.  Under torchrun every rank runs its own shard
(``--batch`` samples per GPU, weak scaling) and rank 0 prints ONE JSON line.

``--impl reference`` times the reference's own CPU implementation of the same step -- the UNMODIFIED reference
(`baseline/_ref`, vendored by ``__graft_entry__.build()``; ``PredictionEngine.train`` around ``DSTDGCN``) on all host
threads, same workload, batch and dropout as the GPU arm, on a bounded sample; it never touches the GPU library.  The GPU
arm additionally reports ``gpu_eager_baseline``: the same reference loop with the model on the B200 (torch eager).

``--dump-outputs DIR`` writes what the last timed step computed to ``DIR/<name>.npy`` (train: the loss, the model state
after the update and the step's gradients; infer: the predictions).  Inputs and weights are seeded, so two builds run
with the same arguments can be compared array for array.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (layout, V, T_in, T_out, dropout)  -- configs/dstdgcn/*.yaml of the reference
    "h36m": ("h36m", 22, 10, 25, 0.1),
    "cmu": ("cmu", 25, 10, 25, 0.1),
    "3dpw": ("3dpw", 23, 10, 30, 0.0),
    "stress": ("h36m", 22, 50, 75, 0.1),     # BASELINE.json configs[4]: 50 -> 75 frames, 256 hidden channels
}
N_LAYERS = 5
FEATURES = {"stress": 256}
DEFAULT_BATCH = {"stress": 32}


def feat(workload):
    return FEATURES.get(workload, 64)


C_FEAT = 64


def dominant_call_roofline(batch, v, t, peak, c=C_FEAT, reps=5):
    """Live CUDA-event timing of the dominant ABI call of the step, `dstd_gc_backward` of an encoder's spatial unit
    (aggmix_bwd + dynadj_bwd + mproj_bwd: ~45 % of the step), against its own algorithmic bytes: x and the output
    gradient are read once, the input gradient is written once (3 activation tiles per sample, fp32)."""
    import torch
    from dstd_gcn_b200 import _lib
    dev, be = torch.device("cuda"), _lib.backend()
    g = torch.Generator().manual_seed(1)
    r = lambda *s, sc=0.2: (torch.randn(*s, generator=g) * sc).to(dev)
    brs = [dict(w_m1=r(2, c, 1, 1), b_m1=r(2), w_m2=r(2, c, 1, 1), b_m2=r(2), w_rm=r(t, 2 * t, 1, 1), b_rm=r(t),
                w_f=r(c, c, 1, 1), b_f=r(c), adj=(torch.rand(v, v, generator=g) > 0.7).float().to(dev), adj_w=r(v, v),
                adj_r=r(v, v)) for _ in range(2)]
    x, go, alpha = r(batch, c, t, v, sc=1.0), r(batch, c, t, v, sc=1.0), torch.tensor([0.3], device=dev)
    out, m, pd, xa = be.gc_forward(x, alpha, brs, None, False)
    xa = xa if xa.numel() else None
    be.gc_backward(x, go, alpha, brs, m, pd, xa, False)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        be.gc_backward(x, go, alpha, brs, m, pd, xa, False)
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / reps
    nbytes = 3 * batch * c * t * v * 4
    ach = nbytes / (us * 1e-6) / 1e9
    return {"call": "dstd_gc_backward, encoder spatial unit (2 branches)", "avg_us": us,
            "algorithmic_bytes_per_call": nbytes, "achieved": ach, "unit": "GB/s", "frac": ach / peak,
            "calls_per_step": 2 * N_LAYERS}


def algorithmic_bytes_per_pass(v, t, c=64, layers=N_LAYERS):
    """SURVEY.md section 8(d): one HBM round trip per DSTDGCB layer, fp32, forward + backward of one model pass."""
    chans = [(6, c)] + [(c, c)] * layers + [(c, 3)]
    fwd = 4 * t * v * sum(ci + co for ci, co in chans)
    bwd = 4 * t * v * sum(2 * ci + co for ci, co in chans)
    return fwd + bwd


def synthetic_batch(n, t, v, t_in, seed, scale_pose=1.0, scale_step=0.05):
    """Seeded synthetic poses with the dataset's padding (dataset/h36m.py:53-57): a random walk per coordinate around a
    per-joint offset; model-input frames t_in.. repeat the last observed frame; the inverse input is the time-reversed
    window padded the same way.  Returns raw [N,T,3V] (inputs, inputs_inv, targets) on the CPU."""
    import torch
    g = torch.Generator().manual_seed(seed)
    base = torch.randn(n, 1, v * 3, generator=g) * scale_pose
    walk = torch.cumsum(torch.randn(n, t, v * 3, generator=g) * scale_step, dim=1)
    seq = base + walk
    inputs = seq.clone()
    inputs[:, t_in:] = seq[:, t_in - 1:t_in]
    rev = torch.flip(seq, dims=[1])
    inputs_inv = rev.clone()
    inputs_inv[:, t_in:] = rev[:, t_in - 1:t_in]
    return inputs.contiguous(), inputs_inv.contiguous(), seq.contiguous()


def perturb(model):
    """Make the dynamic-adjacency path live (alpha, W_s, R_t are zero at init; SURVEY.md appendix D)."""
    import torch
    with torch.no_grad():
        for k, p in model.named_parameters():
            leaf = k.split(".")[-1]
            if leaf in ("alpha_sm", "alpha_tm"):
                p.fill_(0.1)
            elif leaf == "W_s":
                p.fill_(0.05)
            elif leaf == "R_t":
                p.fill_(0.01)
    return model


DUMP_LIMIT = 64_000_000          # bytes


def dump_outputs(out_dir, arrays, limit=DUMP_LIMIT):
    """Write each numpy array of `arrays` to ``out_dir/<name>.npy``: float64 stays float64, integer counters become
    float64, everything else float32.  If the files would exceed `limit` bytes in all, the largest arrays keep a fixed,
    seeded sample of their elements (flattened, in index order), so the same inputs always write the same elements."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    items = sorted(arrays.items(), key=lambda kv: kv[1].size)
    budget = limit
    for i, (name, a) in enumerate(items):
        a = np.asarray(a, dtype=np.float64 if a.dtype == np.float64 or a.dtype.kind in "iu" else np.float32)
        share = (budget // (len(items) - i) - 128) // a.itemsize          # 128 B: the .npy header
        if a.size > share:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, share, replace=False))]
        path = os.path.join(out_dir, name + ".npy")
        np.save(path, a)
        budget -= os.path.getsize(path)
    return limit - budget


def train_step_outputs(step, loss):
    """What a caller of ``TrainStep`` holds after a step: the loss it returned, the model state after the Adam update
    (parameters and BatchNorm running statistics) and the parameter gradients of that step."""
    out = {"loss": loss.detach().cpu().numpy()}
    out.update({f"state.{k}": v.detach().cpu().numpy() for k, v in step.model.state_dict().items()})
    out.update({f"grad.{k}": step.grad_of(k).detach().cpu().numpy() for k, _ in step.flat.named})
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100", "-i", str(self.gpu)], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                smax.append(float(parts[2]))
                power.append(float(parts[3]))
            except ValueError:
                continue
            for nm, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        self.f.close()
        os.unlink(self.f.name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(smax), "power_w_max": max(power),
                "samples": len(sm), "reasons": sorted(reasons)}


# =============================================================================================== reference arms
class _NullLogger:
    def info(self, *a, **k):
        pass


def load_reference():
    """The UNMODIFIED reference hot path + engine loop, vendored by ``__graft_entry__.build()`` into the git-ignored
    ``baseline/_ref/`` (model/dstdgcn.py, model/layers/*, engine/prediction.py, engine/utils/*).  None if absent."""
    ref = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.exists(os.path.join(ref, "engine", "prediction.py")):
        try:
            import __graft_entry__ as ge
            ge.vendor_reference()
        except Exception:
            pass
    if not os.path.exists(os.path.join(ref, "engine", "prediction.py")):
        return None
    if ref not in sys.path:
        sys.path.insert(0, ref)
    import importlib
    return importlib.import_module("model.dstdgcn"), importlib.import_module("engine.prediction")


ENGINE_CFG = {  # configs/dstdgcn/dstdgcn_h36m.yaml:144-160 (the engine section is the same for the three datasets)
    "learn": {"opt": "adam", "lr": 3e-3, "weight_decay": 0, "gamma": 0.9, "step_size": 5},
    "loss": {"joint": ["jl2", 1]}, "n_out": 1, "transform": "tsc", "use_weight": False, "inverse": True, "max_iter": 2000}


def reference_engine(workload, device):
    """``PredictionEngine`` of the reference around the reference ``DSTDGCN`` with the workload's constructor arguments
    (dropout included), exactly as ``runner/base.py:33-37`` assembles them, on `device`."""
    import torch
    ref = load_reference()
    if ref is None:
        return None
    ref_model, ref_engine = ref
    layout, v, t_in, t_out, drop = WORKLOADS[workload]
    torch.manual_seed(777)
    m = ref_model.DSTDGCN(6, t_in, t_out, drop, v, feat(workload), N_LAYERS, layout)
    for p in m.parameters():            # what `.to("cuda")` does to the A_s / R_s alias (SURVEY.md section 0, quirk 1)
        p.data = p.data.clone()
    m = perturb(m).to(device)
    return ref_engine.PredictionEngine(ENGINE_CFG, m, _NullLogger())


def reference_loader(workload, batch, k, seed=777):
    layout, v, t_in, t_out, _ = WORKLOADS[workload]
    t = t_in + t_out
    out = []
    for i in range(min(k, 4)):
        a, b, c = synthetic_batch(batch, t, v, t_in, seed=seed + i)
        out.append((a, b, c, c))
    return [out[i % len(out)] for i in range(k)]


def oracle_step_fn(workload, batch, threads, drop):
    """Fallback when baseline/_ref is absent: the oracle port of engine/prediction.py:215-294 (fp32, torch CPU)."""
    import torch
    from dstd_gcn_b200.model import dstdgcn as std
    from oracle import dstd_oracle as orc
    layout, v, t_in, t_out, _ = WORKLOADS[workload]
    t = t_in + t_out
    torch.set_num_threads(threads)
    torch.manual_seed(777)
    m = perturb(std.DSTDGCN(6, t_in, t_out, 0.0, v, feat(workload), N_LAYERS, layout))
    p = orc.state_from_module(m, torch.float32)
    params = [x for x in p.values() if x.requires_grad]
    opt = torch.optim.Adam(params, lr=3e-3)
    inputs, inputs_inv, targets = synthetic_batch(batch, t, v, t_in, seed=777)

    def step():
        loss = orc.train_loss(p, inputs, inputs_inv, targets)
        opt.zero_grad()
        loss.backward()
        opt.step()
        return float(loss.detach())

    return step


def time_cpu_reference(workload, batch, steps, warmup, threads):
    """(samples/s, s/step, kind) of the reference's CPU path: ``PredictionEngine.train`` of the vendored reference, all
    host threads; the only shim is ``Tensor.cuda`` -> identity (the loop calls ``.cuda()`` on every batch,
    engine/prediction.py:223-225).  Falls back to the oracle port when baseline/_ref is absent."""
    import torch
    torch.set_num_threads(threads)
    eng = reference_engine(workload, "cpu")
    if eng is None:
        step = oracle_step_fn(workload, batch, threads, WORKLOADS[workload][4])
        for _ in range(warmup):
            step()
        t0 = time.perf_counter()
        for _ in range(steps):
            step()
        dt = time.perf_counter() - t0
        return batch * steps / dt, dt / steps, "port"
    real_cuda = torch.Tensor.cuda
    torch.Tensor.cuda = lambda self, *a, **k: self
    try:
        devnull = open(os.devnull, "w")
        err, sys.stderr = sys.stderr, devnull          # tqdm progress bars of the reference loop
        try:
            if warmup:
                eng.train(reference_loader(workload, batch, warmup), 0, max_iter=warmup)
            loader = reference_loader(workload, batch, steps)
            t0 = time.perf_counter()
            eng.train(loader, 0, max_iter=steps)
            dt = time.perf_counter() - t0
        finally:
            sys.stderr = err
            devnull.close()
    finally:
        torch.Tensor.cuda = real_cuda
    return batch * steps / dt, dt / steps, "reference"


def time_gpu_eager_reference(workload, batch, steps, warmup):
    """The same unmodified reference loop with the model on the B200 (torch eager: cuDNN / cuBLAS, TF32 off), the only
    pre-existing Blackwell path of this workload (SURVEY.md section 2.2).  CUDA-event timed around ``train``; includes
    what the reference does every step: the batch upload and the ``loss.item()`` sync."""
    import torch
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    eng = reference_engine(workload, "cuda")
    if eng is None:
        return None
    devnull = open(os.devnull, "w")
    err, sys.stderr = sys.stderr, devnull
    try:
        eng.train(reference_loader(workload, batch, warmup), 0, max_iter=warmup)
        loader = [tuple(x.pin_memory() for x in b) for b in reference_loader(workload, batch, steps)]
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        eng.train(loader, 0, max_iter=steps)
        e1.record()
        torch.cuda.synchronize()
    finally:
        sys.stderr = err
        devnull.close()
    ms = e0.elapsed_time(e1)
    return {"value": batch * steps / (ms * 1e-3), "unit": "samples/s", "ms_per_step": ms / steps, "steps": steps,
            "what": "unmodified reference (baseline/_ref: model/dstdgcn.py + engine/prediction.py PredictionEngine.train) "
                    f"on the same B200, torch {torch.__version__} eager fp32 (TF32 off), batch {batch}, same synthetic "
                    "batches from pinned host memory, loss.item() every step as the reference does"}


def time_gpu_eager_inference(args, ours, host, dev):
    """Eval-mode forward of the unmodified reference module (baseline/_ref, same variant) on the same B200 with OUR
    model's weights and running statistics (so both compute the same function), torch eager fp32, no_grad."""
    import importlib
    import torch
    if load_reference() is None:
        return None
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    mod = importlib.import_module("model.dstdgcn_fast" if args.variant == "dstdgcn_fast" else "model.dstdgcn")
    layout, v, t_in, t_out, drop = WORKLOADS[args.workload]
    ref = mod.DSTDGCN(6, t_in, t_out, drop, v, feat(args.workload), N_LAYERS, layout)
    for p in ref.parameters():
        p.data = p.data.clone()
    ref.load_state_dict(ours.state_dict(), strict=True)
    ref = ref.to(dev).eval()
    xs = [h.to(dev) for h in host]
    with torch.no_grad():
        y = ref(xs[0])
        for _ in range(2):
            ref(xs[1])
        torch.cuda.synchronize()
        k = max(3, min(args.steps, 10))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(k):
            ref(xs[i % len(xs)])
        e1.record()
        torch.cuda.synchronize()
        mine = ours(xs[0])
    ms = e0.elapsed_time(e1) / k
    return {"value": args.batch / (ms * 1e-3), "unit": "samples/s", "ms_per_step": ms, "steps": k,
            "max_abs_diff_vs_this_path": float((mine - y).abs().max()), "output_scale": float(y.abs().max()),
            "what": f"unmodified reference {mod.__name__}.DSTDGCN (baseline/_ref), eval forward, torch eager fp32 (TF32 off), "
                    f"batch {args.batch}, same weights and running statistics"}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    warm = max(min(args.warmup, 2), 1)
    steps = args.steps
    if args.cpu_seconds > 0:            # bound the CPU work: probe one step, then fit the sample into the budget
        _, sec1, _ = time_cpu_reference(args.workload, args.batch, 1, 1, threads)
        steps = max(2, min(args.steps, int(args.cpu_seconds / max(sec1, 1e-3))))
        warm = 1                        # one untimed step on the engine that is timed (the probe ran on its own engine)
    sps, sec, kind = time_cpu_reference(args.workload, args.batch, steps, warm, threads)
    sps32, sec32, _ = time_cpu_reference(args.workload, 32, max(2, min(steps, 10)), 1, threads)
    what = ("unmodified reference (baseline/_ref) PredictionEngine.train" if kind == "reference" else "oracle port")
    sample = (f"{steps} engine steps of batch {args.batch} (fp32, two forwards + backward + Adam each), {what}, "
              f"{sec:.2f} s/step")
    line = {
        "impl": "reference", "metric": "train_samples_per_s", "value": sps, "unit": "samples/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args),
        "cpu_baseline": {"value": sps, "unit": "samples/s", "cores": threads, "kind": kind, "sample": sample},
        "batch32": {"value": sps32, "unit": "samples/s", "ms_per_step": sec32 * 1e3,
                    "note": "the reference's own batch size (configs/dstdgcn/dstdgcn_h36m.yaml), BASELINE.json config 1"},
        "e2e": {"value": sps, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def workload_config(args, batch_override=None):
    layout, v, t_in, t_out, drop = WORKLOADS[args.workload]
    b = batch_override if batch_override is not None else args.batch
    return {"workload": f"DSTD-GCN {args.workload} shape ({v} joints, {t_in}->{t_out} frames, xyz), C={feat(args.workload)}, "
                        f"L={N_LAYERS}, training step with inverse pass, batch {b} per GPU",
            "variant": "dstdgcn", "batch_per_gpu": b, "global_batch": b * args.gpus, "inverse": True,
            "dropout": drop, "l2_policy": "per-step working set (activations + saved tensors) >> 126 MB L2; "
                                          "inputs rotate over 4 distinct batches"}


# =============================================================================================== inference sweep
def run_infer(args, model, be, dev, rank, world, t, v, t_in):
    """Eval-mode forward throughput (engine/prediction.py:340-353): BatchNorm on running statistics, no_grad, the whole
    forward captured in one CUDA graph; replicas only (no collective)."""
    import torch
    import torch.distributed as dist
    host = [synthetic_batch(args.batch, t, v, t_in, seed=777 + rank * 1000 + i)[0].view(args.batch, t, v, 3).pin_memory()
            for i in range(4)]
    with torch.no_grad():
        model.train()
        for i in range(2):                       # move the running statistics off (0, 1) as two training steps would
            model(host[i].to(dev))
        model.eval()
        static_in = host[0].to(dev)
        resident = [h.to(dev) for h in host]
        from dstd_gcn_b200.engine import forward_overlapped
        fwd = (lambda z: forward_overlapped(model, z, args.infer_streams)) if args.infer_streams > 1 else model
        for _ in range(2):
            out = fwd(static_in)
        torch.cuda.synchronize()
        l0 = be.launches
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            static_out = fwd(static_in)
        launches_per_step = be.launches - l0
    out_host = torch.empty_like(static_out, device="cpu").pin_memory()

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(e2e, k):
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(k):
            static_in.copy_(host[i % 4] if e2e else resident[i % 4], non_blocking=True)
            graph.replay()
            if e2e:
                out_host.copy_(static_out, non_blocking=True)
                torch.cuda.current_stream().synchronize()
        e1.record()
        sync_all()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms)

    timed(False, args.warmup)
    sampler = ClockSampler(int(os.environ.get("LOCAL_RANK", "0"))) if rank == 0 else None
    if sampler:
        sampler.start()
    ms = timed(False, args.steps)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"predictions": static_out.cpu().numpy()})
    ms_e2e = timed(True, args.steps)
    if rank == 0:
        total = args.batch * world * args.steps
        sps, sps_e2e = total / (ms * 1e-3), total / (ms_e2e * 1e-3)
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        peak = float(json.load(open(peaks_path))["hbm_gbs"]) if os.path.exists(peaks_path) else 6650.0
        cf = feat(args.workload)
        chans = [(6, cf)] + [(cf, cf)] * N_LAYERS + [(cf, 3)]
        bytes_fwd = 4 * t * v * sum(ci + co for ci, co in chans)
        achieved = sps / world * bytes_fwd / 1e9
        cfg = workload_config(args)
        cfg["workload"] = cfg["workload"].replace("training step with inverse pass", "eval-mode forward (BN on running stats)")
        cfg["variant"] = args.variant
        eager = None
        if not args.no_gpu_eager_baseline:
            try:
                eager = time_gpu_eager_inference(args, model, host, dev)
            except Exception as e:
                eager = {"error": repr(e)}
        print(json.dumps({
            "metric": "infer_samples_per_s", "value": sps, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
            "e2e": {"value": sps_e2e, "unit": "samples/s", "h2d_bytes_per_step": host[0].numel() * 4,
                    "d2h_bytes_per_step": out_host.numel() * 4, "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": launches_per_step * args.steps, "cuda_graph": True, "infer_streams": args.infer_streams,
            "clocks": clocks,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": None, "scope": f"forward only: {bytes_fwd} algorithmic B per sample (SURVEY.md 8d)"},
            "gpu_eager_baseline": eager,
        }), flush=True)
    if world > 1:
        shutdown(dist, torch)


def shutdown(dist, torch):
    """Orderly multi-rank exit: a barrier (rank 0 may arrive late, it times the CPU / eager baselines after the bench;
    the NCCL watchdog allows 10 minutes), then the communicator is destroyed.  Round 1 left through ``os._exit``."""
    torch.cuda.synchronize()
    sys.stdout.flush()
    try:
        dist.barrier()
        torch.cuda.synchronize()
        dist.destroy_process_group()
    except Exception as e:          # never lose the printed line over teardown
        print(f"bench: teardown failed ({e!r}); leaving", file=sys.stderr, flush=True)
        os._exit(0)


def secondary_lines(args, std, dev, resident, layout, v, t_in, t_out, drop):
    """Secondary measurements of the same training step (never the headline): the opt-in all-tcgen05 unit kernels at
    full fp32 parity, and their stated-tolerance modes (DSTD_PRECISION) that show how much of the step is the price of
    1e-4 parity.  Same model, batch, CUDA-graph capture and CUDA-event timing as the main line."""
    import torch
    from dstd_gcn_b200.engine import TrainStep
    out = {}
    modes = [("all_tcgen05_fp32_parity", {"DSTD_UNIT_TC": "1"}, "six bf16 split products per k-step (x = h + m + l): fp32 parity, max-abs 1e-4"),
             ("bf16x2", {"DSTD_PRECISION": "bf16x2"}, "three split products (hh + hm + mh): relative error <= 3e-4 per unit"),
             ("bf16", {"DSTD_PRECISION": "bf16"}, "plain bf16 operands, fp32 accumulate: relative error <= 3e-2 per unit")]
    for name, env, what in modes:
        old = {k: os.environ.get(k) for k in env}
        os.environ.update(env)
        try:
            torch.manual_seed(777)
            m = perturb(std.DSTDGCN(6, t_in, t_out, drop, v, feat(args.workload), N_LAYERS, layout)).to(dev).train()
            st = TrainStep(m, lr=3e-3, inverse=True)
            st.capture(*resident[0])
            for i in range(3):
                st(*resident[i % len(resident)])
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            k = max(3, min(args.steps, 10))
            e0.record()
            for i in range(k):
                st(*resident[i % len(resident)])
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / k
            out[name] = {"value": args.batch / (ms * 1e-3), "unit": "samples/s", "ms_per_step": ms, "steps": k,
                         "precision": what}
        except Exception as e:
            out[name] = {"error": repr(e)}
        finally:
            for k2, v2 in old.items():
                if v2 is None:
                    os.environ.pop(k2, None)
                else:
                    os.environ[k2] = v2
    return out


# =============================================================================================== GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=None, help="samples per GPU per step (default 256; 32 for stress)")
    ap.add_argument("--workload", default="h36m", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--infer-streams", type=int, default=4,
                    help="--mode infer: independent sub-batches of the eval forward on this many streams (1 = one chain)")
    ap.add_argument("--mode", default="train", choices=["train", "infer"],
                    help="train: the headline metric; infer: eval-mode forward sweep (BASELINE.json config 4)")
    ap.add_argument("--variant", default="dstdgcn", choices=["dstdgcn", "dstdgcn_fast"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --batch samples per GPU; strong: --batch is the GLOBAL batch, split over the ranks")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the stated-tolerance / all-tcgen05 secondary lines")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel from Python instead of one CUDA graph")
    ap.add_argument("--cpu-baseline-steps", type=int, default=4)
    ap.add_argument("--cpu-seconds", type=float, default=90.0,
                    help="--impl reference: budget of CPU work for the timed sample (0 = run exactly --steps)")
    ap.add_argument("--no-gpu-eager-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU arm (--impl b200)")
    if args.batch is None:
        args.batch = DEFAULT_BATCH.get(args.workload, 256)
    args.global_batch_fixed = None
    if args.scaling == "strong":
        world_env = int(os.environ.get("WORLD_SIZE", "1"))
        assert args.batch % world_env == 0, "--scaling strong: the global batch must divide by the number of ranks"
        args.global_batch_fixed = args.batch
        args.batch = args.batch // world_env
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch
    import torch.distributed as dist
    from dstd_gcn_b200 import _lib
    from dstd_gcn_b200.engine import TrainStep
    from dstd_gcn_b200.model import dstdgcn as std
    if args.variant == "dstdgcn_fast":
        from dstd_gcn_b200.model import dstdgcn_fast as std

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torch.distributed.run)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    layout, v, t_in, t_out, drop = WORKLOADS[args.workload]
    t = t_in + t_out
    torch.manual_seed(777)                       # identical replicas on every rank
    model = perturb(std.DSTDGCN(6, t_in, t_out, drop, v, feat(args.workload), N_LAYERS, layout)).to(dev).train()
    be = _lib.backend()
    if args.mode == "infer":
        run_infer(args, model, be, dev, rank, world, t, v, t_in)
        return
    step = TrainStep(model, lr=3e-3, inverse=True)

    nbuf = 4
    host = [synthetic_batch(args.batch, t, v, t_in, seed=777 + rank * 1000 + i) for i in range(nbuf)]
    host = [tuple(x.pin_memory() for x in b) for b in host]
    resident = [tuple(x.to(dev) for x in b) for b in host]
    loss_host = torch.empty((), dtype=torch.float32).pin_memory()
    launches_per_step = None
    if not args.no_graph:
        l0 = be.launches
        step.capture(*resident[0])            # whole step -> one CUDA graph (state rolled back after its warm-up)
        launches_per_step = (be.launches - l0) // 3       # 2 warm-up steps + the captured one
        stage = [step._static]
    else:
        stage = [tuple(torch.empty_like(x, device=dev) for x in host[0]) for _ in range(2)]

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    last_loss = [None]

    def run_resident(k):
        for i in range(k):
            last_loss[0] = step(*resident[i % nbuf])

    def run_e2e(k):
        for i in range(k):
            hb, db = host[i % nbuf], stage[i % len(stage)]
            for h, d in zip(hb, db):
                d.copy_(h, non_blocking=True)
            loss = step(*db)
            loss_host.copy_(loss, non_blocking=True)
            torch.cuda.current_stream().synchronize()     # the user reads the loss every step

    def timed(fn, k):
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = be.launches
        e0.record()
        fn(k)
        e1.record()
        sync_all()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms), (launches_per_step * k if launches_per_step is not None else be.launches - l0)

    secondary = None
    run_resident(args.warmup)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    ms, launches = timed(run_resident, args.steps)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, train_step_outputs(step, last_loss[0]))
    run_e2e(2)
    ms_e2e, _ = timed(run_e2e, args.steps)
    if world == 1 and not args.no_secondary and not args.no_graph:
        secondary = secondary_lines(args, std, dev, resident, layout, v, t_in, t_out, drop)

    if rank == 0:
        total = args.batch * world * args.steps
        sps = total / (ms * 1e-3)
        sps_e2e = total / (ms_e2e * 1e-3)
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        else:
            peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
        bytes_pass = algorithmic_bytes_per_pass(v, t, feat(args.workload))
        # DRAM bytes per step as MEASURED EARLIER with ncu (dram__bytes_read+write over every launch of one step) and
        # committed under profiles/: a static figure, not re-measured by this run (traffic_source says which file)
        traffic, traffic_src = None, None
        for rr in ("r02", "r01"):
            tpath = os.path.join(ROOT, "profiles", f"{rr}_dram_traffic_{args.workload}_b{args.batch}.json")
            if os.path.exists(tpath):
                traffic = json.load(open(tpath)).get("dram_bytes_per_step")
                traffic_src = f"profiles/{os.path.basename(tpath)} (static: measured with ncu in an earlier run)"
                break
        passes_per_s_gpu = 2.0 * sps / world                      # inverse=True: two model passes per sample
        achieved = passes_per_s_gpu * bytes_pass / 1e9
        h2d = sum(x.numel() * 4 for x in host[0])
        line = {
            "metric": "train_samples_per_s", "value": sps, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(args),
            "model_passes_per_s": 2.0 * sps,
            "e2e": {"value": sps_e2e, "unit": "samples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                    "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": launches, "cuda_graph": not args.no_graph,
            "clocks": clocks,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "algorithmic_bytes_per_step": 2 * bytes_pass * args.batch,
                         "scope": "whole training step per GPU: algorithmic bytes = one HBM round trip per DSTDGCB "
                                  f"layer fwd+bwd = {bytes_pass} B per model pass (SURVEY.md 8d), 2 passes per sample",
                         "algorithmic_bytes_per_sample": 2 * bytes_pass},
        }
        try:
            line["roofline"]["dominant_call"] = dominant_call_roofline(args.batch, v, t, peak, c=feat(args.workload))
        except Exception as e:      # never lose the bench line over the extra measurement
            line["roofline"]["dominant_call"] = {"error": repr(e)}
        if world == 1 and not args.no_secondary:
            line["secondary"] = secondary
        if world == 1 and not args.no_gpu_eager_baseline:       # baselines are single-GPU legs (rank 0, N = 1 only)
            try:
                line["gpu_eager_baseline"] = time_gpu_eager_reference(args.workload, args.batch, min(args.steps, 10), 3)
            except Exception as e:
                line["gpu_eager_baseline"] = {"error": repr(e)}
        if world == 1 and not args.no_cpu_baseline:
            threads = os.cpu_count() or 1
            v_cpu, sec, kind = time_cpu_reference(args.workload, args.batch, args.cpu_baseline_steps, 1, threads)
            line["cpu_baseline"] = {"value": v_cpu, "unit": "samples/s", "cores": threads, "kind": kind,
                                    "sample": f"{args.cpu_baseline_steps} engine steps of batch {args.batch} (same "
                                              f"workload and batch, fp32, all host threads), {sec:.2f} s/step"}
        print(json.dumps(line), flush=True)
    if world > 1:
        shutdown(dist, torch)


if __name__ == "__main__":
    main()
