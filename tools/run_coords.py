"""Training throughput on 2-D poses (DSTDGCN(4, ...), x [N, T, V, 2]) next to xyz (DSTDGCN(6, ...)).
    python tools/run_coords.py [--steps 50] [--rounds 3] [--out FILE]

Benchmark setup (bench.py's h36m workload): 22 joints, C=64, L=5, 10 -> 25 frames (T=35), dropout 0.1, batch 256,
inverse pass, the whole step captured as one CUDA graph, CUDA-event timing over --steps steps after warm-up.  D = 2 and
D = 3 are measured in alternating runs (--rounds pairs, each a fresh model), so that drift of the shared machine falls
on both.  Only the first layer (2D -> C), the last layer (C -> D), the head, the tail and the loss depend on D.  Prints
one line per run and a JSON summary with the card's name, power limit and SM clocks read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench                                   # noqa: E402
from dstd_gcn_b200.engine import TrainStep     # noqa: E402
from dstd_gcn_b200.model import dstdgcn        # noqa: E402


def card():
    dev = torch.cuda.current_device()
    out = {"name": torch.cuda.get_device_name(dev), "power_limit_w": None}
    try:
        r = subprocess.run(["nvidia-smi", "-i", str(dev), "--query-gpu=power.limit,clocks.sm,clocks.max.sm",
                            "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30)
        pl, sm, smax = (x.strip() for x in r.stdout.strip().split(","))
        out["power_limit_w"], out["sm_clock_mhz"], out["sm_clock_max_mhz"] = float(pl), float(sm), float(smax)
    except Exception as e:           # the figure is then reported as unknown, never guessed
        out["error"] = repr(e)
    return out


def pose_batch(n, t, v, d, t_in, seed):
    """bench.synthetic_batch with D coordinates per joint (the same draws at D = 3): raw [N,T,D*V] (inputs, inputs_inv,
    targets)."""
    g = torch.Generator().manual_seed(seed)
    seq = torch.randn(n, 1, v * d, generator=g) + torch.cumsum(torch.randn(n, t, v * d, generator=g) * 0.05, dim=1)
    inputs = seq.clone()
    inputs[:, t_in:] = seq[:, t_in - 1:t_in]
    rev = torch.flip(seq, dims=[1])
    inputs_inv = rev.clone()
    inputs_inv[:, t_in:] = rev[:, t_in - 1:t_in]
    return inputs.contiguous(), inputs_inv.contiguous(), seq.contiguous()


def train_rate(d, steps, batch):
    dev = torch.device("cuda")
    lay, v, t_in, t_out, drop = bench.WORKLOADS["h36m"]
    torch.manual_seed(777)
    m = bench.perturb(dstdgcn.DSTDGCN(2 * d, t_in, t_out, drop, v, bench.C_FEAT, bench.N_LAYERS, lay)).to(dev).train()
    st = TrainStep(m, lr=3e-3, inverse=True)
    resident = [tuple(x.to(dev) for x in pose_batch(batch, t_in + t_out, v, d, t_in, seed=777 + i)) for i in range(4)]
    st.capture(*resident[0])
    for i in range(3):
        st(*resident[i % 4])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        st(*resident[i % 4])
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return {"samples_per_s": batch / (ms * 1e-3), "ms_per_step": ms}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--out", default=None, help="also write the JSON summary here")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("run_coords.py measures on the GPU; no CUDA device found")
    lay, v, t_in, t_out, drop = bench.WORKLOADS["h36m"]
    res = {"card": card(), "setup": {"V": v, "C": bench.C_FEAT, "L": bench.N_LAYERS, "T": t_in + t_out,
                                     "batch": a.batch, "dropout": drop, "graph": True, "steps": a.steps},
           "runs": []}
    for r in range(a.rounds):
        for d in (2, 3):
            x = train_rate(d, a.steps, a.batch)
            res["runs"].append({"D": d, **x})
            print(f"round {r} D={d}: {x['samples_per_s']:.0f} samples/s ({x['ms_per_step']:.3f} ms/step)")
    for d in (2, 3):
        rates = [x["samples_per_s"] for x in res["runs"] if x["D"] == d]
        res[f"D{d}_samples_per_s"] = {"min": min(rates), "max": max(rates), "mean": sum(rates) / len(rates)}
    res["card_after"] = card()
    c = res["card"]
    print(f"{c['name']}: power limit {c['power_limit_w']} W, SM clock {c.get('sm_clock_mhz')} MHz "
          f"(max {c.get('sm_clock_max_mhz')} MHz); after the runs {res['card_after'].get('sm_clock_mhz')} MHz")
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
