"""Training throughput and BatchNorm cost on registered skeletons of more than 32 joints, next to H3.6M (22 joints).
    python tools/run_skeleton.py [--steps 10] [--out FILE]

Benchmark setup (bench.py's h36m workload): C=64, L=5, 10 -> 25 frames (T=35), dropout 0.1, batch 256, inverse pass,
the whole step captured as one CUDA graph, CUDA-event timing over --steps steps after warm-up.  The 33-, 38- and
55-joint layouts are synthetic tree skeletons registered with graph.register_layout (the joint count is what the
kernels see).  BatchNorm: µs per call of the block BN (residual, T-major -> V-major) and the encoder BN (V-major ->
T-major) at V = 38 and 22, replayed as a CUDA graph.  Prints one line per measurement and a JSON summary with the
card name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench                                   # noqa: E402
from dstd_gcn_b200 import _lib                 # noqa: E402
from dstd_gcn_b200.engine import TrainStep     # noqa: E402
from dstd_gcn_b200.model import dstdgcn        # noqa: E402
from dstd_gcn_b200.model.layers import graph   # noqa: E402
from dstd_gcn_b200.ops import _out_like        # noqa: E402
from run_bn import _graph_us                   # noqa: E402


def register(joints):
    """A tree skeleton of `joints` joints: bone (j // 2, j), part pairs (j, j + 2) every third joint."""
    name = f"tree{joints}"
    graph.register_layout(name, joints, [(j // 2, j) for j in range(1, joints)],
                          [(j, j + 2) for j in range(0, joints - 2, 3)])
    return name


def card():
    dev = torch.cuda.current_device()
    out = {"name": torch.cuda.get_device_name(dev), "power_limit_w": None}
    try:
        r = subprocess.run(["nvidia-smi", "-i", str(dev), "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30)
        pl, smax = (x.strip() for x in r.stdout.strip().split(","))
        out["power_limit_w"], out["sm_clock_max_mhz"] = float(pl), float(smax)
    except Exception as e:           # the figure is then reported as unknown, never guessed
        out["error"] = repr(e)
    return out


def train_rate(lay, v, steps, batch):
    dev = torch.device("cuda")
    _, _, t_in, t_out, drop = bench.WORKLOADS["h36m"]
    torch.manual_seed(777)
    m = bench.perturb(dstdgcn.DSTDGCN(6, t_in, t_out, drop, v, bench.C_FEAT, bench.N_LAYERS, lay)).to(dev).train()
    st = TrainStep(m, lr=3e-3, inverse=True)
    resident = [tuple(x.to(dev) for x in bench.synthetic_batch(batch, t_in + t_out, v, t_in, seed=777 + i))
                for i in range(4)]
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


def bn_us(v, n, reps):
    dev, be = torch.device("cuda"), _lib.backend()
    c, t = bench.C_FEAT, 35
    g = torch.Generator().manual_seed(0)
    gamma, beta = torch.ones(c * v, device=dev), torch.zeros(c * v, device=dev)
    rm, rv = torch.zeros(c * v, device=dev), torch.ones(c * v, device=dev)
    nbt = torch.zeros((), dtype=torch.int64, device=dev)
    prelu = torch.tensor([0.25], device=dev)
    cases = {"block": (torch.randn(n, c, t, v, generator=g).to(dev), torch.randn(n, c, t, v, generator=g).to(dev), 2),
             "encoder": (torch.randn(n, c, v, t, generator=g).to(dev).permute(0, 1, 3, 2), None, 1)}
    res = {}
    for name, (y, r, order) in cases.items():
        ol = _out_like(y, order)
        out, mean, istd = be.bn_act_forward(y, r, gamma, beta, rm, rv, nbt, prelu, None, False, True, 1e-5, 0.1, ol)
        fwd = lambda: be.bn_act_forward(y, r, gamma, beta, rm, rv, nbt, prelu, None, False, True, 1e-5, 0.1, ol)
        bwd = lambda: be.bn_act_backward(y, r, out, gamma, beta, prelu, None, mean, istd, False, True, True)
        res[name] = {"fwd_us": _graph_us(fwd, reps), "bwd_us": _graph_us(bwd, reps)}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--out", default=None, help="also write the JSON summary here")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("run_skeleton.py measures on the GPU; no CUDA device found")
    res = {"card": card(), "setup": {"C": bench.C_FEAT, "L": bench.N_LAYERS, "T": 35, "batch": a.batch,
                                     "dropout": bench.WORKLOADS["h36m"][4], "graph": True, "steps": a.steps},
           "train": {}, "bn": {}}
    for v in (22, 33, 38, 55):
        lay = "h36m" if v == 22 else register(v)
        res["train"][v] = train_rate(lay, v, a.steps, a.batch)
        print(f"train V={v}: {res['train'][v]['samples_per_s']:.0f} samples/s ({res['train'][v]['ms_per_step']:.2f} ms/step)")
    for v in (22, 38):
        res["bn"][v] = bn_us(v, a.batch, a.reps)
        for k, x in res["bn"][v].items():
            print(f"BN V={v} {k}: fwd {x['fwd_us']:.1f} us  bwd {x['bwd_us']:.1f} us")
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
